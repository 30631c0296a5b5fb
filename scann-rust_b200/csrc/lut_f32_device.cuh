// LookupTable::from_query / compute_distance (src/hashes/lut.rs:47-82) in the reference's f32 operation order, shared
// by the façade's per-query kernel (ivf.cu) and the Tree-X-Hybrid byte-code scan (lut_f32_scan_kernel.cuh).
#pragma once

#include <cstdint>

namespace scann {

#ifdef __CUDACC__

// table[s][c] = Σ_j (q[s*ds + j] - cb[s][c][j])², the sequential un-fused sum of SubspaceCodebook::compute_distances;
// the caller's threads split the S*C entries (entries first, first + step, ...)
__device__ __forceinline__ void lut_f32_build(float* lut, const float* q, const float* __restrict__ codebook, int S,
                                              int C, int ds, int first, int step) {
  for (int e = first; e < S * C; e += step) {
    const int s = e / C;
    float sum = 0.0f;
    for (int j = 0; j < ds; ++j) {
      const float d = __fsub_rn(q[s * ds + j], __ldg(codebook + static_cast<size_t>(e) * ds + j));
      sum = __fadd_rn(sum, __fmul_rn(d, d));
    }
    lut[e] = sum;
  }
}

// one step of compute_distance: sum += distances[s][code] (lut_s = row s of the table)
__device__ __forceinline__ float lut_f32_add(float sum, const float* lut_s, uint32_t code) {
  return __fadd_rn(sum, lut_s[code]);
}

// compute_distance of one row-major code row (S bytes), s = 0..S-1 in that order.  The row is fetched with the widest
// aligned loads available (one byte load per subspace made the per-query kernel LSU-bound).
__device__ __forceinline__ float lut_f32_row_distance(const float* lut, const uint8_t* __restrict__ c, int S, int C) {
  float d = 0.0f;
  auto add4 = [&](uint32_t w, int s0) {
#pragma unroll
    for (int j = 0; j < 4; ++j) d = lut_f32_add(d, lut + (s0 + j) * C, (w >> (8 * j)) & 0xFFu);
  };
  if ((S & 15) == 0) {
    for (int s0 = 0; s0 < S; s0 += 16) {
      const uint4 w = __ldg(reinterpret_cast<const uint4*>(c + s0));
      add4(w.x, s0);
      add4(w.y, s0 + 4);
      add4(w.z, s0 + 8);
      add4(w.w, s0 + 12);
    }
  } else if ((S & 3) == 0) {
    for (int s0 = 0; s0 < S; s0 += 4) add4(__ldg(reinterpret_cast<const uint32_t*>(c + s0)), s0);
  } else {
    for (int s = 0; s < S; ++s) d = lut_f32_add(d, lut + s * C, c[s]);
  }
  return d;
}

#endif  // __CUDACC__

}  // namespace scann
