// The Tree-X-Hybrid scan over byte codes with the reference's f32 LookupTable (tree_x_hybrid/mod.rs:297-339,
// hashes/lut.rs:47-82): persistent kernel over the same (leaf, <= G queries) work items as lut16_scan_kernel.
//
// Per work item a CTA of kScanWarps warps
//   (1) stages the G query residuals q - centroid(leaf) in shared memory (skipped without residuals),
//   (2) builds the G f32 tables [S][C] in shared memory with LookupTable::from_query arithmetic (lut_f32_device.cuh),
//   (3) streams the leaf's blocked byte codes once for all G queries — one 256-point block per warp per tile, lane l
//       holding points l*8 .. l*8+7 and 8 x G running sums, sum += table[s][code] for s = 0 .. S-1 in that order
//       (LookupTable::compute_distance bit for bit),
//   (4) keeps an exact running top-R per query ordered by (approx distance, position): 64-bit keys
//       f32_key(distance) << 32 | position in a shared-memory buffer, a warp radix select when it could overflow,
//   (5) writes the <= R survivors {distance bits, position} of every (query, leaf) pair.
// Filtered-out points never enter a list (tree_x_hybrid/mod.rs:327-332).  The batch-wide bound qthr[q] works as in
// lut16_scan_kernel: whenever a leaf holds R candidates, the R-th distance is published with atomicMin, and points above
// the current bound are dropped (points AT the bound are kept, so results do not depend on the order of the items).
#pragma once

#include "lut16_scan_kernel.cuh"
#include "lut_f32_device.cuh"

namespace scann {

// Finds T = the R-th smallest of the c distinct u64 keys in buf (1 <= R < c), compacts buf in place to the R keys <= T
// and returns T.  hist: 256 u32 of shared memory private to the warp.
__device__ __forceinline__ uint64_t warp_select_u64(uint64_t* buf, int c, int R, uint32_t* hist, int lane) {
  uint64_t prefix = 0, mask = 0;
  uint32_t need = static_cast<uint32_t>(R);
  for (int shift = 56; shift >= 0; shift -= 8) {
#pragma unroll
    for (int j = 0; j < 8; ++j) hist[lane + 32 * j] = 0;
    __syncwarp();
    for (int i = lane; i < c; i += 32) {
      const uint64_t k = buf[i];
      if ((k & mask) == prefix) atomicAdd(&hist[static_cast<uint32_t>(k >> shift) & 255u], 1u);
    }
    __syncwarp();
    uint32_t d, below;
    warp_hist_digit(hist, need, lane, d, below);
    need -= below;
    prefix |= static_cast<uint64_t>(d) << shift;
    mask |= 0xFFull << shift;
    __syncwarp();
  }
  const uint64_t T = prefix;
  int write = 0;
  for (int base = 0; base < c; base += 32) {
    const int i = base + lane;
    const uint64_t k = i < c ? buf[i] : ~0ull;
    const bool keep = (i < c) && (k <= T);
    const uint32_t b = __ballot_sync(0xFFFFFFFFu, keep);
    __syncwarp();
    if (keep) buf[write + __popc(b & lanemask_lt())] = k;
    write += __popc(b);
    __syncwarp();
  }
  return T;
}

// inclusive u64 key bound of an f32_key distance bound: every position at or below that distance
__device__ __forceinline__ uint64_t f32_bound_key(uint32_t tk) {
  return tk == 0xFFFFFFFFu ? ~0ull : (static_cast<uint64_t>(tk) << 32) | 0xFFFFFFFFull;
}

// a.codes: the byte codes in 256-point blocks, block b at byte b * S * 256, subspace-major inside (byte s*256 + j =
// subspace s of point j).  C: codes per subspace (the table row length).  a.max_blocks / probe launches are not used.
template <int G, bool FILT>
__global__ void __launch_bounds__(kScanWarps * 32, 1) lut_f32_scan_kernel(const ScanArgs a, const int C) {
  extern __shared__ __align__(16) uint8_t smem[];
  const int SC = a.S * C;
  uint64_t* buf = reinterpret_cast<uint64_t*>(smem);                  // [G][cap] keys
  uint64_t* s_thr = buf + static_cast<size_t>(G) * a.cap;             // [G] inclusive key bound per query
  float* lut = reinterpret_cast<float*>(s_thr + G);                   // [G][S][C]
  float* qres = lut + static_cast<size_t>(G) * SC;                    // [G][dim]
  uint32_t* hist = reinterpret_cast<uint32_t*>(qres + G * a.dim);     // [kScanWarps][256]
  uint32_t* s_cnt = hist + kScanWarps * 256;                          // candidates buffered per query
  uint32_t* s_pair = s_cnt + G;                                       // pair id (q * L + rank)
  uint32_t* s_tau = s_pair + G;                                       // last qthr key seen per query
  uint32_t* s_row = s_tau + G;                                        // FILT: filter row (0xFFFFFFFF = none allowed)
  uint32_t* s_item = s_row + G;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t total_items = a.counters[a.end_idx];
  const uint8_t* codes = reinterpret_cast<const uint8_t*>(a.codes);

  for (;;) {
    __syncthreads();  // previous item's shared memory is dead
    if (tid == 0) *s_item = atomicAdd(&a.counters[1], 1u);
    __syncthreads();
    const uint32_t item = *s_item;
    if (item >= total_items) break;
    const uint4 it = a.items[item];
    const uint32_t leaf = it.x, pbeg = it.y;
    const int ng = static_cast<int>(it.z);
    const uint32_t blk0 = a.blk_off[leaf];
    const int nblk = static_cast<int>(a.blk_off[leaf + 1] - blk0);
    const uint32_t leaf_n = static_cast<uint32_t>(a.pt_off[leaf + 1] - a.pt_off[leaf]);

    // (1) query residuals: q - centroid (src/tree_x_hybrid/mod.rs:309-316)
    for (int idx = tid; idx < ng * a.dim; idx += kScanWarps * 32) {
      const int g = idx / a.dim, d = idx - g * a.dim;
      const uint32_t q = a.sorted_pairs[pbeg + g] / static_cast<uint32_t>(a.L);
      float v = a.queries[static_cast<size_t>(q) * a.dim + d];
      if (a.use_residuals) v = __fsub_rn(v, __ldg(a.centers + static_cast<size_t>(leaf) * a.dim + d));
      qres[idx] = v;
    }
    if (tid < ng) {
      const uint32_t pair = a.sorted_pairs[pbeg + tid];
      const uint32_t q = pair / static_cast<uint32_t>(a.L);
      s_pair[tid] = pair;
      const uint32_t tk = __ldcg(a.qthr + q);
      s_tau[tid] = tk;
      s_thr[tid] = f32_bound_key(tk);
      s_cnt[tid] = 0u;
      if (FILT) {
        const uint32_t row = a.qfilt ? a.qfilt[q] : 0u;
        s_row[tid] = row < a.num_filters ? row : 0xFFFFFFFFu;
      }
    }
    __syncthreads();

    // (2) the G tables
    for (int g = 0; g < ng; ++g)
      lut_f32_build(lut + static_cast<size_t>(g) * SC, qres + g * a.dim, a.codebook, a.S, C, a.ds, tid,
                    kScanWarps * 32);
    __syncthreads();

    // (3)+(4) stream the leaf, one 256-point block per warp per tile
    const int ntiles = (nblk + kScanWarps - 1) / kScanWarps;
    for (int t = 0; t < ntiles; ++t) {
      const int b = t * kScanWarps + warp;
      if (b < nblk) {
        float acc[G][8];
#pragma unroll
        for (int g = 0; g < G; ++g)
#pragma unroll
          for (int i = 0; i < 8; ++i) acc[g][i] = 0.0f;
        const uint2* cb = reinterpret_cast<const uint2*>(codes + (static_cast<size_t>(blk0) + b) * a.S * kBlockPts) + lane;
#pragma unroll 2
        for (int s = 0; s < a.S; ++s) {
          const uint2 w = __ldg(cb + s * (kBlockPts / 8));
#pragma unroll
          for (int g = 0; g < G; ++g) {
            if (g >= ng) continue;
            const float* ls = lut + static_cast<size_t>(g) * SC + s * C;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              acc[g][i] = lut_f32_add(acc[g][i], ls, (w.x >> (8 * i)) & 0xFFu);
              acc[g][4 + i] = lut_f32_add(acc[g][4 + i], ls, (w.y >> (8 * i)) & 0xFFu);
            }
          }
        }
        const uint32_t pos0 = static_cast<uint32_t>(b) * kBlockPts + lane * 8;
        const size_t at = (static_cast<size_t>(blk0) + b) * 32 + lane;
#pragma unroll
        for (int g = 0; g < G; ++g) {
          if (g >= ng) continue;
          uint32_t am = 0xFFu;
          if (FILT) {  // every query of the item reads the byte of its own filter row
            const uint32_t row = s_row[g];
            am = row == 0xFFFFFFFFu ? 0u : a.allow[row * a.allow_stride + at];
          }
          const uint64_t thr = s_thr[g];
          uint64_t* bg = buf + static_cast<size_t>(g) * a.cap;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const uint32_t pos = pos0 + i;
            const uint64_t key = (static_cast<uint64_t>(f32_key(acc[g][i])) << 32) | pos;
            const bool ok = pos < leaf_n && ((am >> i) & 1u) && key <= thr;
            const uint32_t bal = __ballot_sync(0xFFFFFFFFu, ok);
            if (bal == 0u) continue;
            uint32_t base = 0;
            if (lane == __ffs(bal) - 1) base = atomicAdd(&s_cnt[g], static_cast<uint32_t>(__popc(bal)));
            base = __shfl_sync(0xFFFFFFFFu, base, __ffs(bal) - 1);
            if (ok) {
              const uint32_t slot = base + __popc(bal & lanemask_lt());
              if (slot < static_cast<uint32_t>(a.cap)) bg[slot] = key;
            }
          }
        }
      }
      __syncthreads();
      // exact compaction to the R best when the buffer could overflow in the next tile; refresh the bound
      for (int g = warp; g < ng; g += kScanWarps) {
        int c = static_cast<int>(min(s_cnt[g], static_cast<uint32_t>(a.cap)));
        const uint32_t q = s_pair[g] / static_cast<uint32_t>(a.L);
        const int R = a.qR ? static_cast<int>(__ldg(a.qR + q)) : a.R;
        uint64_t thr = s_thr[g];
        if (c > R && (t == ntiles - 1 || c > 2 * R)) {
          thr = warp_select_u64(buf + static_cast<size_t>(g) * a.cap, c, R, hist + warp * 256, lane);
          c = R;
          if (lane == 0) {
            s_cnt[g] = static_cast<uint32_t>(R);
            // this leaf alone holds R allowed points at or below this distance
            atomicMin(a.qthr + q, static_cast<uint32_t>(thr >> 32));
          }
        }
        if (lane == 0) {
          if (t + 1 < ntiles) {
            const uint32_t tk = __ldcg(a.qthr + q);
            if (tk < s_tau[g]) {  // somebody tightened the batch-wide bound
              s_tau[g] = tk;
              thr = min(thr, f32_bound_key(tk));
            }
          }
          s_thr[g] = thr;
        }
      }
      __syncthreads();
    }

    // (5) this item's candidates
    for (int g = warp; g < ng; g += kScanWarps) {
      const uint32_t pair = s_pair[g];
      const uint32_t R = a.qR ? __ldg(a.qR + pair / static_cast<uint32_t>(a.L)) : static_cast<uint32_t>(a.R);
      const int c = static_cast<int>(min(s_cnt[g], R));
      const uint64_t* bg = buf + static_cast<size_t>(g) * a.cap;
      uint2* out = a.cand + static_cast<size_t>(pair) * a.R;
      for (int i = lane; i < c; i += 32) {
        const uint64_t key = bg[i];
        out[i] = make_uint2(__float_as_uint(key_f32(static_cast<uint32_t>(key >> 32))), static_cast<uint32_t>(key));
      }
      if (lane == 0) a.cand_cnt[pair] = static_cast<uint32_t>(c);
    }
  }
}

// Shared memory of one CTA: G tables of S*C floats dominate (48 KB per query at S = 48, C = 256).
inline size_t lut_f32_scan_smem_bytes(int G, int S, int C, int dim, int cap) {
  return static_cast<size_t>(G) * cap * 8 + static_cast<size_t>(G) * 8 + static_cast<size_t>(G) * S * C * 4 +
         static_cast<size_t>(G) * dim * 4 + static_cast<size_t>(kScanWarps) * 256 * 4 + static_cast<size_t>(G) * 4 * 4 +
         4 + 16;
}

}  // namespace scann
