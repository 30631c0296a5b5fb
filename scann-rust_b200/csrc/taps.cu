// Parity taps for the LUT16 pieces and the PQ encoder (index-build helper).  The taps call the same
// device functions as the Tree-AH hot kernel (lut16_device.cuh), so a bit-exact tap means the hot path's
// table build / integer accumulation is bit-exact.
#include <algorithm>

#include "lut16_device.cuh"

namespace scann {

// one warp per query: residual subtraction + LUT16 build
__global__ void __launch_bounds__(128) lut16_build_kernel(const float* __restrict__ cb, int S, int ds,
                                                          const float* __restrict__ queries, int nq,
                                                          const float* __restrict__ centroids,
                                                          uint8_t* __restrict__ lut8, float* __restrict__ bias,
                                                          float* __restrict__ mult) {
  extern __shared__ __align__(16) uint8_t sm[];
  const int dim = S * ds;
  const int S4 = (S + 3) / 4 * 4;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* qres = reinterpret_cast<float*>(sm) + warp * dim;
  uint8_t* l8 = sm + 4 * dim * sizeof(float) + warp * S4 * 16;
  const int q = blockIdx.x * 4 + warp;
  if (q >= nq) return;
  for (int d = lane; d < dim; d += 32) {
    float v = queries[static_cast<size_t>(q) * dim + d];
    if (centroids) v = __fsub_rn(v, centroids[static_cast<size_t>(q) * dim + d]);
    qres[d] = v;
  }
  __syncwarp();
  float m, b;
  warp_build_lut16(qres, cb, S, S4, ds, l8, &m, &b, lane);
  __syncwarp();
  for (int e = lane; e < S * 16; e += 32) lut8[static_cast<size_t>(q) * S * 16 + e] = l8[e];
  if (lane == 0) {
    bias[q] = b;
    mult[q] = m;
  }
}

// row-major PackedCodes4Bit -> blocked layout of a single "leaf" holding all n points
__global__ void repack_flat_kernel(const uint8_t* __restrict__ packed, size_t n, int S, int SG, size_t total_words,
                                   uint32_t* __restrict__ out) {
  size_t w = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (w >= total_words) return;
  int j = static_cast<int>(w & 3);
  int lane = static_cast<int>((w >> 2) & 31);
  size_t rest = w >> 7;
  int sg = static_cast<int>(rest % SG);
  size_t gb = rest / SG;
  int s = sg * 4 + j;
  uint32_t word = 0;
  if (s < S) {
    size_t p0 = gb * kBlockPts + lane * 8;
    int bpp = (S + 1) / 2;
    for (int i = 0; i < 8; ++i) {
      size_t p = p0 + i;
      if (p < n) {
        uint8_t b = packed[p * bpp + (s >> 1)];
        uint32_t nib = (s & 1) ? (b >> 4) : (b & 0x0F);
        word |= nib << (4 * i);
      }
    }
  }
  out[w] = word;
}

// all u32 accumulators of one u8 table over the blocked codes (scan_block<1>, the hot path's lookup)
template <int MODE>
__global__ void __launch_bounds__(256) lut16_scan_all_kernel(const uint4* __restrict__ codes, size_t nblocks, int S,
                                                             int SG, const uint8_t* __restrict__ lut8, size_t n,
                                                             uint32_t* __restrict__ sums, uint32_t one) {
  extern __shared__ __align__(16) uint8_t sm[];
  const int S4 = SG * 4;
  for (int e = threadIdx.x; e < S4 * 16; e += blockDim.x) sm[e] = e < S * 16 ? lut8[e] : 0;
  __syncthreads();
  const uint4* lut = reinterpret_cast<const uint4*>(sm);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (size_t b = static_cast<size_t>(blockIdx.x) * 8 + warp; b < nblocks; b += static_cast<size_t>(gridDim.x) * 8) {
    PackedSums ps[1];
    AccMul mul;
    mul.one = one;
    mul.w15 = 0x80000001u;
    scan_block<1, MODE>(codes + b * SG * 32, SG, lut, S4, lane, mul, ps);
    uint32_t s1[8];
    unpack_sums(ps[0], s1);
    size_t p0 = b * kBlockPts + lane * 8;
    for (int i = 0; i < 8; ++i)
      if (p0 + i < n) sums[p0 + i] = s1[i];
  }
}

// Codebook::encode of (x - centre[assign]) + PackedCodes4Bit::from_codes; one thread per output byte.
// argmin with strict < over codes 0..15 (lowest code wins ties), distances sequential and unfused
// (src/hashes/codebook.rs:82-115).
__global__ void pq_encode_kernel(const float* __restrict__ cb, int S, int ds, const float* __restrict__ x, size_t n,
                                 size_t stride, const float* __restrict__ centers,
                                 const uint32_t* __restrict__ assign, uint8_t* __restrict__ packed) {
  const int bpp = (S + 1) / 2;
  size_t t = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= n * bpp) return;
  size_t p = t / bpp;
  int b = static_cast<int>(t - p * bpp);
  const float* row = x + p * stride;
  const float* cen = (centers && assign) ? centers + static_cast<size_t>(assign[p]) * (static_cast<size_t>(S) * ds)
                                         : nullptr;
  uint8_t byte = 0;
  for (int h = 0; h < 2; ++h) {
    int s = 2 * b + h;
    if (s >= S) break;
    float best = __int_as_float(0x7F800000);
    int bi = 0;
    for (int c = 0; c < 16; ++c) {
      float sum = 0.0f;
      for (int j = 0; j < ds; ++j) {
        float v = row[s * ds + j];
        if (cen) v = __fsub_rn(v, cen[s * ds + j]);
        float d = __fsub_rn(v, __ldg(cb + (static_cast<size_t>(s) * 16 + c) * ds + j));
        sum = __fadd_rn(sum, __fmul_rn(d, d));
      }
      if (sum < best) {
        best = sum;
        bi = c;
      }
    }
    byte |= static_cast<uint8_t>((bi & 0x0F) << (4 * h));
  }
  packed[t] = byte;
}

}  // namespace scann

extern "C" {

scann_status scann_lut16_build(const float* codebook, size_t S, size_t ds, const float* queries, size_t nq,
                               const float* centroids, uint8_t* lut8, float* bias, float* mult, int device,
                               int memspace) {
  using namespace scann;
  if (nq == 0) return SCANN_OK;
  SCANN_REQUIRE(codebook && queries && lut8 && bias && mult, SCANN_INVALID_ARGUMENT, "NULL buffer");
  SCANN_REQUIRE(S >= 1 && S <= 256 && ds >= 1, SCANN_INVALID_ARGUMENT, "bad S/ds");
  SCANN_TRY(check_device(device));
  DeviceGuard g(device);
  const size_t dim = S * ds;
  DevBuf<float> d_cb, d_q, d_c, d_bias, d_mult;
  DevBuf<uint8_t> d_lut;
  const bool host = memspace == SCANN_HOST;
  const float *pq = queries, *pc = centroids, *pcb = codebook;
  uint8_t* pl = lut8;
  float *pb = bias, *pm = mult;
  if (host) {
    SCANN_TRY(d_cb.upload(codebook, S * 16 * ds, SCANN_HOST, 0));
    SCANN_TRY(d_q.upload(queries, nq * dim, SCANN_HOST, 0));
    if (centroids) SCANN_TRY(d_c.upload(centroids, nq * dim, SCANN_HOST, 0));
    SCANN_TRY(d_lut.alloc(nq * S * 16));
    SCANN_TRY(d_bias.alloc(nq));
    SCANN_TRY(d_mult.alloc(nq));
    pcb = d_cb.p;
    pq = d_q.p;
    pc = centroids ? d_c.p : nullptr;
    pl = d_lut.p;
    pb = d_bias.p;
    pm = d_mult.p;
  }
  const size_t S4 = (S + 3) / 4 * 4;
  size_t smem = 4 * dim * sizeof(float) + 4 * S4 * 16;
  SCANN_REQUIRE(smem <= 200 * 1024, SCANN_RESOURCE_EXHAUSTED, "dim too large for the LUT tap");
  if (smem > 48 * 1024)
    SCANN_CUDA(cudaFuncSetAttribute(lut16_build_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    static_cast<int>(smem)));
  lut16_build_kernel<<<static_cast<unsigned>((nq + 3) / 4), 128, smem, 0>>>(
      pcb, static_cast<int>(S), static_cast<int>(ds), pq, static_cast<int>(nq), pc, pl, pb, pm);
  SCANN_CUDA(cudaGetLastError());
  if (host) {
    SCANN_CUDA(cudaMemcpy(lut8, pl, nq * S * 16, cudaMemcpyDeviceToHost));
    SCANN_CUDA(cudaMemcpy(bias, pb, nq * 4, cudaMemcpyDeviceToHost));
    SCANN_CUDA(cudaMemcpy(mult, pm, nq * 4, cudaMemcpyDeviceToHost));
  }
  SCANN_CUDA(cudaDeviceSynchronize());
  return SCANN_OK;
}

scann_status scann_lut16_scan(const uint8_t* packed, size_t n, size_t S, const uint8_t* lut8, uint32_t* sums,
                              int device, int memspace) {
  using namespace scann;
  if (n == 0) return SCANN_OK;
  SCANN_REQUIRE(packed && lut8 && sums, SCANN_INVALID_ARGUMENT, "NULL buffer");
  SCANN_REQUIRE(S >= 1 && S <= 256, SCANN_INVALID_ARGUMENT, "num_subspaces %zu outside 1..256", S);
  SCANN_TRY(check_device(device));
  DeviceGuard g(device);
  const bool host = memspace == SCANN_HOST;
  const size_t bpp = (S + 1) / 2, SG = (S + 3) / 4;
  DevBuf<uint8_t> d_packed, d_lut;
  DevBuf<uint32_t> d_codes, d_sums;
  const uint8_t *pp = packed, *pl = lut8;
  uint32_t* ps = sums;
  if (host) {
    SCANN_TRY(d_packed.upload(packed, n * bpp, SCANN_HOST, 0));
    SCANN_TRY(d_lut.upload(lut8, S * 16, SCANN_HOST, 0));
    SCANN_TRY(d_sums.alloc(n));
    pp = d_packed.p;
    pl = d_lut.p;
    ps = d_sums.p;
  }
  const size_t nblocks = (n + kBlockPts - 1) / kBlockPts;
  const size_t words = nblocks * SG * 128;
  SCANN_TRY(d_codes.alloc(words));
  repack_flat_kernel<<<static_cast<unsigned>((words + 255) / 256), 256>>>(pp, n, static_cast<int>(S),
                                                                          static_cast<int>(SG), words, d_codes.p);
  SCANN_CUDA(cudaGetLastError());
  unsigned grid = static_cast<unsigned>(std::min<size_t>((nblocks + 7) / 8, 148 * 8));
  // same accumulation mode as the product path picks for this S (treeah.cu launch_scan_g)
  auto kern = scan_acc_mode(static_cast<int>(S)) == 3 ? lut16_scan_all_kernel<3> : lut16_scan_all_kernel<2>;
  kern<<<grid, 256, SG * 4 * 16>>>(reinterpret_cast<const uint4*>(d_codes.p), nblocks, static_cast<int>(S),
                                   static_cast<int>(SG), pl, n, ps, 1u);
  SCANN_CUDA(cudaGetLastError());
  if (host) SCANN_CUDA(cudaMemcpy(sums, ps, n * 4, cudaMemcpyDeviceToHost));
  SCANN_CUDA(cudaDeviceSynchronize());
  return SCANN_OK;
}

scann_status scann_pq_encode(const float* codebook, size_t S, size_t ds, const float* x, size_t n, size_t stride,
                             const float* centers, const uint32_t* assign, uint8_t* packed, int device,
                             int memspace) {
  using namespace scann;
  if (n == 0) return SCANN_OK;
  SCANN_REQUIRE(codebook && x && packed, SCANN_INVALID_ARGUMENT, "NULL buffer");
  SCANN_REQUIRE((centers == nullptr) == (assign == nullptr), SCANN_INVALID_ARGUMENT,
                "centers and assign go together");
  SCANN_REQUIRE(S >= 1 && S <= 256 && ds >= 1 && stride >= S * ds, SCANN_INVALID_ARGUMENT, "bad S/ds/stride");
  SCANN_REQUIRE(memspace == SCANN_DEVICE || memspace == SCANN_HOST, SCANN_INVALID_ARGUMENT, "bad memspace");
  SCANN_TRY(check_device(device));
  DeviceGuard g(device);
  const size_t bpp = (S + 1) / 2;
  const bool host = memspace == SCANN_HOST;
  DevBuf<float> d_cb, d_x, d_cen;
  DevBuf<uint32_t> d_as;
  DevBuf<uint8_t> d_out;
  const float *pcb = codebook, *px = x, *pcen = centers;
  const uint32_t* pas = assign;
  uint8_t* po = packed;
  if (host) {
    SCANN_REQUIRE(centers == nullptr, SCANN_UNIMPLEMENTED,
                  "host-memory residual encode is not supported; pass device pointers");
    SCANN_TRY(d_cb.upload(codebook, S * 16 * ds, SCANN_HOST, 0));
    SCANN_TRY(d_x.upload(x, n * stride, SCANN_HOST, 0));
    SCANN_TRY(d_out.alloc(n * bpp));
    pcb = d_cb.p;
    px = d_x.p;
    po = d_out.p;
  }
  size_t total = n * bpp;
  pq_encode_kernel<<<static_cast<unsigned>((total + 255) / 256), 256>>>(pcb, static_cast<int>(S), static_cast<int>(ds),
                                                                        px, n, stride, pcen, pas, po);
  SCANN_CUDA(cudaGetLastError());
  if (host) SCANN_CUDA(cudaMemcpy(packed, po, total, cudaMemcpyDeviceToHost));
  SCANN_CUDA(cudaDeviceSynchronize());
  return SCANN_OK;
}

}  // extern "C"
