// BruteForceSearcher<f32> (src/brute_force/searcher.rs:77-208) and ScalarQuantizedBruteForceSearcher
// (src/brute_force/scalar_quantized.rs:168-326) on the GPU.
//
// The reference streams the whole database once per query (one_to_many_* kernels) and pushes N
// distances through a binary heap.  Here a batch is a dense contraction Q x X^T:
//   1. bf_gemm_kernel      128x128x16 register-tiled f32 kernel (8x8 micro-tiles, double-buffered shared
//                          memory; int8 rows are widened while staging).  Fused distance epilogue:
//                          SqL2/L2 -> |q|^2 + |x|^2 - 2 q.x, Dot -> -q.x (negated as the reference does).
//                          Scores go to an L2-resident tile [<=1024 queries][16384 rows].
//   2. bf_select_kernel    per query: exact running top-kc over the tile (threshold filter + radix
//                          select, common.cuh), kc = k + 32 candidates carried between row tiles.
//   3. rescore_topk_kernel exact distance of the kc candidates in the reference's AVX2+FMA order
//                          (bit-identical floats), final order (distance, id), top-k   (select.cu)
// The GEMM scores only rank candidates; every distance that is returned comes from step 3.
//
// Default path for dim <= 256 — tensor cores (tc_gemm.cu: tcgen05.mma bf16, TMEM accumulators, TMA operands):
//   a. DENSE scores v = hx - q~.x~ of a strided sample of <= 16384 rows; per query an upper bound v_k of the k-th
//      smallest sample score (hence of the k-th best over all rows), from a 256-bucket histogram of the row.
//   b. thr[q] = v_k + 2*eps_q, eps_q = a rigorous bound on |v - exact| (bf16 operand rounding: 2^-7 |q| max|x| for f32 rows, 2^-8 for int8 rows,
//      plus f32 accumulation slack).  Any row with v > thr is beaten by the k sample rows whatever the
//      rounding did, so it cannot be among the exact top-k.
//   c. FILTER pass over all rows appends the rows with v <= thr to per-query lists.  From 32768 rows on it runs in two
//      passes: the first eighth of the rows under the sample's bound, then bf_tighten_kernel replaces the bound by
//      (kk-th smallest score among the prefix survivors) + 2*eps — the same argument with real rows in place of sample
//      rows — and the other seven eighths run under it (2.8k -> a few hundred survivors per query at C2).
//   d. rescore_lists_kernel: second certification inside the list (only the rows within 2*eps of the list's k-th
//      smallest score can be in the top-k: k + a few tens), exact distances of those in the reference's AVX2 order,
//      (distance, id) order.
// Results are therefore the exact top-k by the reference's own f32 distances, not "top-k up to GEMM rounding".
// A list overflow (cap 4096: huge k, or massively duplicated rows) sends that query chunk through steps 1-3.  Steps 1-3
// carry k + 32 candidates ranked by an f32 GEMM score without an error-bound argument: exact unless more than 32 rows
// lie within that GEMM's rounding error of the k-th distance (DESIGN.md section 6).
#include <string.h>

#include <algorithm>

#include "kernels.h"

namespace scann {

constexpr int kBM = 128, kBN = 128, kBK = 16;
constexpr int kQTile = 1024;    // queries per score tile
constexpr int kNTile = 16384;   // rows per score tile
constexpr int kBfMargin = 32;   // extra candidates kept beyond k

__global__ void pad_queries_kernel(const float* __restrict__ q, size_t nq, size_t dim, size_t dim_pad, size_t rows_pad,
                                   float* __restrict__ out, float* __restrict__ qn) {
  size_t r = static_cast<size_t>(blockIdx.x) * (blockDim.x / 32) + threadIdx.x / 32;
  int lane = threadIdx.x & 31;
  if (r >= rows_pad) return;
  float s = 0.0f;
  for (size_t d = lane; d < dim_pad; d += 32) {
    float v = (r < nq && d < dim) ? q[r * dim + d] : 0.0f;
    out[r * dim_pad + d] = v;
    s = fmaf(v, v, s);
  }
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, o);
  if (lane == 0) qn[r] = s;
}

// db rows -> compact zero-padded rows [n_pad][dim_pad] (+ squared norms of the values the GEMM sees)
template <bool I8>
__global__ void pad_rows_kernel(const void* __restrict__ src, size_t n, size_t dim, size_t stride, size_t dim_pad,
                                size_t n_pad, void* __restrict__ dst, float* __restrict__ xn, float scale) {
  size_t r = static_cast<size_t>(blockIdx.x) * (blockDim.x / 32) + threadIdx.x / 32;
  int lane = threadIdx.x & 31;
  if (r >= n_pad) return;
  float s = 0.0f;
  for (size_t d = lane; d < dim_pad; d += 32) {
    bool in = r < n && d < dim;
    if (I8) {
      int8_t v = in ? static_cast<const int8_t*>(src)[r * stride + d] : 0;
      static_cast<int8_t*>(dst)[r * dim_pad + d] = v;
      float f = static_cast<float>(v) * scale;
      s = fmaf(f, f, s);
    } else {
      float v = in ? static_cast<const float*>(src)[r * stride + d] : 0.0f;
      static_cast<float*>(dst)[r * dim_pad + d] = v;
      s = fmaf(v, v, s);
    }
  }
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, o);
  if (lane == 0) xn[r] = s;
}

template <bool I8>
__global__ void __launch_bounds__(256) bf_gemm_kernel(const float* __restrict__ A, const void* __restrict__ Bv, int Kd,
                                                      const float* __restrict__ qn, const float* __restrict__ xn,
                                                      float scale, int measure, float* __restrict__ C, int ldc) {
  __shared__ __align__(16) float As[2][kBK][kBM];
  __shared__ __align__(16) float Bs[2][kBK][kBN];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const size_t m0 = static_cast<size_t>(blockIdx.y) * kBM, n0 = static_cast<size_t>(blockIdx.x) * kBN;
  const float* Bf = static_cast<const float*>(Bv);
  const int8_t* Bi = static_cast<const int8_t*>(Bv);

  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.0f;

  // staging registers
  float4 ra[2], rb[2];
  uint4 rbi = make_uint4(0, 0, 0, 0);
  auto gload = [&](int k0) {
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      int idx = tid + i * 256, row = idx >> 2, kq = idx & 3;
      ra[i] = *reinterpret_cast<const float4*>(A + (m0 + row) * Kd + k0 + kq * 4);
      if (!I8) rb[i] = *reinterpret_cast<const float4*>(Bf + (n0 + row) * Kd + k0 + kq * 4);
    }
    if (I8 && tid < kBN) rbi = *reinterpret_cast<const uint4*>(Bi + (n0 + tid) * Kd + k0);
  };
  auto sstore = [&](int buf) {
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      int idx = tid + i * 256, row = idx >> 2, kq = idx & 3;
      As[buf][kq * 4 + 0][row] = ra[i].x;
      As[buf][kq * 4 + 1][row] = ra[i].y;
      As[buf][kq * 4 + 2][row] = ra[i].z;
      As[buf][kq * 4 + 3][row] = ra[i].w;
      if (!I8) {
        Bs[buf][kq * 4 + 0][row] = rb[i].x;
        Bs[buf][kq * 4 + 1][row] = rb[i].y;
        Bs[buf][kq * 4 + 2][row] = rb[i].z;
        Bs[buf][kq * 4 + 3][row] = rb[i].w;
      }
    }
    if (I8 && tid < kBN) {
      const uint32_t w[4] = {rbi.x, rbi.y, rbi.z, rbi.w};
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        int8_t v = static_cast<int8_t>((w[j >> 2] >> (8 * (j & 3))) & 0xFF);
        Bs[buf][j][tid] = static_cast<float>(v);
      }
    }
  };

  const int nk = Kd / kBK;
  gload(0);
  sstore(0);
  __syncthreads();
  for (int kt = 0; kt < nk; ++kt) {
    const int cur = kt & 1;
    if (kt + 1 < nk) gload((kt + 1) * kBK);
#pragma unroll
    for (int kk = 0; kk < kBK; ++kk) {
      const float4 a0 = *reinterpret_cast<const float4*>(&As[cur][kk][ty * 4]);
      const float4 a1 = *reinterpret_cast<const float4*>(&As[cur][kk][64 + ty * 4]);
      const float4 b0 = *reinterpret_cast<const float4*>(&Bs[cur][kk][tx * 4]);
      const float4 b1 = *reinterpret_cast<const float4*>(&Bs[cur][kk][64 + tx * 4]);
      const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    if (kt + 1 < nk) {
      sstore(cur ^ 1);
      __syncthreads();
    }
  }

  // fused distance epilogue
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const size_t m = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
    const float qq = qn[m];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const size_t nb = n0 + (h == 0 ? tx * 4 : 64 + tx * 4);
      float o[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float dot = acc[i][h * 4 + j];
        if (I8) dot *= scale;
        o[j] = (measure == SCANN_DOT) ? -dot : (qq + xn[nb + j] - 2.0f * dot);
      }
      *reinterpret_cast<float4*>(C + m * ldc + nb) = make_float4(o[0], o[1], o[2], o[3]);
    }
  }
}

constexpr int kBfChunk = 2048;

// per query: merge the carried top-kc state with the `ncols` scores of this row tile
__global__ void __launch_bounds__(256) bf_select_kernel(const float* __restrict__ scores, int ldc, int ncols,
                                                        uint32_t row0, uint64_t* __restrict__ state, int have, int kc) {
  extern __shared__ __align__(16) uint8_t sm[];
  const int p2 = next_pow2(kc < 1 ? 1 : kc);
  uint64_t* buf = reinterpret_cast<uint64_t*>(sm);
  uint64_t* out = buf + (kc + kBfChunk);
  uint32_t* hist = reinterpret_cast<uint32_t*>(out + p2);
  const size_t q = blockIdx.x;
  const float* row = scores + q * ldc;
  uint64_t* st = state + q * kc;
  // once kc candidates are carried, nothing >= the current worst can enter
  uint64_t thr0 = (have >= kc) ? st[kc - 1] + 1 : ~0ull;
  auto gen = [&](int i) -> uint64_t {
    if (i < have) return st[i];
    int c = i - have;
    return (static_cast<uint64_t>(f32_key(row[c])) << 32) | (row0 + static_cast<uint32_t>(c));
  };
  int m = block_topr_sorted<256, kBfChunk>(gen, have + ncols, kc, buf, out, hist, thr0);
  __syncthreads();
  for (int j = threadIdx.x; j < kc; j += 256) st[j] = j < m ? out[j] : ~0ull;
}

__global__ void state_to_cand_kernel(const uint64_t* __restrict__ state, size_t total, uint32_t* __restrict__ cand) {
  size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= total) return;
  uint64_t k = state[i];
  cand[i] = k == ~0ull ? 0xFFFFFFFFu : static_cast<uint32_t>(k & 0xFFFFFFFFu);
}


// Steps a+b fused, one warp per query: thr[q] = (upper bound of the k-th smallest sample score) + 2*eps_q.  The bound
// comes from a 256-bucket histogram of the query's sample row (common.cuh warp_kth_upper_bound) — any value >= the
// k-th smallest keeps the certification argument, and it is 4x cheaper than an exact select of the row.
__global__ void __launch_bounds__(256) bf_bound_kernel(const float* __restrict__ dense, int ld, int ncols, int kk,
                                                       const float* __restrict__ qn, float xmax2, size_t nq,
                                                       int rows_i8, float* __restrict__ thr) {
  __shared__ uint32_t s_hist[8][256];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const size_t q = static_cast<size_t>(blockIdx.x) * 8 + warp;
  if (q >= nq) return;
  const float inf = __int_as_float(0x7F800000);
  const float vU = warp_kth_upper_bound(dense + q * ld, ncols, static_cast<uint32_t>(kk), s_hist[warp], lane);
  const float nqr = sqrtf(qn[q]), nx = sqrtf(xmax2);
  const float eps = tc_rank_eps(nqr, nx, rows_i8 != 0);  // common.cuh
  float t = vU + 2.0f * eps;
  t = t + fabsf(t) * 1e-6f;
  if (lane == 0) thr[q] = (t == t) ? t : inf;
}

// Step c', one warp per query, after the FILTER pass over a PREFIX of the rows: the prefix survivors are real rows with
// known scores, so (an upper bound of) the kk-th smallest score among them bounds the kk-th smallest score over all rows
// just like the sample did — and much more tightly (a 1/8 prefix holds ~kk/8-th-quantile rows where the 16384-row sample
// holds the kk/0.016-th).  thr[q] only ever tightens; a list that is short of kk entries or overflowed keeps its bound.
__global__ void __launch_bounds__(256) bf_tighten_kernel(const unsigned long long* __restrict__ lists,
                                                         const uint32_t* __restrict__ cnt, uint32_t cap, int kk,
                                                         const float* __restrict__ qn, float xmax2, size_t nq,
                                                         int rows_i8, float* __restrict__ thr) {
  __shared__ uint32_t s_hist[8][256];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const size_t q = static_cast<size_t>(blockIdx.x) * 8 + warp;
  if (q >= nq) return;
  const uint32_t c = cnt[q];
  if (c < static_cast<uint32_t>(kk) || c > cap) return;
  const unsigned long long* l = lists + q * cap;
  const float vU = warp_kth_upper_bound_of(
      [&](int i) { return key_f32(static_cast<uint32_t>(l[i] >> 32)); }, static_cast<int>(c),
      static_cast<uint32_t>(kk), s_hist[warp], lane);
  const float eps = tc_rank_eps(sqrtf(qn[q]), sqrtf(xmax2), rows_i8 != 0);
  float t = vU + 2.0f * eps;
  t = t + fabsf(t) * 1e-6f;
  if (lane == 0 && t == t && t < thr[q]) thr[q] = t;
}

// radius search: thr[q] in score units so that every row whose exact distance can be <= radius passes the filter
//   SqL2: d <= r  <=>  (d - |q|^2)/2 <= (r - |q|^2)/2;  L2: d <= r^2;  Dot: -q.x <= r
__global__ void bf_radius_thr_kernel(const float* __restrict__ qn, float xmax2, float radius, int measure, size_t nq,
                                     int rows_i8, float* __restrict__ thr) {
  const size_t q = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (q >= nq) return;
  const float nqr = sqrtf(qn[q]), nx = sqrtf(xmax2);
  const float eps = tc_rank_eps(nqr, nx, rows_i8 != 0);
  float t;
  if (measure == SCANN_DOT) t = radius;
  else if (measure == SCANN_L2) t = radius < 0.0f ? -1.0f - qn[q] : 0.5f * (radius * radius * 1.000001f - qn[q]);
  else t = 0.5f * (radius - qn[q]);
  t = t + eps + fabsf(t) * 1e-6f;
  thr[q] = (t == t) ? t : __int_as_float(0x7F800000);
}

__global__ void bf_overflow_kernel(const uint32_t* __restrict__ cnt, size_t nq, uint32_t cap, uint32_t* flag) {
  const size_t q = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (q < nq && cnt[q] > cap) atomicOr(flag, 1u);
}

constexpr size_t kTcQTile = 4096;      // queries per tensor-core chunk
constexpr size_t kTcSampleTiles = 128; // 128-row tiles in the threshold sample (16384 rows)
constexpr size_t kTcCap = 4096;        // candidate list capacity per query
constexpr size_t kTcTwoPassTiles = 256;  // two FILTER passes from 32768 rows on
constexpr size_t kTcTwoPassMaxK = 512;    // ... and while the prefix lists can be expected to hold kk entries

struct BfCore {
  int device = 0;
  size_t n = 0, dim = 0, dim_pad = 0, n_pad = 0;
  int measure = SCANN_SQL2;
  bool i8 = false;
  float scale = 1.0f;
  DevBuf<float> rows_f;   // [n_pad][dim_pad]
  DevBuf<int8_t> rows_i;  // [n_pad][dim_pad]
  DevBuf<float> xn;       // [n_pad]
  // tensor-core ranking operands (tc_gemm.cu)
  bool tc = false;
  DevBuf<uint16_t> rows_bf;  // [tc_rows_pad(n)][tc_kpad(dim)] bf16
  DevBuf<float> hx;          // [tc_rows_pad(n)]
  DevBuf<float> d_small;     // [0] max |x|^2, [1] overflow flag (as u32)
  float xmax2 = 0.0f;
  uint32_t* h_flag = nullptr;  // pinned
  uint64_t stat_tc_chunks = 0, stat_legacy_chunks = 0;
  Workspace ws;
  std::mutex mu;
  StreamOrder order;
  cudaStream_t stream = nullptr;

  scann_status init(const void* db, size_t n_, size_t dim_, size_t stride, int measure_, bool i8_, float scale_,
                    int device_, int memspace) {
    device = device_;
    n = n_;
    dim = dim_;
    measure = measure_;
    i8 = i8_;
    scale = scale_;
    dim_pad = (dim + kBK - 1) / kBK * kBK;
    n_pad = (n + kBN - 1) / kBN * kBN;
    SCANN_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    if (n == 0) return SCANN_OK;
    SCANN_TRY(xn.alloc(n_pad));
    unsigned grid = static_cast<unsigned>((n_pad + 7) / 8);
    if (i8) {
      DevBuf<int8_t> tmp;
      const int8_t* src = static_cast<const int8_t*>(db);
      if (memspace == SCANN_HOST) {
        SCANN_TRY(tmp.upload(src, n * stride, SCANN_HOST, stream));
        src = tmp.p;
      }
      SCANN_TRY(rows_i.alloc(n_pad * dim_pad));
      pad_rows_kernel<true><<<grid, 256, 0, stream>>>(src, n, dim, stride, dim_pad, n_pad, rows_i.p, xn.p, scale);
      SCANN_CUDA(cudaGetLastError());
      SCANN_CUDA(cudaStreamSynchronize(stream));
    } else {
      DevBuf<float> tmp;
      const float* src = static_cast<const float*>(db);
      if (memspace == SCANN_HOST) {
        SCANN_TRY(tmp.upload(src, n * stride, SCANN_HOST, stream));
        src = tmp.p;
      }
      SCANN_TRY(rows_f.alloc(n_pad * dim_pad));
      pad_rows_kernel<false><<<grid, 256, 0, stream>>>(src, n, dim, stride, dim_pad, n_pad, rows_f.p, xn.p, 1.0f);
      SCANN_CUDA(cudaGetLastError());
      SCANN_CUDA(cudaStreamSynchronize(stream));
    }
    const char* no_tc = getenv("SCANN_BF_NO_TC");
    if (tc_supported(dim) && !(no_tc && no_tc[0] == '1')) {
      const size_t kpad = tc_kpad(dim), rpad = tc_rows_pad(n);
      SCANN_TRY(rows_bf.alloc(rpad * kpad));
      SCANN_TRY(hx.alloc(rpad));
      SCANN_TRY(d_small.alloc(2));
      SCANN_TRY(tc_prepare_rows(i8 ? static_cast<const void*>(rows_i.p) : static_cast<const void*>(rows_f.p), i8, n,
                                dim, dim_pad, scale, measure != SCANN_DOT, rows_bf.p, hx.p, d_small.p, stream));
      SCANN_CUDA(cudaMemcpyAsync(&xmax2, d_small.p, sizeof(float), cudaMemcpyDeviceToHost, stream));
      SCANN_CUDA(cudaStreamSynchronize(stream));
      SCANN_CUDA(cudaMallocHost(reinterpret_cast<void**>(&h_flag), sizeof(uint32_t)));
      tc = true;
    }
    return SCANN_OK;
  }

  // ---- legacy CUDA-core chunk (dim > 256, list overflow, SCANN_BF_NO_TC=1): steps 1-3 of the file header ----
  // qsrc: device queries [nqc][dim]; writes device outputs oid/od [nqc][k], oc [nqc]
  scann_status legacy_chunk(const float* qsrc, size_t nqc, size_t k, size_t kc, uint32_t* oid, float* od, uint32_t* oc,
                            cudaStream_t s) {
    const size_t qt = std::min<size_t>(kQTile, (nqc + kBM - 1) / kBM * kBM);
    const size_t nt = std::min<size_t>(kNTile, n_pad);
    float* Apad = ws.take<float>(qt * dim_pad);
    float* qn = ws.take<float>(qt);
    float* scores = ws.take<float>(qt * nt);
    uint64_t* state = ws.take<uint64_t>(qt * kc);
    uint32_t* cand = ws.take<uint32_t>(qt * kc);
    const int p2 = next_pow2(static_cast<int>(kc));
    const size_t sel_smem = (kc + kBfChunk + p2) * 8 + 264 * 4;
    SCANN_CUDA(cudaFuncSetAttribute(bf_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    static_cast<int>(sel_smem)));
    for (size_t q0 = 0; q0 < nqc; q0 += qt) {
      const size_t nq1 = std::min(qt, nqc - q0);
      const size_t rows_pad = (nq1 + kBM - 1) / kBM * kBM;
      const float* q1 = qsrc + q0 * dim;
      pad_queries_kernel<<<static_cast<unsigned>((rows_pad + 7) / 8), 256, 0, s>>>(q1, nq1, dim, dim_pad, rows_pad,
                                                                                   Apad, qn);
      for (size_t r0 = 0; r0 < n; r0 += nt) {
        const size_t ncols = std::min(nt, n - r0);
        const size_t cols_pad = (ncols + kBN - 1) / kBN * kBN;
        dim3 grid(static_cast<unsigned>(cols_pad / kBN), static_cast<unsigned>(rows_pad / kBM));
        if (i8)
          bf_gemm_kernel<true><<<grid, 256, 0, s>>>(Apad, rows_i.p + r0 * dim_pad, static_cast<int>(dim_pad), qn,
                                                    xn.p + r0, scale, measure, scores, static_cast<int>(nt));
        else
          bf_gemm_kernel<false><<<grid, 256, 0, s>>>(Apad, rows_f.p + r0 * dim_pad, static_cast<int>(dim_pad), qn,
                                                     xn.p + r0, 1.0f, measure, scores, static_cast<int>(nt));
        const int have = static_cast<int>(std::min(kc, r0));
        bf_select_kernel<<<static_cast<unsigned>(nq1), 256, sel_smem, s>>>(scores, static_cast<int>(nt),
                                                                           static_cast<int>(ncols),
                                                                           static_cast<uint32_t>(r0), state, have,
                                                                           static_cast<int>(kc));
      }
      SCANN_CUDA(cudaGetLastError());
      state_to_cand_kernel<<<static_cast<unsigned>((nq1 * kc + 255) / 256), 256, 0, s>>>(state, nq1 * kc, cand);
      SCANN_TRY(launch_rescore_topk(rescore_params(q1), cand, nq1, kc, k, oid + q0 * k, od + q0 * k, oc + q0, s));
    }
    ++stat_legacy_chunks;
    return SCANN_OK;
  }
  size_t legacy_need(size_t nqc, size_t kc) const {
    const size_t qt = std::min<size_t>(kQTile, (nqc + kBM - 1) / kBM * kBM);
    const size_t nt = std::min<size_t>(kNTile, n_pad);
    return Workspace::padded(qt * dim_pad * 4) + Workspace::padded(qt * 4) + Workspace::padded(qt * nt * 4) +
           Workspace::padded(qt * kc * 8) + Workspace::padded(qt * kc * 4);
  }

  RescoreParams rescore_params(const float* q) const {
    RescoreParams rp;
    rp.queries = q;
    rp.dim = dim;
    rp.raw = i8 ? nullptr : rows_f.p;
    rp.raw_i8 = i8 ? rows_i.p : nullptr;
    rp.scale = scale;
    rp.stride = dim_pad;
    rp.measure = measure;
    return rp;
  }

  // ---- tensor-core chunk: steps a-d of the file header.  *overflow = 1 when some list overflowed (outputs are then
  // not written and the caller runs legacy_chunk).  Synchronises the stream (the overflow flag is read on the host).
  // the threshold sample is every stride-th 128-row tile over the WHOLE row range (a stride rounded down left the last
  // rows of the array unsampled: sorted data then has its best rows outside the sample and the lists overflow)
  size_t tc_sample_stride() const {
    const size_t tiles = tc_rows_pad(n) / 128;
    return std::max<size_t>(1, (tiles + kTcSampleTiles - 1) / kTcSampleTiles);
  }
  size_t tc_sample_tiles() const {
    const size_t tiles = tc_rows_pad(n) / 128, stride = tc_sample_stride();
    return (tiles + stride - 1) / stride;  // <= kTcSampleTiles; tile (tc_sample_tiles() - 1) * stride is the last one hit
  }
  size_t tc_need(size_t nqc, size_t kk) const {
    const size_t qpad = tc_queries_pad(nqc, dim);
    return Workspace::padded(qpad * tc_kpad(dim) * 2) + Workspace::padded(qpad * 4) +
           Workspace::padded(nqc * tc_sample_tiles() * 128 * 4) +
           Workspace::padded(nqc * 4) * 2 + Workspace::padded(nqc * kTcCap * 8);
  }
  scann_status tc_chunk(const float* qsrc, size_t nqc, size_t k, size_t kk, uint32_t* oid, float* od, uint32_t* oc,
                        cudaStream_t s, bool* overflow) {
    const size_t kpad = tc_kpad(dim), qpad = tc_queries_pad(nqc, dim), rpad = tc_rows_pad(n);
    const size_t tiles = rpad / 128, stiles = tc_sample_tiles(), scols = stiles * 128;
    uint16_t* qbf = ws.take<uint16_t>(qpad * kpad);
    float* qn = ws.take<float>(qpad);
    float* dense = ws.take<float>(nqc * scols);
    float* thr = ws.take<float>(nqc);
    uint32_t* cnt = ws.take<uint32_t>(nqc);
    unsigned long long* lists = ws.take<unsigned long long>(nqc * kTcCap);
    uint32_t* flag = reinterpret_cast<uint32_t*>(d_small.p + 1);
    SCANN_TRY(tc_prepare_queries(qsrc, nqc, dim, i8 ? scale : 1.0f, qbf, qn, s));
    TcScoreParams p;
    p.q_bf16 = qbf;
    p.nq = nqc;
    p.dim = dim;
    p.rows_bf16 = rows_bf.p;
    p.rows_pad_total = rpad;
    p.hx = hx.p;
    p.row0 = 0;
    p.nrows = scols;
    p.tile_stride = tc_sample_stride();  // >= 1; the sample is every tile_stride-th 128-row tile
    p.filter = false;
    p.dense = dense;
    p.ld = scols;
    p.thr = nullptr;
    p.cand = nullptr;
    p.cap = kTcCap;
    p.cand_cnt = nullptr;
    p.sms = sm_count(device);
    SCANN_TRY(launch_tc_scores(p, s));  // a. sample scores
    // b. certified threshold from the sample
    bf_bound_kernel<<<static_cast<unsigned>((nqc + 7) / 8), 256, 0, s>>>(dense, static_cast<int>(scols),
                                                                        static_cast<int>(scols), static_cast<int>(kk),
                                                                        qn, xmax2, nqc, i8 ? 1 : 0, thr);
    SCANN_CUDA(cudaMemsetAsync(cnt, 0, nqc * 4, s));
    SCANN_CUDA(cudaMemsetAsync(flag, 0, 4, s));
    p.nrows = rpad;
    p.tile_stride = 1;
    p.filter = true;
    p.hx_is_zero = measure == SCANN_DOT;
    p.dense = nullptr;
    p.thr = thr;
    p.cand = lists;
    p.cand_cnt = cnt;
    // c. all rows, survivors into the lists — in two passes when the data is large: the first eighth of the rows under
    // the sample's bound, then the rest under the bound its survivors give (4x fewer survivors per query at C2, and the
    // FILTER epilogue's time is what its survivors cost)
    const size_t pre_tiles = (tiles >= kTcTwoPassTiles && kk <= kTcTwoPassMaxK) ? tiles / 8 : 0;
    if (pre_tiles > 0) {
      p.nrows = pre_tiles * 128;
      SCANN_TRY(launch_tc_scores(p, s));
      bf_tighten_kernel<<<static_cast<unsigned>((nqc + 7) / 8), 256, 0, s>>>(
          lists, cnt, static_cast<uint32_t>(kTcCap), static_cast<int>(kk), qn, xmax2, nqc, i8 ? 1 : 0, thr);
      SCANN_CUDA(cudaGetLastError());
      p.row0 = pre_tiles * 128;
      p.nrows = rpad - pre_tiles * 128;
    }
    SCANN_TRY(launch_tc_scores(p, s));
    bf_overflow_kernel<<<static_cast<unsigned>((nqc + 255) / 256), 256, 0, s>>>(cnt, nqc, kTcCap, flag);
    // d. exact re-score (harmless if a list overflowed: the outputs are rewritten by the legacy chunk)
    SCANN_TRY(launch_rescore_lists(rescore_params(qsrc), lists, cnt, nqc, kTcCap, k, n, oid, od, oc, s,
                                   __builtin_huge_valf(), nullptr, qn, xmax2));
    uint32_t f = 0;
    SCANN_TRY(read_flag(s, &f));
    *overflow = f != 0;
    if (!*overflow) ++stat_tc_chunks;
    return SCANN_OK;
  }

  // the device flag (d_small[1]) once the work enqueued on s has finished
  scann_status read_flag(cudaStream_t s, uint32_t* v) {
    SCANN_CUDA(cudaMemcpyAsync(h_flag, d_small.p + 1, 4, cudaMemcpyDeviceToHost, s));
    SCANN_CUDA(cudaStreamSynchronize(s));
    *v = *h_flag;
    return SCANN_OK;
  }

  // BruteForceSearcher::search_radius (searcher.rs:142-167) for a batch: every row with distance <= radius, ascending
  // (distance, id), at most max_results per query.  Tensor-core path only (dim <= 256).
  scann_status search_radius(const float* queries, size_t nq, size_t qdim, float radius, size_t max_results,
                             uint32_t* ids, float* dists, uint32_t* counts, int memspace, void* user_stream) {
    if (nq == 0) return SCANN_OK;
    SCANN_REQUIRE(queries && counts, SCANN_INVALID_ARGUMENT, "NULL buffer");
    std::lock_guard<std::mutex> lock(mu);
    CallScope call(device, order, memspace, user_stream, stream);
    const cudaStream_t s = call.s;
    if (n == 0) {
      if (memspace == SCANN_HOST) memset(counts, 0, nq * sizeof(uint32_t));
      else SCANN_CUDA(cudaMemsetAsync(counts, 0, nq * sizeof(uint32_t), s));
      return SCANN_OK;
    }
    SCANN_REQUIRE(qdim == dim, SCANN_INVALID_ARGUMENT, "Query dimensionality does not match dataset");
    SCANN_REQUIRE(ids && dists && max_results >= 1 && max_results < kTcCap, SCANN_INVALID_ARGUMENT,
                  "max_results must be in 1..%zu", kTcCap - 1);
    SCANN_REQUIRE(tc, SCANN_UNIMPLEMENTED, "radius search runs on the tensor-core path (dim <= 256)");
    const size_t k = max_results;
    const size_t chunk = std::min<size_t>(kTcQTile, nq);
    const size_t kpad = tc_kpad(dim), rpad = tc_rows_pad(n);
    const QueryOut outs[] = {{ids, k * 4}, {dists, k * 4}, {counts, 4}};
    SCANN_TRY(ws.reserve(Workspace::padded(tc_queries_pad(chunk, dim) * kpad * 2) +
                         Workspace::padded(tc_queries_pad(chunk, dim) * 4) + Workspace::padded(chunk * 4) * 2 +
                         Workspace::padded(chunk * kTcCap * 8) + 4096 + staging_bytes(memspace, chunk, dim, outs)));
    // the flag collects every chunk's truncation (the kernels only set bits); every chunk is finished before the
    // truncation is reported: all outputs are written
    uint32_t* flag = reinterpret_cast<uint32_t*>(d_small.p + 1);
    SCANN_CUDA(cudaMemsetAsync(flag, 0, 4, s));
    SCANN_TRY(run_query_chunks(ws, memspace, s, queries, nq, dim, chunk, outs,
                               [&](const float* qsrc, size_t, size_t nqc, void* const* o) -> scann_status {
      uint16_t* qbf = ws.take<uint16_t>(tc_queries_pad(chunk, dim) * kpad);
      float* qn = ws.take<float>(tc_queries_pad(chunk, dim));
      float* thr = ws.take<float>(chunk);
      uint32_t* cnt = ws.take<uint32_t>(chunk);
      unsigned long long* lists = ws.take<unsigned long long>(chunk * kTcCap);
      SCANN_TRY(tc_prepare_queries(qsrc, nqc, dim, i8 ? scale : 1.0f, qbf, qn, s));
      bf_radius_thr_kernel<<<static_cast<unsigned>((nqc + 255) / 256), 256, 0, s>>>(qn, xmax2, radius, measure, nqc, i8 ? 1 : 0, thr);
      SCANN_CUDA(cudaMemsetAsync(cnt, 0, nqc * 4, s));
      TcScoreParams p;
      p.q_bf16 = qbf;
      p.nq = nqc;
      p.dim = dim;
      p.rows_bf16 = rows_bf.p;
      p.rows_pad_total = rpad;
      p.hx = hx.p;
      p.row0 = 0;
      p.nrows = rpad;
      p.filter = true;
      p.hx_is_zero = measure == SCANN_DOT;
      p.dense = nullptr;
      p.ld = 0;
      p.thr = thr;
      p.cand = lists;
      p.cap = kTcCap;
      p.cand_cnt = cnt;
      p.sms = sm_count(device);
      SCANN_TRY(launch_tc_scores(p, s));
      bf_overflow_kernel<<<static_cast<unsigned>((nqc + 255) / 256), 256, 0, s>>>(cnt, nqc, kTcCap, flag);
      return launch_rescore_lists(rescore_params(qsrc), lists, cnt, nqc, kTcCap, k, n, static_cast<uint32_t*>(o[0]),
                                  static_cast<float*>(o[1]), static_cast<uint32_t*>(o[2]), s, radius, flag);
    }));
    uint32_t truncated = 0;
    SCANN_TRY(read_flag(s, &truncated));
    SCANN_REQUIRE(!truncated, SCANN_RESOURCE_EXHAUSTED,
                  "more than max_results = %zu points lie within the radius for some query (results are truncated "
                  "to the nearest ones)", max_results);
    return SCANN_OK;
  }

  scann_status search(const float* queries, size_t nq, size_t qdim, size_t k, uint32_t* ids, float* dists,
                      uint32_t* counts, int memspace, void* user_stream) {
    if (nq == 0) return SCANN_OK;  // searcher.rs:175-177
    SCANN_REQUIRE(queries && counts, SCANN_INVALID_ARGUMENT, "NULL buffer");
    std::lock_guard<std::mutex> lock(mu);
    CallScope call(device, order, memspace, user_stream, stream);
    const cudaStream_t s = call.s;
    if (n == 0) {  // empty dataset -> Ok(vec![]) (searcher.rs:78-80) before any dimension check
      if (memspace == SCANN_HOST) memset(counts, 0, nq * sizeof(uint32_t));
      else SCANN_CUDA(cudaMemsetAsync(counts, 0, nq * sizeof(uint32_t), s));
      return SCANN_OK;
    }
    SCANN_REQUIRE(qdim == dim, SCANN_INVALID_ARGUMENT,
                  "Query dimensionality %zu does not match dataset dimensionality %zu", qdim, dim);
    SCANN_REQUIRE(k >= 1 && ids && dists, SCANN_INVALID_ARGUMENT, "k must be >= 1 and outputs non-NULL");
    const size_t kk = std::min(k, n);                  // k clamped to n (searcher.rs:91)
    const size_t kc = std::min(n, kk + kBfMargin);     // candidates carried per query (legacy path)
    SCANN_REQUIRE(kc <= 2048, SCANN_INVALID_ARGUMENT, "k = %zu too large (max %d)", k, 2048 - kBfMargin);
    // tensor cores when the expected list length (k scaled from the sample to all rows) leaves head-room in the lists
    const bool use_tc = tc && static_cast<double>(kk) * static_cast<double>(tc_rows_pad(n)) /
                                      static_cast<double>(tc_sample_tiles() * 128) <= kTcCap / 2;
    const size_t chunk = std::min<size_t>(use_tc ? kTcQTile : kQTile, nq);
    size_t need = legacy_need(chunk, kc);
    if (use_tc) need = std::max(need, tc_need(chunk, kk));
    const QueryOut outs[] = {{ids, k * 4}, {dists, k * 4}, {counts, 4}};
    SCANN_TRY(ws.reserve(need + staging_bytes(memspace, chunk, dim, outs) + 4096));
    return run_query_chunks(ws, memspace, s, queries, nq, dim, chunk, outs,
                            [&](const float* qsrc, size_t, size_t nqc, void* const* o) -> scann_status {
      uint32_t* oid = static_cast<uint32_t*>(o[0]);
      float* od = static_cast<float*>(o[1]);
      uint32_t* oc = static_cast<uint32_t*>(o[2]);
      const size_t mark = ws.used;
      bool overflow = true;
      if (use_tc) SCANN_TRY(tc_chunk(qsrc, nqc, k, kk, oid, od, oc, s, &overflow));
      if (overflow) {
        ws.used = mark;
        SCANN_TRY(legacy_chunk(qsrc, nqc, k, kc, oid, od, oc, s));
      }
      return SCANN_OK;
    });
  }

  ~BfCore() {
    if (h_flag) cudaFreeHost(h_flag);
    if (stream) cudaStreamDestroy(stream);
  }
};

// ---- scalar quantiser (build helper) -----------------------------------------------------------
// QuantizationStats::from_dataset (src/quantization/mod.rs:77-110): f32 min/max (order-independent, parallel)
__global__ void __launch_bounds__(256) sq8_stats_kernel(const float* __restrict__ db, size_t n, size_t dim,
                                                        size_t stride,
                                                        float* __restrict__ mm /* min,max as ordered u32 */) {
  __shared__ uint32_t s_mn[256], s_mx[256];
  uint32_t mn = 0xFFFFFFFFu, mx = 0;
  const size_t total = n * dim;
  for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    size_t r = i / dim, d = i - r * dim;
    uint32_t kf = f32_key(db[r * stride + d]);
    mn = min(mn, kf);
    mx = max(mx, kf);
  }
  s_mn[threadIdx.x] = mn;
  s_mx[threadIdx.x] = mx;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      s_mn[threadIdx.x] = min(s_mn[threadIdx.x], s_mn[threadIdx.x + o]);
      s_mx[threadIdx.x] = max(s_mx[threadIdx.x], s_mx[threadIdx.x + o]);
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    atomicMin(reinterpret_cast<uint32_t*>(mm), s_mn[0]);
    atomicMax(reinterpret_cast<uint32_t*>(mm) + 1, s_mx[0]);
  }
}

// The f64 sums of QuantizationStats::from_dataset are SEQUENTIAL in the reference (mod.rs:84-94): every add rounds, so
// the result depends on the order and a parallel reduction differs in the last bits — enough to move mean/std by an
// f32 ulp and codes across a rounding boundary.  This kernel replays the reference's order exactly: one thread adds
// the values in row-major order (sum and sum of squares are two independent dependent chains; v*v is exact in f64)
// out of a shared-memory chunk while the other warps stage the next chunk.  Build-time only: ~0.5 s per 128M values.
constexpr int kSeqChunk = 4096;  // 2 x 16 KB of static shared memory
__global__ void __launch_bounds__(256) sq8_seqsum_kernel(const float* __restrict__ db, size_t n, size_t dim,
                                                         size_t stride, double* __restrict__ acc /* sum, sumsq */) {
  __shared__ float buf[2][kSeqChunk];
  const size_t total = n * dim;
  const size_t nchunks = (total + kSeqChunk - 1) / kSeqChunk;
  auto load = [&](size_t c, int b) {  // warps 1..7
    const size_t base = c * kSeqChunk;
    for (int i = threadIdx.x - 32; i < kSeqChunk; i += 224) {
      const size_t e = base + i;
      float v = 0.0f;
      if (e < total) {
        const size_t r = e / dim, d = e - r * dim;
        v = db[r * stride + d];
      }
      buf[b][i] = v;
    }
  };
  if (threadIdx.x >= 32) load(0, 0);
  __syncthreads();
  double sum = 0.0, sq = 0.0;
  for (size_t c = 0; c < nchunks; ++c) {
    const int b = static_cast<int>(c & 1);
    if (threadIdx.x >= 32) {
      if (c + 1 < nchunks) load(c + 1, b ^ 1);
    } else if (threadIdx.x == 0) {
      const size_t left = total - c * kSeqChunk;
      const int m = left < static_cast<size_t>(kSeqChunk) ? static_cast<int>(left) : kSeqChunk;
      const float4* p4 = reinterpret_cast<const float4*>(buf[b]);
      int i = 0;
      for (; i + 4 <= m; i += 4) {
        const float4 v = p4[i >> 2];
        const double a0 = static_cast<double>(v.x), a1 = static_cast<double>(v.y), a2 = static_cast<double>(v.z),
                     a3 = static_cast<double>(v.w);
        sum = __dadd_rn(__dadd_rn(__dadd_rn(__dadd_rn(sum, a0), a1), a2), a3);
        sq = __dadd_rn(__dadd_rn(__dadd_rn(__dadd_rn(sq, __dmul_rn(a0, a0)), __dmul_rn(a1, a1)), __dmul_rn(a2, a2)),
                       __dmul_rn(a3, a3));
      }
      for (; i < m; ++i) {
        const double a0 = static_cast<double>(buf[b][i]);
        sum = __dadd_rn(sum, a0);
        sq = __dadd_rn(sq, __dmul_rn(a0, a0));
      }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    acc[0] = sum;
    acc[1] = sq;
  }
}

// ScalarQuantizer::quantize_value (src/quantization/scalar.rs:162-166)
__global__ void sq8_quantize_kernel(const float* __restrict__ db, size_t n, size_t dim, size_t stride, float mn,
                                    float mx, float inv_scale, int8_t* __restrict__ out) {
  size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n * dim) return;
  size_t r = i / dim, d = i - r * dim;
  float v = db[r * stride + d];
  float c = v;
  if (c < mn) c = mn;
  if (c > mx) c = mx;
  float rr = roundf(__fmul_rn(__fsub_rn(c, mn), inv_scale));
  int qi;
  if (!(rr == rr)) qi = 0;
  else if (rr >= 2147483648.0f) qi = 2147483647;
  else if (rr <= -2147483648.0f) qi = -2147483647 - 1;
  else qi = static_cast<int>(rr);
  qi = min(max(qi, 0), 255);
  out[i] = static_cast<int8_t>(static_cast<uint8_t>(qi));
}

}  // namespace scann

struct scann_bf {
  scann::BfCore core;
};
struct scann_sq8 {
  scann::BfCore core;
};

extern "C" {

scann_status scann_bf_create(const float* db, size_t n, size_t dim, size_t stride, int measure, int device,
                             int memspace, scann_bf** out) {
  using namespace scann;
  SCANN_REQUIRE(out != nullptr, SCANN_INVALID_ARGUMENT, "out is NULL");
  *out = nullptr;
  SCANN_REQUIRE(measure == SCANN_SQL2 || measure == SCANN_L2 || measure == SCANN_DOT, SCANN_UNIMPLEMENTED,
                "distance measure %d is outside the GPU hot path (SqL2, L2, Dot)", measure);
  SCANN_REQUIRE(n == 0 || (db != nullptr && dim > 0 && stride >= dim), SCANN_INVALID_ARGUMENT, "bad dataset arguments");
  SCANN_REQUIRE(n < 0xFFFFFFFFull, SCANN_INVALID_ARGUMENT, "dataset too large for u32 ids");
  SCANN_TRY(check_device(device));
  DeviceGuard g(device);
  scann_bf* h = new scann_bf();
  scann_status st = h->core.init(db, n, dim, stride, measure, false, 1.0f, device, memspace);
  if (st != SCANN_OK) {
    scann_bf_destroy(h);
    return st;
  }
  *out = h;
  return SCANN_OK;
}

scann_status scann_bf_search(scann_bf* h, const float* queries, size_t nq, size_t qdim, size_t k, uint32_t* ids,
                             float* dists, uint32_t* counts, int memspace, void* stream) {
  SCANN_REQUIRE(h != nullptr, SCANN_FAILED_PRECONDITION, "searcher not built");
  return h->core.search(queries, nq, qdim, k, ids, dists, counts, memspace, stream);
}

scann_status scann_bf_search_radius(scann_bf* h, const float* queries, size_t nq, size_t qdim, float radius,
                                    size_t max_results, uint32_t* ids, float* dists, uint32_t* counts, int memspace,
                                    void* stream) {
  SCANN_REQUIRE(h != nullptr, SCANN_FAILED_PRECONDITION, "searcher not built");
  return h->core.search_radius(queries, nq, qdim, radius, max_results, ids, dists, counts, memspace, stream);
}

scann_status scann_bf_path_stats(scann_bf* h, uint64_t* tc_chunks, uint64_t* legacy_chunks) {
  using namespace scann;
  SCANN_REQUIRE(h && tc_chunks && legacy_chunks, SCANN_INVALID_ARGUMENT, "NULL argument");
  std::lock_guard<std::mutex> lock(h->core.mu);
  *tc_chunks = h->core.stat_tc_chunks;
  *legacy_chunks = h->core.stat_legacy_chunks;
  return SCANN_OK;
}

void scann_bf_destroy(scann_bf* h) {
  if (!h) return;
  scann::DeviceGuard g(h->core.device);
  cudaDeviceSynchronize();
  delete h;
}

scann_status scann_sq8_create(const int8_t* codes, size_t n, size_t dim, float scale, int measure, int device,
                              int memspace, scann_sq8** out) {
  using namespace scann;
  SCANN_REQUIRE(out != nullptr, SCANN_INVALID_ARGUMENT, "out is NULL");
  *out = nullptr;
  SCANN_REQUIRE(measure == SCANN_SQL2 || measure == SCANN_L2 || measure == SCANN_DOT, SCANN_UNIMPLEMENTED,
                "distance measure %d is outside the GPU hot path (SqL2, L2, Dot)", measure);
  SCANN_REQUIRE(n == 0 || (codes != nullptr && dim > 0), SCANN_INVALID_ARGUMENT, "bad dataset arguments");
  SCANN_REQUIRE(n < 0xFFFFFFFFull, SCANN_INVALID_ARGUMENT, "dataset too large for u32 ids");
  SCANN_TRY(check_device(device));
  DeviceGuard g(device);
  scann_sq8* h = new scann_sq8();
  scann_status st = h->core.init(codes, n, dim, dim, measure, true, scale, device, memspace);
  if (st != SCANN_OK) {
    scann_sq8_destroy(h);
    return st;
  }
  *out = h;
  return SCANN_OK;
}

scann_status scann_sq8_search(scann_sq8* h, const float* queries, size_t nq, size_t qdim, size_t k, uint32_t* ids,
                              float* dists, uint32_t* counts, int memspace, void* stream) {
  SCANN_REQUIRE(h != nullptr, SCANN_FAILED_PRECONDITION, "searcher not built");
  return h->core.search(queries, nq, qdim, k, ids, dists, counts, memspace, stream);
}

scann_status scann_sq8_path_stats(scann_sq8* h, uint64_t* tc_chunks, uint64_t* legacy_chunks) {
  using namespace scann;
  SCANN_REQUIRE(h && tc_chunks && legacy_chunks, SCANN_INVALID_ARGUMENT, "NULL argument");
  std::lock_guard<std::mutex> lock(h->core.mu);
  *tc_chunks = h->core.stat_tc_chunks;
  *legacy_chunks = h->core.stat_legacy_chunks;
  return SCANN_OK;
}

void scann_sq8_destroy(scann_sq8* h) {
  if (!h) return;
  scann::DeviceGuard g(h->core.device);
  cudaDeviceSynchronize();
  delete h;
}

scann_status scann_sq8_quantize(const float* db, size_t n, size_t dim, size_t stride, int8_t* codes, float* cal4,
                                int device, int memspace) {
  using namespace scann;
  SCANN_REQUIRE(n > 0 && dim > 0, SCANN_INVALID_ARGUMENT, "Cannot quantize empty dataset");  // scalar.rs:199-201
  SCANN_REQUIRE(db && codes && cal4 && stride >= dim, SCANN_INVALID_ARGUMENT, "bad arguments");
  SCANN_TRY(check_device(device));
  DeviceGuard g(device);
  const bool host = memspace == SCANN_HOST;
  DevBuf<float> d_db;
  DevBuf<int8_t> d_codes;
  DevBuf<double> d_acc;
  DevBuf<float> d_mm;
  const float* src = db;
  if (host) {
    SCANN_TRY(d_db.upload(db, n * stride, SCANN_HOST, 0));
    src = d_db.p;
    SCANN_TRY(d_codes.alloc(n * dim));
  }
  SCANN_TRY(d_acc.alloc(2));
  SCANN_TRY(d_mm.alloc(2));
  SCANN_CUDA(cudaMemset(d_acc.p, 0, 2 * sizeof(double)));
  uint32_t init_mm[2] = {0xFFFFFFFFu, 0u};
  SCANN_CUDA(cudaMemcpy(d_mm.p, init_mm, sizeof(init_mm), cudaMemcpyHostToDevice));
  sq8_stats_kernel<<<148 * 4, 256>>>(src, n, dim, stride, d_mm.p);  // min / max (order-independent)
  sq8_seqsum_kernel<<<1, 256>>>(src, n, dim, stride, d_acc.p);                // sums in the reference's order
  SCANN_CUDA(cudaGetLastError());
  double acc[2];
  uint32_t mmk[2];
  SCANN_CUDA(cudaMemcpy(acc, d_acc.p, sizeof(acc), cudaMemcpyDeviceToHost));
  SCANN_CUDA(cudaMemcpy(mmk, d_mm.p, sizeof(mmk), cudaMemcpyDeviceToHost));
  auto unkey = [](uint32_t k) {
    uint32_t u = (k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k;
    float f;
    memcpy(&f, &u, 4);
    return f;
  };
  // Host-side scalar epilogue of QuantizationStats::from_dataset + ScalarQuantizer::calibrate
  // (quantization/mod.rs:96-102, scalar.rs:112-129) on the sequentially accumulated f64 sums: bit-identical to the
  // reference's calibration.
  const double count = static_cast<double>(n) * static_cast<double>(dim);
  const float data_min = unkey(mmk[0]), data_max = unkey(mmk[1]);
  const float mean = static_cast<float>(acc[0] / count);
  const float var = (n * dim > 1) ? static_cast<float>((acc[1] - acc[0] * acc[0] / count) / (count - 1.0)) : 0.0f;
  const float sd = sqrtf(var);
  const float range0 = 3.0f * sd;
  float mn = fmaxf(mean - range0, data_min);
  float mx = fminf(mean + range0, data_max);
  float range = mx - mn;
  float scale = 1.0f, inv_scale = 1.0f;
  if (range > 1e-10f) {
    scale = range / 255.0f;
    inv_scale = 255.0f / range;
  }
  int8_t* dst = host ? d_codes.p : codes;
  size_t total = n * dim;
  sq8_quantize_kernel<<<static_cast<unsigned>((total + 255) / 256), 256>>>(src, n, dim, stride, mn, mx, inv_scale, dst);
  SCANN_CUDA(cudaGetLastError());
  if (host) SCANN_CUDA(cudaMemcpy(codes, dst, total, cudaMemcpyDeviceToHost));
  SCANN_CUDA(cudaDeviceSynchronize());
  float cal[4] = {mn, mx, scale, inv_scale};
  if (host) memcpy(cal4, cal, sizeof(cal));
  else SCANN_CUDA(cudaMemcpy(cal4, cal, sizeof(cal), cudaMemcpyHostToDevice));
  return SCANN_OK;
}

}  // extern "C"
