// TreePartitioner, query side (src/partitioning/tree_partitioner.rs:175-229).
//
// center_dist_kernel: squared-L2 from every query to every centre in the reference's exact order —
// sequential over dimensions, d = q - c, sum += d*d, never fused (compute_center_distances /
// squared_distance, :175-192).  The arithmetic is K*D*3 flops per query (C3: 0.58 MFLOP) so it runs on
// the CUDA cores bit-exactly instead of going through a tensor-core GEMM plus re-score; at a 10k
// batch it is ~1 % of the Tree-AH step.  Layout: centres transposed to [D][K] so consecutive threads
// read consecutive centres (coalesced), 8 queries per CTA staged in shared memory as [D][8] so one
// centre value is reused for 8 queries from two LDS.128.
//
// part_select_kernel: the reference sorts all K (dist, id) pairs with a stable sort and takes the
// first L (:206-222).  Stable order by OrderedFloat == ascending (dist, id), so an exact radix select
// of the L smallest 64-bit keys (f32_key(dist) << 32 | id) followed by a bitonic sort of the winners
// returns the identical token list.
#include <stdlib.h>

#include <algorithm>

#include "kernels.h"

namespace scann {

constexpr int kPartQ = 8;

__global__ void __launch_bounds__(256) center_dist_kernel(const float* __restrict__ centersT, int K, int dim,
                                                          const float* __restrict__ queries, int nq,
                                                          float* __restrict__ out) {
  extern __shared__ __align__(16) float qsT[];  // [dim][8]
  const int q0 = blockIdx.x * kPartQ;
  for (int i = threadIdx.x; i < dim * kPartQ; i += blockDim.x) {
    int d = i / kPartQ, qi = i % kPartQ;
    qsT[i] = (q0 + qi < nq) ? queries[static_cast<size_t>(q0 + qi) * dim + d] : 0.0f;
  }
  __syncthreads();
  const float4* qs4 = reinterpret_cast<const float4*>(qsT);
  for (int c = blockIdx.y * blockDim.x + threadIdx.x; c < K; c += gridDim.y * blockDim.x) {
    float acc[kPartQ];
#pragma unroll
    for (int i = 0; i < kPartQ; ++i) acc[i] = 0.0f;
    for (int d = 0; d < dim; ++d) {
      const float cv = __ldg(centersT + static_cast<size_t>(d) * K + c);
      const float4 a = qs4[d * 2], b = qs4[d * 2 + 1];
      const float qv[kPartQ] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < kPartQ; ++i) {
        float df = __fsub_rn(qv[i], cv);
        acc[i] = __fadd_rn(acc[i], __fmul_rn(df, df));
      }
    }
#pragma unroll
    for (int i = 0; i < kPartQ; ++i)
      if (q0 + i < nq) out[static_cast<size_t>(q0 + i) * K + c] = acc[i];
  }
}

constexpr int kSelChunk = 2048;

__global__ void __launch_bounds__(256) part_select_kernel(const float* __restrict__ dist, int K, int L,
                                                          uint32_t* __restrict__ tokens, float* __restrict__ dists) {
  extern __shared__ __align__(16) uint8_t sm[];
  const int R = L < K ? L : K;
  const int p2 = next_pow2(R < 1 ? 1 : R);
  uint64_t* buf = reinterpret_cast<uint64_t*>(sm);
  uint64_t* out = buf + (R + kSelChunk);
  uint32_t* hist = reinterpret_cast<uint32_t*>(out + p2);
  const size_t q = blockIdx.x;
  const float* row = dist + q * K;
  auto gen = [&](int i) -> uint64_t { return (static_cast<uint64_t>(f32_key(row[i])) << 32) | static_cast<uint32_t>(i); };
  int m = block_topr_sorted<256, kSelChunk>(gen, K, R, buf, out, hist);
  for (int j = threadIdx.x; j < L; j += blockDim.x) {
    if (j < m) {
      uint64_t k = out[j];
      tokens[q * L + j] = static_cast<uint32_t>(k & 0xFFFFFFFFu);
      if (dists) dists[q * L + j] = key_f32(static_cast<uint32_t>(k >> 32));
    } else {
      tokens[q * L + j] = 0xFFFFFFFFu;
      if (dists) dists[q * L + j] = __int_as_float(0x7F800000);
    }
  }
}

// ---- tensor-core centroid scoring (tc_gemm.cu) + exact top-L -------------------------------------------------------
// The north-star shape of this stage: the query x centroid contraction runs on tcgen05 (bf16 operands, f32 TMEM
// accumulators) and produces RANKING scores v = |c|^2/2 - q~.c~ = (|q - c|^2 - |q|^2)/2 + rounding.  One warp per query
// then (1) bounds the L-th smallest score v_L from above with a 256-bucket histogram of the row (vU >= v_L),
// (2) keeps every centre with v <= vU + 2*eps (eps = rigorous
// bound on |v - exact|, as in brute_force.cu: any centre outside the set is beaten by L centres inside it), (3) scores
// the ~L survivors exactly in the reference's sequential un-fused order (tree_partitioner.rs:175-192) and (4) sorts them
// by (distance, id) = the reference's stable sort.  Tokens and distances are bit-identical to the exact kernel's.
constexpr int kPtWarps = 4;      // queries per CTA
constexpr int kPtCap = 512;      // survivors per query held in shared memory (L <= 1024 -> see launch)

__device__ __forceinline__ float exact_center_distance(const float* __restrict__ qs, const float* __restrict__ c,
                                                       int dim) {
  float acc = 0.0f;
  if ((dim & 3) == 0) {
    const float4* c4 = reinterpret_cast<const float4*>(c);
    for (int d = 0; d < dim; d += 4) {
      const float4 x = __ldg(c4 + (d >> 2));
      float df = __fsub_rn(qs[d], x.x);
      acc = __fadd_rn(acc, __fmul_rn(df, df));
      df = __fsub_rn(qs[d + 1], x.y);
      acc = __fadd_rn(acc, __fmul_rn(df, df));
      df = __fsub_rn(qs[d + 2], x.z);
      acc = __fadd_rn(acc, __fmul_rn(df, df));
      df = __fsub_rn(qs[d + 3], x.w);
      acc = __fadd_rn(acc, __fmul_rn(df, df));
    }
  } else {
    for (int d = 0; d < dim; ++d) {
      const float df = __fsub_rn(qs[d], __ldg(c + d));
      acc = __fadd_rn(acc, __fmul_rn(df, df));
    }
  }
  return acc;
}

template <int CAP>
__global__ void __launch_bounds__(kPtWarps * 32) part_tc_select_kernel(
    float* __restrict__ dense, int ld, const float* __restrict__ centers, int K, int dim,
    const float* __restrict__ queries, const float* __restrict__ qn, float cmax2, int nq, int L,
    uint32_t* __restrict__ tokens, float* __restrict__ dists) {
  extern __shared__ __align__(16) uint8_t sm[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q = blockIdx.x * kPtWarps + warp;
  if (q >= nq) return;
  const int P2 = CAP;  // power of two
  uint8_t* base = sm + static_cast<size_t>(warp) * (P2 * 8 + 256 * 4 + P2 * 4 + ((dim + 3) & ~3) * 4);
  uint64_t* keys = reinterpret_cast<uint64_t*>(base);          // [CAP]
  uint32_t* hist = reinterpret_cast<uint32_t*>(keys + P2);     // [256]
  uint32_t* cand = hist + 256;                                 // [CAP]
  float* qs = reinterpret_cast<float*>(cand + P2);             // [dim]
  for (int d = lane; d < dim; d += 32) qs[d] = queries[static_cast<size_t>(q) * dim + d];
  float* row = dense + static_cast<size_t>(q) * ld;
  const int Leff = L < K ? L : K;
  const float inf = __int_as_float(0x7F800000);

  // (1) an upper bound vU >= v_L of the L-th smallest ranking score (256-bucket histogram of the row, common.cuh)
  const float vU = warp_kth_upper_bound(row, K, static_cast<uint32_t>(Leff), hist, lane);
  // (2) certified threshold (same bound as bf_bound_kernel in brute_force.cu)
  const float nqr = sqrtf(qn[q]), nx = sqrtf(cmax2);
  const float eps = tc_rank_eps(nqr, nx, false);
  float thr = vU + 2.0f * eps;
  thr = thr + fabsf(thr) * 1e-6f;
  if (!(thr == thr)) thr = inf;

  // (3) survivors
  int m = 0;
  for (int b0 = 0; b0 < K; b0 += 32) {
    const int i = b0 + lane;
    const bool keep = i < K && !(row[i] > thr);  // NaN scores are kept (scored exactly below)
    const uint32_t bal = __ballot_sync(0xFFFFFFFFu, keep);
    if (keep) {
      const int pos = m + __popc(bal & lanemask_lt());
      if (pos < CAP) cand[pos] = static_cast<uint32_t>(i);
    }
    m += __popc(bal);
  }
  __syncwarp();
  uint32_t* tok = tokens + static_cast<size_t>(q) * L;
  float* dst = dists ? dists + static_cast<size_t>(q) * L : nullptr;
  if (m <= CAP) {
    // (4) exact distances of the survivors, (5) bitonic sort by (distance, id)
    int p2 = 1;
    while (p2 < m) p2 <<= 1;
    for (int j = lane; j < p2; j += 32) {
      uint64_t key = ~0ull;
      if (j < m) {
        const uint32_t id = cand[j];
        const float d = exact_center_distance(qs, centers + static_cast<size_t>(id) * dim, dim);
        key = (static_cast<uint64_t>(f32_key(d)) << 32) | id;
      }
      keys[j] = key;
    }
    __syncwarp();
    for (int kk = 2; kk <= p2; kk <<= 1) {
      for (int j = kk >> 1; j > 0; j >>= 1) {
        for (int i = lane; i < p2; i += 32) {
          const int ixj = i ^ j;
          if (ixj > i) {
            const bool asc = (i & kk) == 0;
            const uint64_t x = keys[i], y = keys[ixj];
            if ((x > y) == asc) {
              keys[i] = y;
              keys[ixj] = x;
            }
          }
        }
        __syncwarp();
      }
    }
    for (int j = lane; j < L; j += 32) {
      const bool ok = j < Leff;
      const uint64_t key = ok ? keys[j] : ~0ull;
      tok[j] = ok ? static_cast<uint32_t>(key & 0xFFFFFFFFu) : 0xFFFFFFFFu;
      if (dst) dst[j] = ok ? key_f32(static_cast<uint32_t>(key >> 32)) : inf;
    }
  } else {
    // more survivors than shared memory holds (massively tied centres): exact distance of every centre into the row,
    // then L rounds of "smallest (distance, id) key above the previous one".  Slow, correct, never on real indices.
    for (int i = lane; i < K; i += 32) row[i] = exact_center_distance(qs, centers + static_cast<size_t>(i) * dim, dim);
    __syncwarp();
    uint64_t last = 0;
    bool first = true;
    for (int j = 0; j < L; ++j) {
      uint64_t best = ~0ull;
      if (j < Leff) {
        for (int i = lane; i < K; i += 32) {
          const uint64_t key = (static_cast<uint64_t>(f32_key(row[i])) << 32) | static_cast<uint32_t>(i);
          if ((first || key > last) && key < best) best = key;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const uint64_t other = __shfl_xor_sync(0xFFFFFFFFu, best, o);
          best = other < best ? other : best;
        }
        last = best;
        first = false;
      }
      if (lane == 0) {
        const bool ok = j < Leff;
        tok[j] = ok ? static_cast<uint32_t>(best & 0xFFFFFFFFu) : 0xFFFFFFFFu;
        if (dst) dst[j] = ok ? key_f32(static_cast<uint32_t>(best >> 32)) : inf;
      }
    }
  }
}

static size_t part_tc_smem(int cap, size_t dim) {
  return static_cast<size_t>(kPtWarps) * (cap * 8 + 256 * 4 + cap * 4 + ((dim + 3) & ~size_t(3)) * 4);
}

static bool part_tc_usable(size_t K, size_t dim) {
  const char* e = getenv("SCANN_PART_NO_TC");
  if (e && e[0] == '1') return false;
  return tc_supported(dim) && K >= 256;  // small K: the exact kernel alone is cheaper than the extra launches
}

static scann_status part_tc_prepare(const float* centers, size_t K, size_t dim, PartTc* out, cudaStream_t s) {
  const size_t kpad = tc_kpad(dim), rpad = tc_rows_pad(K);
  if (out->cbf.n != rpad * kpad) SCANN_TRY(out->cbf.alloc(rpad * kpad));  // kept across CentreScorer::set
  if (out->hx.n != rpad) SCANN_TRY(out->hx.alloc(rpad));
  if (out->small.n != 1) SCANN_TRY(out->small.alloc(1));
  SCANN_TRY(tc_prepare_rows(centers, false, K, dim, dim, 1.0f, true, out->cbf.p, out->hx.p, out->small.p, s));
  SCANN_CUDA(cudaMemcpyAsync(&out->cmax2, out->small.p, sizeof(float), cudaMemcpyDeviceToHost, s));
  SCANN_CUDA(cudaStreamSynchronize(s));
  out->ready = true;
  return SCANN_OK;
}

// scratch (CentreScorer::take_scratch): the bf16 queries, their norms and the dense scores [nq][rpad]
static scann_status launch_partition_tc(const PartTc& tc, const float* centers, size_t K, size_t dim,
                                        const float* queries, size_t nq, size_t L, uint32_t* tokens, float* dists,
                                        uint16_t* qbf, float* qn, float* dense, int sms, cudaStream_t s) {
  if (nq == 0 || L == 0) return SCANN_OK;
  SCANN_REQUIRE(L <= 1024, SCANN_INVALID_ARGUMENT, "partitions_to_search %zu > 1024 unsupported", L);
  const size_t rpad = tc_rows_pad(K);
  SCANN_TRY(tc_prepare_queries(queries, nq, dim, 1.0f, qbf, qn, s));
  TcScoreParams sp;
  sp.q_bf16 = qbf;
  sp.nq = nq;
  sp.dim = dim;
  sp.rows_bf16 = tc.cbf.p;
  sp.rows_pad_total = rpad;
  sp.hx = tc.hx.p;
  sp.row0 = 0;
  sp.nrows = rpad;
  sp.filter = false;
  sp.dense = dense;
  sp.ld = rpad;
  sp.thr = nullptr;
  sp.cand = nullptr;
  sp.cap = 0;
  sp.cand_cnt = nullptr;
  sp.sms = sms;
  SCANN_TRY(launch_tc_scores(sp, s));
  const unsigned grid = static_cast<unsigned>((nq + kPtWarps - 1) / kPtWarps);
  // survivors = L + the centres inside the 2*eps certification band; the band holds hundreds of centres when K is in
  // the tens of thousands, and a list overflow means the slow exact pass over every centre (C5, L = 256: 45 ms per batch)
  if (L <= 128 || (L <= 384 && K <= 16384)) {
    const size_t smem = part_tc_smem(512, dim);
    SCANN_CUDA(cudaFuncSetAttribute(part_tc_select_kernel<512>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    static_cast<int>(smem)));
    part_tc_select_kernel<512><<<grid, kPtWarps * 32, smem, s>>>(dense, static_cast<int>(rpad), centers,
                                                               static_cast<int>(K), static_cast<int>(dim), queries, qn,
                                                               tc.cmax2, static_cast<int>(nq), static_cast<int>(L),
                                                               tokens, dists);
  } else {
    const size_t smem = part_tc_smem(2048, dim);
    SCANN_CUDA(cudaFuncSetAttribute(part_tc_select_kernel<2048>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    static_cast<int>(smem)));
    part_tc_select_kernel<2048><<<grid, kPtWarps * 32, smem, s>>>(dense, static_cast<int>(rpad), centers,
                                                                static_cast<int>(K), static_cast<int>(dim), queries,
                                                                qn, tc.cmax2, static_cast<int>(nq),
                                                                static_cast<int>(L), tokens, dists);
  }
  SCANN_CUDA(cudaGetLastError());
  return SCANN_OK;
}

__global__ void transpose_kernel(const float* __restrict__ in, size_t rows, size_t cols, float* __restrict__ out) {
  __shared__ float tile[32][33];
  size_t c0 = static_cast<size_t>(blockIdx.x) * 32, r0 = static_cast<size_t>(blockIdx.y) * 32;
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    size_t r = r0 + j, c = c0 + threadIdx.x;
    tile[j][threadIdx.x] = (r < rows && c < cols) ? in[r * cols + c] : 0.0f;
  }
  __syncthreads();
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    size_t c = c0 + j, r = r0 + threadIdx.x;
    if (r < rows && c < cols) out[c * rows + r] = tile[threadIdx.x][j];
  }
}

static void launch_transpose(const float* in, size_t rows, size_t cols, float* out, cudaStream_t s) {
  dim3 grid(static_cast<unsigned>((cols + 31) / 32), static_cast<unsigned>((rows + 31) / 32));
  transpose_kernel<<<grid, dim3(32, 8), 0, s>>>(in, rows, cols, out);
}

// centersT: [dim][K] transposed centres; scratch: [nq][K] f32
static scann_status launch_partition(const float* centersT, size_t K, size_t dim, const float* queries, size_t nq,
                                     size_t L, uint32_t* tokens, float* dists, float* scratch, cudaStream_t s) {
  if (nq == 0 || L == 0) return SCANN_OK;
  SCANN_REQUIRE(L <= 1024, SCANN_INVALID_ARGUMENT, "partitions_to_search %zu > 1024 unsupported", L);
  {
    unsigned gy = static_cast<unsigned>((K + 255) / 256);
    if (gy > 64) gy = 64;
    dim3 grid(static_cast<unsigned>((nq + kPartQ - 1) / kPartQ), gy);
    size_t smem = dim * kPartQ * sizeof(float);
    if (smem > 48 * 1024)
      SCANN_CUDA(cudaFuncSetAttribute(center_dist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      static_cast<int>(smem)));
    center_dist_kernel<<<grid, 256, smem, s>>>(centersT, static_cast<int>(K), static_cast<int>(dim), queries,
                                               static_cast<int>(nq), scratch);
    SCANN_CUDA(cudaGetLastError());
  }
  {
    int R = static_cast<int>(L < K ? L : K);
    int p2 = next_pow2(R < 1 ? 1 : R);
    size_t smem = (static_cast<size_t>(R) + kSelChunk + p2) * sizeof(uint64_t) + 264 * sizeof(uint32_t);
    part_select_kernel<<<static_cast<unsigned>(nq), 256, smem, s>>>(scratch, static_cast<int>(K), static_cast<int>(L),
                                                                    tokens, dists);
    SCANN_CUDA(cudaGetLastError());
  }
  return SCANN_OK;
}

scann_status CentreScorer::set(const float* centers, size_t K, size_t dim, int memspace, cudaStream_t s) {
  K_ = K;
  dim_ = dim;
  if (centers_.n != K * dim) SCANN_TRY(centers_.alloc(K * dim));
  if (centersT_.n != K * dim) SCANN_TRY(centersT_.alloc(K * dim));
  SCANN_CUDA(cudaMemcpyAsync(centers_.p, centers, K * dim * sizeof(float), in_kind(memspace), s));
  launch_transpose(centers_.p, K, dim, centersT_.p, s);
  int device = 0;
  SCANN_CUDA(cudaGetDevice(&device));
  sms_ = sm_count(device);
  tc_.ready = false;
  if (part_tc_usable(K, dim)) SCANN_TRY(part_tc_prepare(centers_.p, K, dim, &tc_, s));
  SCANN_CUDA(cudaStreamSynchronize(s));
  return SCANN_OK;
}

CentreScorer::Scratch CentreScorer::take_scratch(Workspace& ws, size_t nq) const {
  Scratch sc;
  if (tc_.ready) {
    const size_t qpad = tc_queries_pad(nq, dim_);
    sc.qbf = ws.take<uint16_t>(qpad * tc_kpad(dim_));
    sc.qn = ws.take<float>(qpad);
  }
  sc.scores = ws.take<float>(nq * (tc_.ready ? tc_rows_pad(K_) : K_));
  return sc;
}

scann_status CentreScorer::select(const float* queries, size_t nq, size_t L, uint32_t* tokens, float* dists,
                                  Workspace& ws, cudaStream_t s) const {
  const Scratch sc = take_scratch(ws, nq);
  SCANN_TRY(ws.check("partition"));
  if (tc_.ready)
    return launch_partition_tc(tc_, centers_.p, K_, dim_, queries, nq, L, tokens, dists, sc.qbf, sc.qn, sc.scores, sms_,
                               s);
  return launch_partition(centersT_.p, K_, dim_, queries, nq, L, tokens, dists, sc.scores, s);
}

}  // namespace scann

// ------------------------------------------------------------------------------------------ C ABI
struct scann_part {
  int device = 0;
  size_t K = 0, dim = 0;
  scann::CentreScorer scorer;
  scann::Workspace ws;
  std::mutex mu;
  scann::StreamOrder order;
  cudaStream_t stream = nullptr;
  ~scann_part() {
    if (stream) cudaStreamDestroy(stream);
  }
};

extern "C" {

scann_status scann_part_create(const float* centers, size_t K, size_t dim, int device, int memspace,
                               scann_part** out) {
  using namespace scann;
  SCANN_REQUIRE(out != nullptr, SCANN_INVALID_ARGUMENT, "out is NULL");
  *out = nullptr;
  SCANN_REQUIRE(centers != nullptr && K > 0 && dim > 0, SCANN_INVALID_ARGUMENT,
                "Cannot partition empty dataset");  // tree_partitioner.rs:49-51
  SCANN_TRY(check_device(device));
  DeviceGuard g(device);
  scann_part* h = new scann_part();
  h->device = device;
  h->K = K;
  h->dim = dim;
  scann_status st;
  if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess)
    st = cuda_fail(cudaGetLastError(), "cudaStreamCreate", __FILE__, __LINE__);
  else
    st = h->scorer.set(centers, K, dim, memspace, h->stream);
  if (st != SCANN_OK) {
    scann_part_destroy(h);
    return st;
  }
  *out = h;
  return SCANN_OK;
}

scann_status scann_part_update(scann_part* h, const float* centers, int memspace) {
  using namespace scann;
  SCANN_REQUIRE(h != nullptr, SCANN_FAILED_PRECONDITION, "Partitioner not built");
  SCANN_REQUIRE(centers != nullptr, SCANN_INVALID_ARGUMENT, "NULL buffer");
  std::lock_guard<std::mutex> lock(h->mu);
  DeviceGuard g(h->device);
  if (memspace == SCANN_DEVICE) SCANN_CUDA(cudaDeviceSynchronize());  // the caller's array was produced on another stream
  return h->scorer.set(centers, h->K, h->dim, memspace, h->stream);
}

scann_status scann_part_select(scann_part* h, const float* queries, size_t nq, size_t qdim, size_t L,
                               uint32_t* tokens, float* dists, int memspace, void* stream) {
  using namespace scann;
  SCANN_REQUIRE(h != nullptr, SCANN_FAILED_PRECONDITION, "Partitioner not built");  // tree_partitioner.rs:197-198
  if (nq == 0 || L == 0) return SCANN_OK;
  SCANN_REQUIRE(queries && tokens, SCANN_INVALID_ARGUMENT, "NULL buffer");
  SCANN_REQUIRE(qdim == h->dim, SCANN_INVALID_ARGUMENT, "Query dimensionality %zu does not match dataset dimensionality %zu",
                qdim, h->dim);
  SCANN_REQUIRE(L <= 1024, SCANN_INVALID_ARGUMENT, "partitions_to_search %zu > 1024 unsupported", L);
  std::lock_guard<std::mutex> lock(h->mu);
  CallScope call(h->device, h->order, memspace, stream, h->stream);
  // bounded scratch: process the batch in chunks of queries
  size_t chunk = (size_t(2) << 30) / (h->K * sizeof(float));  // dense score scratch: 2 GiB keeps >= 8192 rows per pass at K = 65,536
  if (chunk < 1) chunk = 1;
  if (chunk > nq) chunk = nq;
  const QueryOut outs[] = {{tokens, L * sizeof(uint32_t)}, {dists, L * sizeof(float)}};
  SCANN_TRY(h->ws.reserve(Workspace::count([&](Workspace& w) {
    take_staging(w, memspace, chunk, h->dim, outs);
    h->scorer.take_scratch(w, chunk);
  })));
  return run_query_chunks(h->ws, memspace, call.s, queries, nq, h->dim, chunk, outs,
                          [&](const float* q, size_t, size_t nqc, void* const* o) {
                            return h->scorer.select(q, nqc, L, static_cast<uint32_t*>(o[0]), static_cast<float*>(o[1]),
                                                    h->ws, call.s);
                          });
}

void scann_part_destroy(scann_part* h) {
  if (!h) return;
  scann::DeviceGuard g(h->device);
  cudaDeviceSynchronize();
  delete h;
}

}  // extern "C"
