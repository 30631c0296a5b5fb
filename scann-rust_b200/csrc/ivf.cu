// The Scann façade's two tree modes that score every member of the probed leaves (SURVEY §8a a13, §8f-2/3):
//   Scann::search_partitioned (src/scann.rs:215-253)  exact distance of every member of the L closest leaves,
//                                                     stable sort by distance, first k
//   Scann::search_tree_ah     (src/scann.rs:256-294)  "variant B": ONE f32 LookupTable of the un-centred query
//                                                     (src/hashes/lut.rs:47-82) over byte codes indexed by datapoint
//                                                     id, every member of the L leaves, stable sort, first k;
//                                                     with K = 1 this is AsymmetricHasher::search's scoring
//                                                     (src/hashes/hasher.rs:162-185)
// plus ReorderingHelper::reorder (src/utils/reordering.rs:23-54) of the k results.
//
// One CTA per query streams the concatenated member lists of its leaves:
//   exact mode: 8 adjacent lanes score one member in the reference's AVX2+FMA lane order (common.cuh
//               exact_pair_distance: lane-wise FMA, the fixed hsum tree, un-fused scalar tail), so the value is
//               bit-identical to x86.rs:72-165 and every load is a full 32-byte sector of the member's row;
//   LUT mode  : a thread per member — 16-byte loads of its code row, sequential f32 sum of S table entries, the table
//               in shared memory.
// (exact_pair_distance_1t, the single-thread restatement of the same order, re-scores the k results for `reorder`.)
// Keys (ordered distance << 32 | position in the concatenated candidate list) go through the block-wide streaming
// top-k (common.cuh); ascending keys = the reference's stable sort by distance.
// Bound: HBM (exact mode gathers D*4-byte rows: Σ|leaf| * D * 4 B per query; LUT mode S bytes per member).
#include <algorithm>

#include "kernels.h"

namespace scann {

namespace {

constexpr int kIvfChunk = 2048;

// x86.rs:72-96 (dot), :139-165 (sqL2), hsum :31-44 — single-thread restatement of the 8-lane kernel
__device__ __forceinline__ float exact_pair_distance_1t(const float* __restrict__ q, const float* __restrict__ x,
                                                        int dim, int measure, bool vec) {
  float acc[8];
#pragma unroll
  for (int l = 0; l < 8; ++l) acc[l] = 0.0f;
  const int chunks = dim >> 3;
  for (int i = 0; i < chunks; ++i) {
    float xv[8];
    if (vec) {  // rows 16-byte aligned (stride % 4 == 0)
      const float4 x0 = __ldg(reinterpret_cast<const float4*>(x + i * 8));
      const float4 x1 = __ldg(reinterpret_cast<const float4*>(x + i * 8 + 4));
      xv[0] = x0.x, xv[1] = x0.y, xv[2] = x0.z, xv[3] = x0.w, xv[4] = x1.x, xv[5] = x1.y, xv[6] = x1.z, xv[7] = x1.w;
    } else {
#pragma unroll
      for (int l = 0; l < 8; ++l) xv[l] = __ldg(x + i * 8 + l);
    }
#pragma unroll
    for (int l = 0; l < 8; ++l) {
      const float a = q[i * 8 + l];
      if (measure == SCANN_DOT) {
        acc[l] = fmaf(a, xv[l], acc[l]);
      } else {
        const float d = __fsub_rn(a, xv[l]);
        acc[l] = fmaf(d, d, acc[l]);
      }
    }
  }
  // ((a0+a4)+(a1+a5)) + ((a2+a6)+(a3+a7))
  const float t0 = __fadd_rn(acc[0], acc[4]), t1 = __fadd_rn(acc[1], acc[5]);
  const float t2 = __fadd_rn(acc[2], acc[6]), t3 = __fadd_rn(acc[3], acc[7]);
  float r = __fadd_rn(__fadd_rn(t0, t1), __fadd_rn(t2, t3));
  for (int j = chunks * 8; j < dim; ++j) {
    const float a = q[j], b = __ldg(x + j);
    if (measure == SCANN_DOT) {
      r = __fadd_rn(r, __fmul_rn(a, b));
    } else {
      const float d = __fsub_rn(a, b);
      r = __fadd_rn(r, __fmul_rn(d, d));
    }
  }
  if (measure == SCANN_DOT) return -r;
  if (measure == SCANN_L2) return __fsqrt_rn(r);
  return r;
}

struct IvfArgs {
  const uint32_t* tokens;   // [nq][L]
  const uint64_t* pt_off;   // [K+1]
  const uint32_t* ids;      // [n] grouped by partition
  const float* raw;         // [N][stride] or null
  size_t stride;
  const float* queries;     // [nq][dim]
  const float* codebook;    // [S][C][ds] or null
  const uint8_t* codes;     // [N][S] by datapoint id, or null
  int dim, L, k, measure, lut_mode, S, C, ds;
  uint32_t K;
  int reorder_measure;      // >= 0: re-score the k results exactly and re-sort (ReorderingHelper::reorder)
  uint32_t* out_ids;
  float* out_dists;
  uint32_t* out_counts;
};

__global__ void __launch_bounds__(256) ivf_topk_kernel(const IvfArgs a) {
  extern __shared__ __align__(16) uint8_t sm[];
  const int p2 = next_pow2(a.k < 1 ? 1 : a.k);
  uint64_t* buf = reinterpret_cast<uint64_t*>(sm);               // [k + chunk]
  uint64_t* out = buf + (a.k + kIvfChunk);                       // [p2]
  uint32_t* hist = reinterpret_cast<uint32_t*>(out + p2);        // [264]
  uint32_t* prefix = hist + 264;                                 // [L + 1]
  float* qs = reinterpret_cast<float*>(prefix + (a.L + 1));      // [dim]
  float* lut = qs + ((a.dim + 3) & ~3);                          // [S * C] (LUT mode)
  const int tid = threadIdx.x;
  const size_t q = blockIdx.x;
  for (int d = tid; d < a.dim; d += 256) qs[d] = a.queries[q * a.dim + d];
  for (int r = tid; r < a.L; r += 256) {
    const uint32_t leaf = a.tokens[q * a.L + r];
    prefix[r + 1] = leaf < a.K ? static_cast<uint32_t>(a.pt_off[leaf + 1] - a.pt_off[leaf]) : 0u;
  }
  __syncthreads();
  if (tid == 0) {
    prefix[0] = 0;
    for (int r = 0; r < a.L; ++r) prefix[r + 1] += prefix[r];
  }
  if (a.lut_mode) {  // LookupTable::from_query: sequential un-fused squared distance to every centroid
    for (int e = tid; e < a.S * a.C; e += 256) {
      const int s = e / a.C;
      float sum = 0.0f;
      for (int j = 0; j < a.ds; ++j) {
        const float d = __fsub_rn(qs[s * a.ds + j], __ldg(a.codebook + static_cast<size_t>(e) * a.ds + j));
        sum = __fadd_rn(sum, __fmul_rn(d, d));
      }
      lut[e] = sum;
    }
  }
  __syncthreads();
  const int total = static_cast<int>(prefix[a.L]);
  const bool vec = (a.stride & 3) == 0 && (reinterpret_cast<uintptr_t>(a.raw) & 15) == 0;
  auto member = [&](int i) -> uint32_t {
    int lo = 0, hi = a.L;  // largest r with prefix[r] <= i
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (prefix[mid] <= static_cast<uint32_t>(i)) lo = mid;
      else hi = mid;
    }
    const uint32_t leaf = a.tokens[q * a.L + lo];
    return a.ids[a.pt_off[leaf] + (static_cast<uint32_t>(i) - prefix[lo])];
  };
  int cur = 0;  // leaf rank of this thread's previous candidate: block_topr_sorted calls gen with increasing i
  auto gen = [&](int i) -> uint64_t {
    while (cur + 1 < a.L && prefix[cur + 1] <= static_cast<uint32_t>(i)) ++cur;
    const uint32_t id = a.ids[a.pt_off[a.tokens[q * a.L + cur]] + (static_cast<uint32_t>(i) - prefix[cur])];
    float d;
    if (a.lut_mode) {
      // LookupTable::compute_distance: sum += distances[s][code_s] for s = 0..S-1, in that order.  The code row is
      // fetched with the widest aligned loads available (one byte load per subspace made the kernel LSU-bound).
      const uint8_t* c = a.codes + static_cast<size_t>(id) * a.S;
      d = 0.0f;
      auto add4 = [&](uint32_t w, int s0) {
#pragma unroll
        for (int j = 0; j < 4; ++j) d = __fadd_rn(d, lut[(s0 + j) * a.C + ((w >> (8 * j)) & 0xFFu)]);
      };
      if ((a.S & 15) == 0) {
        for (int s0 = 0; s0 < a.S; s0 += 16) {
          const uint4 w = __ldg(reinterpret_cast<const uint4*>(c + s0));
          add4(w.x, s0);
          add4(w.y, s0 + 4);
          add4(w.z, s0 + 8);
          add4(w.w, s0 + 12);
        }
      } else if ((a.S & 3) == 0) {
        for (int s0 = 0; s0 < a.S; s0 += 4) add4(__ldg(reinterpret_cast<const uint32_t*>(c + s0)), s0);
      } else {
        for (int s = 0; s < a.S; ++s) d = __fadd_rn(d, lut[s * a.C + c[s]]);
      }
    } else {
      d = exact_pair_distance_1t(qs, a.raw + static_cast<size_t>(id) * a.stride, a.dim, a.measure, vec);
    }
    return (static_cast<uint64_t>(f32_key(d)) << 32) | static_cast<uint32_t>(i);
  };
  int m;
  if (a.lut_mode) {
    m = block_topr_sorted<256, kIvfChunk>(gen, total, a.k, buf, out, hist);
  } else {
    // exact mode: 8 lanes per member read its row as full 32-byte sectors (x86.rs lane order, common.cuh
    // exact_pair_distance) — a thread per member touched twice as many sectors with a quarter of the loads in flight
    int cur8 = 0;
    auto gen8 = [&](int i, int sub) -> uint64_t {
      while (cur8 + 1 < a.L && prefix[cur8 + 1] <= static_cast<uint32_t>(i)) ++cur8;
      const uint32_t id = a.ids[a.pt_off[a.tokens[q * a.L + cur8]] + (static_cast<uint32_t>(i) - prefix[cur8])];
      const float d = exact_pair_distance<false>(qs, a.raw + static_cast<size_t>(id) * a.stride, a.dim, a.measure, 0.0f, sub);
      return (static_cast<uint64_t>(f32_key(d)) << 32) | static_cast<uint32_t>(i);
    };
    m = block_topr_sorted_grouped<256, kIvfChunk, 8>(gen8, total, a.k, buf, out, hist);
  }
  // out[0..m): ascending (distance, candidate position) keys
  if (a.reorder_measure >= 0 && a.raw != nullptr) {
    for (int j = tid; j < p2; j += 256) {
      uint64_t key = ~0ull;
      if (j < m) {
        const uint32_t id = member(static_cast<int>(out[j] & 0xFFFFFFFFu));
        const float d = exact_pair_distance_1t(qs, a.raw + static_cast<size_t>(id) * a.stride, a.dim, a.reorder_measure, vec);
        key = (static_cast<uint64_t>(f32_key(d)) << 32) | static_cast<uint32_t>(j);  // ties keep the previous order
        buf[j] = id;
      }
      out[j] = key;
    }
    __syncthreads();
    block_bitonic_sort<256>(out, p2);
    for (int j = tid; j < a.k; j += 256) {
      const bool ok = j < m;
      a.out_ids[q * a.k + j] = ok ? static_cast<uint32_t>(buf[out[j] & 0xFFFFFFFFu]) : 0xFFFFFFFFu;
      a.out_dists[q * a.k + j] = ok ? key_f32(static_cast<uint32_t>(out[j] >> 32)) : __int_as_float(0x7F800000);
    }
  } else {
    for (int j = tid; j < a.k; j += 256) {
      const bool ok = j < m;
      a.out_ids[q * a.k + j] = ok ? member(static_cast<int>(out[j] & 0xFFFFFFFFu)) : 0xFFFFFFFFu;
      a.out_dists[q * a.k + j] = ok ? key_f32(static_cast<uint32_t>(out[j] >> 32)) : __int_as_float(0x7F800000);
    }
  }
  if (tid == 0) a.out_counts[q] = static_cast<uint32_t>(m);
}

}  // namespace

}  // namespace scann

// create-time validation: every member id must index the per-datapoint arrays (raw rows / codes).  The reference skips
// such entries through dataset.get(idx); a malformed index is refused here instead of read out of bounds by the kernels.
__global__ void ids_in_range_kernel(const uint32_t* __restrict__ ids, size_t n, uint32_t limit, uint32_t* __restrict__ bad) {
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n && ids[i] >= limit) atomicAdd(bad, 1u);
}

struct scann_ivf {
  int device = 0;
  size_t K = 0, dim = 0, n = 0, num_raw = 0, stride = 0, S = 0, C = 0, ds = 0;
  scann::CentreScorer part;
  scann::DevBuf<float> raw, codebook;
  scann::DevBuf<uint32_t> ids;
  scann::DevBuf<uint64_t> pt_off;
  scann::DevBuf<uint8_t> codes;
  scann::Workspace ws;
  std::mutex mu;
  scann::StreamOrder order;
  cudaStream_t stream = nullptr;
  ~scann_ivf() {
    if (stream) cudaStreamDestroy(stream);
  }
};

extern "C" {

void scann_ivf_destroy(scann_ivf* h) {
  if (!h) return;
  scann::DeviceGuard g(h->device);
  cudaDeviceSynchronize();
  delete h;
}

scann_status scann_ivf_create(const float* centers, size_t K, size_t dim, const uint32_t* ids,
                              const uint64_t* part_offsets, size_t n, const float* raw, size_t num_raw, size_t stride,
                              const float* codebook, size_t S, size_t C, const uint8_t* codes_by_id, int device,
                              int memspace, scann_ivf** out) {
  using namespace scann;
  SCANN_REQUIRE(out != nullptr, SCANN_INVALID_ARGUMENT, "out is NULL");
  *out = nullptr;
  SCANN_REQUIRE(centers && K > 0 && dim > 0 && ids && part_offsets, SCANN_INVALID_ARGUMENT, "bad index arguments");
  SCANN_REQUIRE(n > 0, SCANN_INVALID_ARGUMENT, "Dataset cannot be empty");  // scann.rs:66-68
  SCANN_REQUIRE(raw == nullptr || stride >= dim, SCANN_INVALID_ARGUMENT, "stride < dim");
  SCANN_REQUIRE((codebook == nullptr) == (codes_by_id == nullptr), SCANN_INVALID_ARGUMENT,
                "codebook and codes go together");
  if (codebook) {
    SCANN_REQUIRE(S >= 1 && C >= 1 && C <= 256, SCANN_INVALID_ARGUMENT, "bad codebook shape");
    SCANN_REQUIRE(dim % S == 0, SCANN_INVALID_ARGUMENT, "Dimensionality %zu must be divisible by num_subspaces %zu",
                  dim, S);  // codebook.rs:154-159
    SCANN_REQUIRE(S * C * 4 <= 160 * 1024, SCANN_RESOURCE_EXHAUSTED, "lookup table of %zu x %zu floats does not fit",
                  S, C);
  }
  SCANN_TRY(check_device(device));
  DeviceGuard g(device);
  scann_ivf* h = new scann_ivf();
  h->device = device;
  h->K = K;
  h->dim = dim;
  h->n = n;
  h->num_raw = num_raw;
  h->stride = stride;
  h->S = codebook ? S : 0;
  h->C = codebook ? C : 0;
  h->ds = codebook ? dim / S : 0;
  scann_status st = SCANN_OK;
  do {
    if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) {
      st = cuda_fail(cudaGetLastError(), "cudaStreamCreate", __FILE__, __LINE__);
      break;
    }
    cudaStream_t s = h->stream;
    std::vector<uint64_t> off(K + 1);
    if (memspace == SCANN_HOST) {
      std::copy(part_offsets, part_offsets + K + 1, off.begin());
    } else if (cudaMemcpy(off.data(), part_offsets, (K + 1) * 8, cudaMemcpyDeviceToHost) != cudaSuccess) {
      st = cuda_fail(cudaGetLastError(), "copy part_offsets", __FILE__, __LINE__);
      break;
    }
    bool okoff = off[0] == 0 && off[K] == n;
    for (size_t l = 0; l < K && okoff; ++l) okoff = off[l] <= off[l + 1];
    if (!okoff) {
      set_error("part_offsets must be non-decreasing from 0 to n");
      st = SCANN_INVALID_ARGUMENT;
      break;
    }
    if ((st = h->part.set(centers, K, dim, memspace, s)) != SCANN_OK) break;
    if ((st = h->ids.upload(ids, n, memspace, s)) != SCANN_OK) break;
    if ((st = h->pt_off.upload(off.data(), K + 1, SCANN_HOST, s)) != SCANN_OK) break;
    if (raw && (st = h->raw.upload(raw, num_raw * stride, memspace, s)) != SCANN_OK) break;
    if (codebook) {
      if ((st = h->codebook.upload(codebook, S * C * h->ds, memspace, s)) != SCANN_OK) break;
      if ((st = h->codes.upload(codes_by_id, num_raw * S, memspace, s)) != SCANN_OK) break;
    }
    if ((raw || codebook) && n > 0) {
      scann::DevBuf<uint32_t> bad;
      if ((st = bad.alloc(1)) != SCANN_OK) break;
      cudaMemsetAsync(bad.p, 0, 4, s);
      ids_in_range_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, s>>>(h->ids.p, n, static_cast<uint32_t>(
          std::min<size_t>(num_raw, 0xFFFFFFFFull)), bad.p);
      uint32_t nbad = 0;
      if (cudaMemcpyAsync(&nbad, bad.p, 4, cudaMemcpyDeviceToHost, s) != cudaSuccess || cudaStreamSynchronize(s) != cudaSuccess) {
        st = cuda_fail(cudaGetLastError(), "ivf_create id check", __FILE__, __LINE__);
        break;
      }
      if (nbad != 0) {
        set_error("%u member ids are >= the %zu datapoints of the dataset", nbad, num_raw);
        st = SCANN_INVALID_ARGUMENT;
        break;
      }
    }
    if (cudaStreamSynchronize(s) != cudaSuccess || cudaGetLastError() != cudaSuccess) {
      st = cuda_fail(cudaGetLastError(), "ivf_create sync", __FILE__, __LINE__);
      break;
    }
  } while (0);
  if (st != SCANN_OK) {
    scann_ivf_destroy(h);
    return st;
  }
  *out = h;
  return SCANN_OK;
}

// mode 0 = Scann::search_partitioned (exact `measure`), mode 1 = Scann::search_tree_ah (f32 LUT);
// reorder_measure >= 0 re-scores the k results exactly (Scann::search_impl :198-209), -1 = off
scann_status scann_ivf_search(scann_ivf* h, int mode, const float* queries, size_t nq, size_t qdim, size_t L, size_t k,
                              int measure, int reorder_measure, uint32_t* ids, float* dists, uint32_t* counts,
                              int memspace, void* stream) {
  using namespace scann;
  SCANN_REQUIRE(h != nullptr, SCANN_FAILED_PRECONDITION, "searcher not built");
  if (nq == 0) return SCANN_OK;
  SCANN_REQUIRE(queries && ids && dists && counts, SCANN_INVALID_ARGUMENT, "NULL buffer");
  SCANN_REQUIRE(qdim == h->dim, SCANN_INVALID_ARGUMENT,
                "Query dimensionality %zu does not match dataset dimensionality %zu", qdim, h->dim);
  SCANN_REQUIRE(L >= 1 && L <= 1024, SCANN_INVALID_ARGUMENT, "partitions_to_search %zu outside 1..1024", L);
  SCANN_REQUIRE(k >= 1 && k <= 2048, SCANN_INVALID_ARGUMENT, "k %zu outside 1..2048", k);
  SCANN_REQUIRE(mode == 0 || mode == 1, SCANN_INVALID_ARGUMENT, "mode must be 0 (partitioned) or 1 (tree-ah)");
  SCANN_REQUIRE(measure == SCANN_SQL2 || measure == SCANN_L2 || measure == SCANN_DOT, SCANN_UNIMPLEMENTED,
                "distance measure %d is outside the GPU hot path (SqL2, L2, Dot)", measure);
  if (mode == 0) SCANN_REQUIRE(h->raw.p != nullptr, SCANN_FAILED_PRECONDITION, "Dataset not stored");
  if (mode == 1) SCANN_REQUIRE(h->codes.p != nullptr, SCANN_FAILED_PRECONDITION, "index has no hasher");
  if (reorder_measure >= 0) SCANN_REQUIRE(h->raw.p != nullptr, SCANN_FAILED_PRECONDITION, "Dataset not stored");
  std::lock_guard<std::mutex> lock(h->mu);
  CallScope call(h->device, h->order, memspace, stream, h->stream);
  const size_t K = h->K;
  if (L > K) L = K;
  size_t chunk = std::min(nq, std::max<size_t>(1, (size_t(256) << 20) / (K * 4)));
  const size_t scr = h->part.scratch_bytes(chunk);
  const QueryOut outs[] = {{ids, k * 4}, {dists, k * 4}, {counts, 4}};
  SCANN_TRY(h->ws.reserve(Workspace::padded(scr) + Workspace::padded(chunk * L * 4) + 4096 +
                          staging_bytes(memspace, chunk, h->dim, outs)));
  const int p2 = next_pow2(static_cast<int>(k));
  const size_t smem = (k + kIvfChunk + p2) * 8 + 264 * 4 + (L + 1) * 4 + ((h->dim + 3) & ~size_t(3)) * 4 +
                      (mode == 1 ? h->S * h->C * 4 : 0) + 16;
  SCANN_REQUIRE(smem <= 227 * 1024, SCANN_RESOURCE_EXHAUSTED, "search needs %zu B of shared memory", smem);
  SCANN_CUDA(cudaFuncSetAttribute(ivf_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  return run_query_chunks(h->ws, memspace, call.s, queries, nq, h->dim, chunk, outs,
                          [&](const float* dq, size_t, size_t nqc, void* const* o) -> scann_status {
                            void* scratch = h->ws.take<uint8_t>(scr);
                            uint32_t* tokens = h->ws.take<uint32_t>(chunk * L);
                            SCANN_TRY(h->part.select(dq, nqc, L, tokens, nullptr, scratch, call.s));
                            IvfArgs a;
                            a.tokens = tokens;
                            a.pt_off = h->pt_off.p;
                            a.ids = h->ids.p;
                            a.raw = h->raw.p;
                            a.stride = h->stride;
                            a.queries = dq;
                            a.codebook = h->codebook.p;
                            a.codes = h->codes.p;
                            a.dim = static_cast<int>(h->dim);
                            a.L = static_cast<int>(L);
                            a.k = static_cast<int>(k);
                            a.measure = measure;
                            a.lut_mode = mode;
                            a.S = static_cast<int>(h->S);
                            a.C = static_cast<int>(h->C);
                            a.ds = static_cast<int>(h->ds);
                            a.K = static_cast<uint32_t>(K);
                            a.reorder_measure = reorder_measure;
                            a.out_ids = static_cast<uint32_t*>(o[0]);
                            a.out_dists = static_cast<float*>(o[1]);
                            a.out_counts = static_cast<uint32_t*>(o[2]);
                            ivf_topk_kernel<<<static_cast<unsigned>(nqc), 256, smem, call.s>>>(a);
                            SCANN_CUDA(cudaGetLastError());
                            return SCANN_OK;
                          });
}

}  // extern "C"
