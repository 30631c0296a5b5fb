// Tree-AH / Tree-X-Hybrid search with the LUT16 path (src/tree_x_hybrid/mod.rs:245-364 composed with
// src/hashes/lut16.rs and src/hashes/lut16_simd.rs; SURVEY.md §3.3, §3.5).
//
// Per batch (all on one stream, no host synchronisation inside):
//   1. partition        exact centroid scoring + top-L tokens                      (partition.cu)
//   2. worklist         (query, rank) pairs are grouped BY LEAF: count -> scan -> scatter -> items.
//                       A work item = one leaf + up to G pairs that probe it.
//   3. lut16_scan       persistent kernel, one CTA per work item: builds the G residual LUT16 tables
//                       in shared memory (bit-exact quantiser), streams the leaf's blocked 4-bit codes
//                       ONCE for all G queries (register-LUT PRMT lookups, integer accumulation),
//                       keeps an exact running top-R per query (threshold filter + radix select in
//                       shared memory) and writes <= R (approx distance, position) candidates per pair.
//   4. merge_reorder    one CTA per query: exact top-R of the <= L*R candidates by
//                       (approx distance, leaf rank, position), exact distance of the R raw rows in the
//                       reference's AVX2 order, final order by (exact distance, approx rank), top-k.
//
// What the reference does per leaf is FastTopNeighbors(R) + concat + stable sort + truncate(R)
// (:283-290, :322-338); the global top-R by approximate distance is a subset of the union of the
// per-leaf top-R lists, so steps 3+4 return the same candidate set except for the order inside exact
// ties of the approximate distance (BASELINE.json exempts those).
#include <algorithm>

#include <stdlib.h>

#include "kernels.h"
#include "lut16_scan_kernel.cuh"
#include "lut_f32_scan_kernel.cuh"
#include "tcscan.h"

namespace scann {

// ------------------------------------------------------------------------------------ index build
// Converts PackedCodes4Bit rows (src/hashes/lut16.rs:43-61; row-major, low nibble = even subspace)
// to the blocked layout documented in lut16_device.cuh.  One thread per output u32.
__global__ void repack_blocked_kernel(const uint8_t* __restrict__ packed, const uint32_t* __restrict__ blk_leaf,
                                      const uint32_t* __restrict__ blk_off, const uint64_t* __restrict__ pt_off,
                                      int S, int SG, size_t total_words, uint32_t* __restrict__ out) {
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
    uint32_t leaf = blk_leaf[gb];
    uint64_t p0 = pt_off[leaf] + static_cast<uint64_t>(gb - blk_off[leaf]) * kBlockPts + lane * 8;
    uint64_t pend = pt_off[leaf + 1];
    int bpp = (S + 1) / 2;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      uint64_t p = p0 + i;
      if (p < pend) {
        uint8_t b = packed[p * bpp + (s >> 1)];
        uint32_t nib = (s & 1) ? (b >> 4) : (b & 0x0F);
        word |= nib << (4 * i);
      }
    }
  }
  out[w] = word;
}

// Converts byte codes (Codebook::encode rows, row-major [n][S] in leaf order) to the same 256-point blocks, stored
// subspace-major inside a block: byte s*256 + j of a block is subspace s of its point j, so lane l of a warp reads
// points l*8 .. l*8+7 of one subspace as 8 contiguous bytes (lut_f32_scan_kernel).  One thread per output u32 (4 points
// of one subspace); codes >= C are counted into *bad (the scan would read outside the table row).
__global__ void repack_bytes_kernel(const uint8_t* __restrict__ codes, const uint32_t* __restrict__ blk_leaf,
                                    const uint32_t* __restrict__ blk_off, const uint64_t* __restrict__ pt_off, int S,
                                    uint32_t C, size_t total_words, uint32_t* __restrict__ out, uint32_t* __restrict__ bad) {
  const size_t w = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (w >= total_words) return;
  const int j4 = static_cast<int>(w & 63);
  const size_t rest = w >> 6;
  const int s = static_cast<int>(rest % S);
  const size_t gb = rest / S;
  const uint32_t leaf = blk_leaf[gb];
  const uint64_t p0 = pt_off[leaf] + static_cast<uint64_t>(gb - blk_off[leaf]) * kBlockPts + j4 * 4, pend = pt_off[leaf + 1];
  uint32_t word = 0, nbad = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    if (p0 + i < pend) {
      const uint32_t c = codes[(p0 + i) * S + s];
      nbad += c >= C ? 1u : 0u;
      word |= c << (8 * i);
    }
  }
  out[w] = word;
  if (nbad) atomicAdd(bad, nbad);
}

// --------------------------------------------------------------------------------------- worklist
// Pairs that probe a leaf with no rows on this shard (empty partition, or a partition owned by another
// GPU) produce no work item; their candidate count stays 0.
//
// Pairs come in two classes: A = the query's closest leaf (rank 0), B = the rest.  Class-A items are laid out (and
// scanned) first: the closest leaf almost always yields the smallest "R-th best" distance, so the batch-wide bound
// tau_q is in place before the bulk of the work starts — and on a sharded index the class-A bounds of all shards can
// be min-reduced between the two phases (scann_treeah_search_begin / _end).  A "virtual leaf" v = leaf + K * class.
// T = ranks in class A: 1 (the closest leaf) normally; the T closest leaves when the tensor-core scan takes the rest
constexpr uint32_t kWlPad = 8;  // words between two atomic counters of the worklist passes (one per 32-byte sector)

__device__ __forceinline__ uint32_t wl_virtual_leaf(uint32_t leaf, size_t p, uint32_t L, uint32_t K, uint32_t T) {
  // pairs of one chunk fit 32 bits (nq * L * R * 8 <= 2 GiB): a 64-bit modulo costs ~150 instructions per pair and made the
  // count / scatter kernels 0.09 ms each at 640k pairs
  return leaf + ((static_cast<uint32_t>(p) % L) >= T ? K : 0u);
}

__global__ void wl_count_kernel(const uint32_t* __restrict__ tokens, size_t P, uint32_t K, uint32_t L, uint32_t T,
                                const uint64_t* __restrict__ pt_off, uint32_t* __restrict__ leaf_cnt) {
  size_t p = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (p >= P) return;
  uint32_t leaf = tokens[p];
  // one counter per 32-byte sector (kWlPad words apart): the L2 serialises atomics on a sector, and 8 packed counters
  // meant ~1300 serialised updates per sector at C3 (0.09 ms for 640k pairs)
  if (leaf < K && pt_off[leaf + 1] > pt_off[leaf]) atomicAdd(&leaf_cnt[wl_virtual_leaf(leaf, p, L, K, T) * kWlPad], 1u);
}

__global__ void wl_unpad_kernel(const uint32_t* __restrict__ padded, uint32_t n, uint32_t* __restrict__ dense) {
  const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v < n) dense[v] = padded[static_cast<size_t>(v) * kWlPad];
}

// Exclusive scans of pair counts and item counts over the 2K virtual leaves (three small kernels so that K = 65,536
// partitions do not serialise on one CTA), plus the algorithmic scan bytes of this batch (Σ pairs * leaf_size *
// bytes_per_point) for the roofline.  Position i of the scan order is virtual leaf
//   v(i) = perm[i] for i < K (class A), K + perm[i - K] otherwise (class B)
// with perm = leaves by descending size (longest items first), so the persistent scan kernel's atomic-counter
// schedule ends on the smallest items and the tail stays short.
constexpr int kWlBlock = 256;

__device__ __forceinline__ void wl_entry(uint32_t i, uint32_t K, int G, const uint32_t* __restrict__ perm,
                                         const uint32_t* __restrict__ leaf_cnt, const uint64_t* __restrict__ pt_off,
                                         uint32_t bpp, uint32_t& v, uint32_t& pc, uint32_t& ic,
                                         unsigned long long& bytes) {
  v = i < K ? perm[i] : K + perm[i - K];
  const uint32_t l = v >= K ? v - K : v;
  pc = leaf_cnt[v];
  ic = (pc + G - 1) / G;
  bytes = static_cast<unsigned long long>(pc) * (pt_off[l + 1] - pt_off[l]) * bpp;
}

// (1) per-block totals
__global__ void __launch_bounds__(kWlBlock) wl_reduce_kernel(const uint32_t* __restrict__ leaf_cnt, uint32_t K, int G,
                                                             const uint32_t* __restrict__ perm,
                                                             const uint64_t* __restrict__ pt_off, uint32_t bpp,
                                                             uint32_t* __restrict__ blk_pair,
                                                             uint32_t* __restrict__ blk_item,
                                                             unsigned long long* __restrict__ blk_bytes) {
  __shared__ uint32_t s_p[kWlBlock], s_i[kWlBlock];
  __shared__ unsigned long long s_b[kWlBlock];
  const uint32_t i = blockIdx.x * kWlBlock + threadIdx.x;
  uint32_t v, pc = 0, ic = 0;
  unsigned long long by = 0;
  if (i < 2 * K) wl_entry(i, K, G, perm, leaf_cnt, pt_off, bpp, v, pc, ic, by);
  s_p[threadIdx.x] = pc;
  s_i[threadIdx.x] = ic;
  s_b[threadIdx.x] = by;
  __syncthreads();
  for (int o = kWlBlock / 2; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      s_p[threadIdx.x] += s_p[threadIdx.x + o];
      s_i[threadIdx.x] += s_i[threadIdx.x + o];
      s_b[threadIdx.x] += s_b[threadIdx.x + o];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    blk_pair[blockIdx.x] = s_p[0];
    blk_item[blockIdx.x] = s_i[0];
    blk_bytes[blockIdx.x] = s_b[0];
  }
}

// (2) one CTA: exclusive scan of the block totals (in place), batch totals -> counters / stats
__global__ void __launch_bounds__(1024) wl_scan_blocks_kernel(uint32_t* __restrict__ blk_pair,
                                                              uint32_t* __restrict__ blk_item,
                                                              const unsigned long long* __restrict__ blk_bytes,
                                                              uint32_t nblocks,
                                                              uint32_t* __restrict__ counters /* [0]=items,[1]=next */,
                                                              unsigned long long* __restrict__ stats) {
  __shared__ uint32_t s_p[1024], s_i[1024];
  __shared__ unsigned long long s_b[1024];
  const uint32_t per = (nblocks + 1023) / 1024;
  const uint32_t b = threadIdx.x * per, e = min(nblocks, b + per);
  uint32_t pc = 0, ic = 0;
  unsigned long long by = 0;
  for (uint32_t j = b; j < e; ++j) {
    pc += blk_pair[j];
    ic += blk_item[j];
    by += blk_bytes[j];
  }
  s_p[threadIdx.x] = pc;
  s_i[threadIdx.x] = ic;
  s_b[threadIdx.x] = by;
  __syncthreads();
  for (int o = 1; o < 1024; o <<= 1) {  // Hillis-Steele inclusive scan
    uint32_t vp = 0, vi = 0;
    unsigned long long vb = 0;
    if (threadIdx.x >= o) {
      vp = s_p[threadIdx.x - o];
      vi = s_i[threadIdx.x - o];
      vb = s_b[threadIdx.x - o];
    }
    __syncthreads();
    s_p[threadIdx.x] += vp;
    s_i[threadIdx.x] += vi;
    s_b[threadIdx.x] += vb;
    __syncthreads();
  }
  uint32_t pbase = s_p[threadIdx.x] - pc, ibase = s_i[threadIdx.x] - ic;
  for (uint32_t j = b; j < e; ++j) {
    const uint32_t p = blk_pair[j], it = blk_item[j];
    blk_pair[j] = pbase;
    blk_item[j] = ibase;
    pbase += p;
    ibase += it;
  }
  if (threadIdx.x == 1023) {
    counters[0] = s_i[1023];
    counters[1] = 0;
    if (stats) {
      atomicAdd(&stats[0], s_b[1023]);
      atomicAdd(&stats[1], static_cast<unsigned long long>(s_p[1023]));
    }
  }
}

// (3) per-block exclusive scan + block offset -> pair_start / item_start of every virtual leaf; counters[2] = first
// class-B item = number of class-A items
__global__ void __launch_bounds__(kWlBlock) wl_offsets_kernel(const uint32_t* __restrict__ leaf_cnt, uint32_t K, int G,
                                                              const uint32_t* __restrict__ perm,
                                                              const uint64_t* __restrict__ pt_off, uint32_t bpp,
                                                              const uint32_t* __restrict__ blk_pair,
                                                              const uint32_t* __restrict__ blk_item,
                                                              uint32_t* __restrict__ pair_start,
                                                              uint32_t* __restrict__ item_start,
                                                              uint32_t* __restrict__ counters) {
  __shared__ uint32_t s_p[kWlBlock], s_i[kWlBlock];
  const uint32_t i = blockIdx.x * kWlBlock + threadIdx.x;
  uint32_t v = 0, pc = 0, ic = 0;
  unsigned long long by = 0;
  if (i < 2 * K) wl_entry(i, K, G, perm, leaf_cnt, pt_off, bpp, v, pc, ic, by);
  s_p[threadIdx.x] = pc;
  s_i[threadIdx.x] = ic;
  __syncthreads();
  for (int o = 1; o < kWlBlock; o <<= 1) {
    uint32_t vp = 0, vi = 0;
    if (threadIdx.x >= o) {
      vp = s_p[threadIdx.x - o];
      vi = s_i[threadIdx.x - o];
    }
    __syncthreads();
    s_p[threadIdx.x] += vp;
    s_i[threadIdx.x] += vi;
    __syncthreads();
  }
  if (i < 2 * K) {
    const uint32_t ps = blk_pair[blockIdx.x] + s_p[threadIdx.x] - pc, is = blk_item[blockIdx.x] + s_i[threadIdx.x] - ic;
    pair_start[v] = ps;
    item_start[v] = is;
    if (i == K) counters[2] = is;
  }
}

__global__ void wl_scatter_kernel(const uint32_t* __restrict__ tokens, size_t P, uint32_t K, uint32_t L, uint32_t T,
                                  const uint64_t* __restrict__ pt_off, const uint32_t* __restrict__ pair_start,
                                  uint32_t* __restrict__ cursor, uint32_t* __restrict__ sorted_pairs) {
  size_t p = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (p >= P) return;
  uint32_t leaf = tokens[p];
  if (leaf < K && pt_off[leaf + 1] > pt_off[leaf]) {
    const uint32_t v = wl_virtual_leaf(leaf, p, L, K, T);
    uint32_t slot = atomicAdd(&cursor[static_cast<size_t>(v) * kWlPad], 1u);
    sorted_pairs[pair_start[v] + slot] = static_cast<uint32_t>(p);
  }
}

__global__ void wl_items_kernel(const uint32_t* __restrict__ leaf_cnt, uint32_t K, int G,
                                const uint32_t* __restrict__ pair_start, const uint32_t* __restrict__ item_start,
                                uint4* __restrict__ items) {
  uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= 2 * K) return;
  const uint32_t l = v >= K ? v - K : v;
  uint32_t c = leaf_cnt[v], pb = pair_start[v], ib = item_start[v];
  for (uint32_t g = 0; g * G < c; ++g) items[ib + g] = make_uint4(l, pb + g * G, min(static_cast<uint32_t>(G), c - g * G), 0u);
}

// restrict filters: F id-indexed allow bitmaps [F][row_bytes] (bit i of byte i/8, LSB first) -> [F][total] bytes, one
// per (block, lane) in scan order.  One thread per (block, lane) reads its 8 ids once and writes its byte of every row.
__global__ void build_allow_kernel(const uint8_t* __restrict__ allow_by_id, size_t row_bytes, size_t F, size_t num_ids,
                                   const uint32_t* __restrict__ blk_leaf, const uint32_t* __restrict__ blk_off,
                                   const uint64_t* __restrict__ pt_off, const uint32_t* __restrict__ ids,
                                   size_t total /* blocks * 32 */, uint8_t* __restrict__ out) {
  size_t t = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= total) return;
  const uint32_t gb = static_cast<uint32_t>(t >> 5), lane = static_cast<uint32_t>(t & 31);
  const uint32_t leaf = blk_leaf[gb];
  const uint64_t p0 = pt_off[leaf] + static_cast<uint64_t>(gb - blk_off[leaf]) * kBlockPts + lane * 8, pend = pt_off[leaf + 1];
  uint32_t id[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) id[i] = p0 + i < pend ? ids[p0 + i] : 0xFFFFFFFFu;  // past the leaf: never allowed
  for (size_t f = 0; f < F; ++f) {
    const uint8_t* row = allow_by_id + f * row_bytes;
    uint32_t m = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if (id[i] < num_ids && ((row[id[i] >> 3] >> (id[i] & 7)) & 1u)) m |= 1u << i;
    out[f * total + t] = static_cast<uint8_t>(m);
  }
}

// Per-query parameters of scann_treeah_search_with_params, after the partition stage of a chunk: a query keeps its
// first min(L_q, L) tokens (its top-L_q leaves are a prefix of its top-L leaves) and every other rank gets no token, so
// no later stage sees it (they all skip tokens >= K).  qR / qk receive each query's R and k; a query with a value out
// of range (1 <= L_q <= L_call, R_q <= R, 1 <= k_q <= k) gets R = 0 and no token, hence count 0.  Lq / Rq / kq:
// nullptr = the scalar.  One thread per (query, rank).
__global__ void query_params_kernel(uint32_t* __restrict__ tokens, size_t P, uint32_t L, uint32_t L_call, uint32_t R,
                                    uint32_t k, const uint32_t* __restrict__ Lq, const uint32_t* __restrict__ Rq,
                                    const uint32_t* __restrict__ kq, uint32_t* __restrict__ qR,
                                    uint32_t* __restrict__ qk) {
  const size_t p = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (p >= P) return;
  const uint32_t p32 = static_cast<uint32_t>(p);  // 32-bit: see wl_virtual_leaf
  const uint32_t q = p32 / L, rank = p32 - q * L;
  const uint32_t lq = Lq ? Lq[q] : L_call, rq = Rq ? Rq[q] : R, kv = kq ? kq[q] : k;
  const bool ok = lq >= 1 && lq <= L_call && rq <= R && kv >= 1 && kv <= k;
  if (!ok || rq == 0 || rank >= lq) tokens[p] = 0xFFFFFFFFu;
  if (rank == 0) {
    qR[q] = ok ? rq : 0u;
    qk[q] = ok ? kv : 0u;
  }
}

// qthr <-> caller-visible f32 bounds (scann_treeah_search_begin / _end)
__global__ void tau_in_kernel(const float* __restrict__ tau, size_t nq, uint32_t* __restrict__ qthr) {
  size_t q = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (q >= nq) return;
  const float t = tau[q];
  const uint32_t k = (t == t && t < __int_as_float(0x7F800000)) ? f32_key(t) : 0xFFFFFFFFu;
  qthr[q] = min(qthr[q], k);
}
__global__ void tau_out_kernel(const uint32_t* __restrict__ qthr, size_t nq, float* __restrict__ tau) {
  size_t q = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (q >= nq) return;
  const uint32_t k = qthr[q];
  tau[q] = k == 0xFFFFFFFFu ? __int_as_float(0x7F800000) : key_f32(k);
}

// Tensor-core mode, after the full scan of the class-A ranks: one warp per query lowers qthr[q] to the R-th smallest
// approx distance over the union of its T class-A lists, when they hold at least R points.  Any R points of the probed
// leaves prove a bound, and the R-th of the union is never above the R-th of one of its lists (the bound a single leaf
// publishes).  Distances of different leaves have different quantisations, so the select runs on the f32 keys.
// qR: per-query R_q <= R (R is the list stride); nullptr = R for every query.
__global__ void __launch_bounds__(256) union_bound_kernel(const uint2* __restrict__ cand,
                                                          const uint32_t* __restrict__ cand_cnt, size_t nq, uint32_t L,
                                                          uint32_t T, uint32_t R, const uint32_t* __restrict__ qR,
                                                          uint32_t* __restrict__ qthr) {
  __shared__ uint32_t hist_all[8][256];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint32_t* hist = hist_all[warp];
  const size_t q = static_cast<size_t>(blockIdx.x) * 8 + warp;
  if (q >= nq) return;
  const size_t pair0 = q * L;
  const uint32_t Rq = qR ? qR[q] : R;
  if (Rq == 0) return;  // no candidates, nothing to bound: a select of 0 points would publish a meaningless key
  uint32_t total = 0;
  for (uint32_t r = 0; r < T; ++r) total += cand_cnt[pair0 + r];
  if (total < Rq) return;
  uint32_t prefix = 0, mask = 0, need = Rq;
  for (int shift = 24; shift >= 0; shift -= 8) {
#pragma unroll
    for (int k = 0; k < 8; ++k) hist[lane + 32 * k] = 0;
    __syncwarp();
    for (uint32_t r = 0; r < T; ++r) {
      const uint32_t c = cand_cnt[pair0 + r];
      const uint2* list = cand + (pair0 + r) * R;
      for (uint32_t i = lane; i < c; i += 32) {
        const uint32_t k = f32_key(__uint_as_float(list[i].x));
        if ((k & mask) == prefix) atomicAdd(&hist[(k >> shift) & 255u], 1u);
      }
    }
    __syncwarp();
    uint32_t d, below;
    warp_hist_digit(hist, need, lane, d, below);
    need -= below;
    prefix |= d << shift;
    mask |= 0xFFu << shift;
    __syncwarp();
  }
  if (lane == 0) qthr[q] = min(qthr[q], prefix);
}

// --------------------------------------------------------------------------- merge + exact reorder
struct MergeArgs {
  const uint2* cand;
  const uint32_t* cand_cnt;
  const uint32_t* tokens;
  const uint64_t* pt_off;
  const uint32_t* ids;
  const float* raw;
  size_t stride;
  size_t num_raw;
  int raw_by_pos;  // raw rows are stored in leaf order (row = pt_off[leaf] + position) instead of by datapoint id
  const float* queries;
  int dim, L, R, k, measure;
  uint32_t K;
  uint32_t* out_ids;
  float* out_dists;
  uint32_t* out_counts;
  uint32_t* cand_ids;
  float* cand_dists;
  uint32_t* cand_counts;
  // tensor-core scan (tcscan.cu): per-query candidate lists; queries with qflag set come from the per-pair lists
  const unsigned long long* qcand;
  const uint32_t* qcnt;
  const uint32_t* qflag;
  uint32_t qcap;
  // scann_treeah_search_with_params (merge_reorder_kernel<.., PQ = true>): per-query R_q <= R and k_q <= k; R and k
  // stay the row strides of the candidate lists and the outputs
  const uint32_t* qR;
  const uint32_t* qk;
};

constexpr int kMergeChunk = 2048;       // streaming chunk of the merge when a query can have L * R candidates
constexpr int kMergeChunkSmall = 512;   // after a tensor-core scan a query has a few hundred: smaller CTAs, 16 per SM
constexpr int kMergeThreads = 128;

// PQ: per-query R and k (a.qR / a.qk), a template flag so that the plain search's kernel carries none of it
template <int NT, int CHUNK, bool PQ>
__global__ void __launch_bounds__(NT) merge_reorder_kernel(const MergeArgs a) {
  extern __shared__ __align__(16) uint8_t sm[];
  const int p2 = next_pow2(a.R < 1 ? 1 : a.R);
  uint64_t* buf = reinterpret_cast<uint64_t*>(sm);              // [R + chunk]
  uint64_t* out = buf + (a.R + CHUNK);                          // [p2]
  uint32_t* hist = reinterpret_cast<uint32_t*>(out + p2);       // [264]
  uint32_t* prefix = hist + 264;                                // [L + 1]
  uint32_t* cid = prefix + (a.L + 1);                           // [p2] datapoint ids
  uint32_t* crow = cid + p2;                                    // [p2] raw row of each candidate
  float* qs = reinterpret_cast<float*>(crow + p2);              // [dim]
  const int tid = threadIdx.x;
  const size_t q = blockIdx.x;

  // tensor-core mode: the per-pair lists hold the class-A ranks (all ranks for a flagged query), the per-query list
  // every other point with approx distance <= tau_q (ignored for a flagged query: it may have overflowed)
  const int nlist = (a.qcand != nullptr && a.qflag[q] == 0u) ? static_cast<int>(min(a.qcnt[q], a.qcap)) : 0;
  for (int r = tid; r < a.L; r += NT) {
    uint32_t leaf = a.tokens[q * a.L + r];
    prefix[r + 1] = leaf < a.K ? a.cand_cnt[q * a.L + r] : 0u;
  }
  for (int d = tid; d < a.dim; d += NT) qs[d] = a.queries[q * a.dim + d];
  __syncthreads();
  if (tid < 32) {  // inclusive scan of the per-leaf candidate counts by one warp
    const int per = (a.L + 31) / 32, b = tid * per, e = min(a.L, b + per);
    uint32_t sum = 0;
    for (int r = b; r < e; ++r) sum += prefix[r + 1];
    uint32_t incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
      if (tid >= o) incl += v;
    }
    uint32_t run = incl - sum;
    for (int r = b; r < e; ++r) {
      run += prefix[r + 1];
      prefix[r + 1] = run;
    }
    if (tid == 0) prefix[0] = 0;
  }
  __syncthreads();
  const int total = static_cast<int>(prefix[a.L]);
  const uint2* cq = a.cand + q * static_cast<size_t>(a.L) * a.R;
  const unsigned long long* lq = a.qcand + (a.qcand ? q * static_cast<size_t>(a.qcap) : 0);
  auto gen = [&](int i) -> uint64_t {
    if (i >= total) return lq[i - total];  // keys are already (distance, leaf rank, position)
    int lo = 0, hi = a.L;  // largest r with prefix[r] <= i
    while (hi - lo > 1) {
      int mid = (lo + hi) >> 1;
      if (prefix[mid] <= static_cast<uint32_t>(i)) lo = mid;
      else hi = mid;
    }
    uint2 c = cq[static_cast<size_t>(lo) * a.R + (i - prefix[lo])];
    return (static_cast<uint64_t>(f32_key(__uint_as_float(c.x))) << 32) | (static_cast<uint64_t>(lo) << 22) | c.y;
  };
  const int Rq = PQ ? static_cast<int>(a.qR[q]) : a.R;
  const int m = block_topr_sorted<NT, CHUNK>(gen, total + nlist, Rq, buf, out, hist);

  // the R approximate candidates, in (approx distance, leaf rank, position) order
  for (int j = tid; j < p2; j += NT) {
    uint32_t id = 0xFFFFFFFFu, row = 0xFFFFFFFFu;
    float ad = __int_as_float(0x7F800000);
    if (j < m) {
      uint64_t key = out[j];
      uint32_t r = static_cast<uint32_t>((key >> 22) & 1023u), pos = static_cast<uint32_t>(key & 0x3FFFFFu);
      uint32_t leaf = a.tokens[q * a.L + r];
      const uint64_t at = a.pt_off[leaf] + pos;
      id = a.ids[at];
      row = a.raw_by_pos ? static_cast<uint32_t>(at) : id;
      ad = key_f32(static_cast<uint32_t>(key >> 32));
    }
    cid[j] = id;
    crow[j] = row;
    if (a.cand_ids && j < a.R) {
      a.cand_ids[q * a.R + j] = id;
      a.cand_dists[q * a.R + j] = ad;
    }
  }
  if (a.cand_counts && tid == 0) a.cand_counts[q] = static_cast<uint32_t>(m);
  __syncthreads();

  uint64_t* fin = buf;  // [p2] final keys
  if (a.raw != nullptr) {
    // exact distance of every candidate row, 8 lanes per row (src/tree_x_hybrid/mod.rs:342-364)
    const int grp = tid >> 3, sub = tid & 7;
#pragma unroll 2  // two passes' row loads in flight: the pass is a chain of dependent global loads
    for (int j0 = 0; j0 < m; j0 += NT / 8) {
      int j = j0 + grp;
      bool valid = j < m;
      // a row index outside the raw array (malformed index: the reference skips it via dataset.get(idx)) is dropped
      const uint32_t ri = crow[valid ? j : 0];
      const bool have = ri < a.num_raw;
      const float* row = a.raw + static_cast<size_t>(have ? ri : 0u) * a.stride;
      float d = exact_pair_distance<false>(qs, row, a.dim, a.measure, 0.0f, sub);
      if (valid && sub == 0)
        fin[j] = have ? ((static_cast<uint64_t>(f32_key(d)) << 32) | static_cast<uint32_t>(j)) : ~0ull;
    }
    for (int j = m + tid; j < p2; j += NT) fin[j] = ~0ull;
    __syncthreads();
    block_bitonic_sort<NT>(fin, p2);  // stable by construction: ties broken by approximate rank j
  } else {
    for (int j = tid; j < p2; j += NT)
      fin[j] = j < m ? ((out[j] & 0xFFFFFFFF00000000ull) | static_cast<uint32_t>(j)) : ~0ull;
    __syncthreads();
  }
  const int kq = PQ ? static_cast<int>(a.qk[q]) : a.k;
  // a query with R_q == 0 gets the row of a search with R == 0, whose distances are padded with 0x7F7F7F7F
  const float pad = PQ && Rq == 0 ? __int_as_float(0x7F7F7F7F) : __int_as_float(0x7F800000);
  int kk = kq < m ? kq : m;
  while (kk > 0 && fin[kk - 1] == ~0ull) --kk;  // candidates whose raw row does not exist were dropped (sorted last)
  for (int j = tid; j < a.k; j += NT) {
    if (j < kk) {
      uint64_t key = fin[j];
      a.out_ids[q * a.k + j] = cid[key & 0xFFFFFFFFu];
      a.out_dists[q * a.k + j] = key_f32(static_cast<uint32_t>(key >> 32));
    } else {
      a.out_ids[q * a.k + j] = 0xFFFFFFFFu;
      a.out_dists[q * a.k + j] = pad;
    }
  }
  if (tid == 0) a.out_counts[q] = static_cast<uint32_t>(kk);
}

static size_t merge_smem_bytes(int R, int L, int dim, int chunk) {
  int p2 = next_pow2(R < 1 ? 1 : R);
  return (static_cast<size_t>(R) + chunk + p2) * 8 + 264 * 4 + (static_cast<size_t>(L) + 1) * 4 +
         static_cast<size_t>(p2) * 8 + static_cast<size_t>(dim) * 4 + 16;
}

}  // namespace scann

// ------------------------------------------------------------------------------------------ C ABI
struct scann_treeah {
  int device = 0;
  size_t K = 0, dim = 0, S = 0, ds = 0, SG = 0, n = 0, num_raw = 0, stride = 0;
  int use_residuals = 1, reorder_measure = SCANN_SQL2, pos_bits = 18;
  uint32_t max_leaf = 0;
  // code format: false = nibble codes scanned through LUT16 (scann_treeah_create_ex), true = byte codes with C codes per
  // subspace scanned through the f32 LookupTable (scann_treeah_create_lut_f32, lut_f32_scan_kernel.cuh)
  bool f32lut = false;
  size_t C = 16;
  scann::CentreScorer part;  // the partition stage; part.centers() are the f32 centres of the residual LUTs
  scann::DevBuf<float> codebook, raw;
  const float* raw_p = nullptr;  // raw.p, or the caller's device array (SCANN_TREEAH_BORROW_RAW)
  bool raw_by_pos = false;       // SCANN_TREEAH_RAW_BY_POSITION
  bool reorder_on = true;        // scann_treeah_set_reorder: exact re-score of the R candidates (needs raw)
  scann::DevBuf<uint32_t> codes, ids, blk_off, leaf_perm;  // leaf_perm: leaves by descending size
  scann::DevBuf<uint32_t> blk_leaf;                        // leaf of every 256-point block
  scann::DevBuf<uint8_t> allow_blk;                        // restrict filter in block order (scann_treeah_set_filter)
  scann::DevBuf<uint8_t> packed_rm;                        // PackedCodes4Bit rows in leaf order (tensor-core scan, tcscan.cu)
  bool tc_ok = false;                                      // the tensor-core scan can serve this index
  uint64_t stat_tc = 0, stat_lut = 0;                      // chunks scanned by the tensor-core / the register-LUT kernel
  bool filter_on = false;
  size_t num_blocks = 0;
  scann::DevBuf<uint64_t> pt_off;
  scann::DevBuf<unsigned long long> stats;  // [0] algorithmic scan bytes, [1] pairs of the last search
  scann::Workspace ws;
  std::mutex mu;
  scann::StreamOrder order;  // device work of successive calls, across streams
  cudaStream_t stream = nullptr;
  int sms = 148;
  // the chunk being searched, between its two phases (treeah_phase1 / treeah_phase2): treeah_plan, treeah_take_chunk
  struct Chunk {
    const float* dq = nullptr;
    size_t nq = 0, L = 0, R = 0, k = 0;
    int G = 8;              // queries per register-LUT work item
    bool use_tc = false;    // probe + tensor-core scan of the other ranks
    int T = 1;              // ranks in class A of the worklist
    bool partition = true;  // the chunk partitions its queries (else the caller passed the tokens)
    bool params = false;    // per-query R / k (scann_treeah_search_with_params)
    uint32_t *tokens = nullptr, *counters = nullptr, *cand_cnt = nullptr, *qthr = nullptr;
    uint2* cand = nullptr;
    // worklist buffers (rebuilt over the flagged queries' tokens after a tensor-core scan)
    uint32_t *leaf_cnt = nullptr, *pair_start = nullptr, *item_start = nullptr, *wl_blk_pair = nullptr,
             *wl_blk_item = nullptr, *sorted_pairs = nullptr;
    unsigned long long* wl_blk_bytes = nullptr;
    uint4* items = nullptr;
    uint32_t *qR = nullptr, *qk = nullptr;  // per-query R / k when params, else nullptr
    scann::ScanArgs a;
  } ck;
  bool split_active = false;  // between scann_treeah_search_begin and _end / _abort: other entry points are refused
  // optional live profiling: (stage, start, end) CUDA-event spans; stages 0 partition, 1 worklist, 2 scan, 3 merge
  bool profiling = false;
  struct Span {
    int stage;
    cudaEvent_t e0, e1;
  };
  std::vector<Span> prof_spans;
  struct TcSpan {
    cudaEvent_t e[3];
  };
  std::vector<TcSpan> tc_spans;  // (before LUT build, before scan, after scan) of every tensor-core scan while profiling
  uint64_t prof_launches = 0;
  void span_begin(int stage, cudaStream_t s) {
    if (!profiling) return;
    Span sp{stage, nullptr, nullptr};
    if (cudaEventCreate(&sp.e0) != cudaSuccess || cudaEventCreate(&sp.e1) != cudaSuccess) return;
    cudaEventRecord(sp.e0, s);
    prof_spans.push_back(sp);
  }
  void span_end(cudaStream_t s) {
    if (!profiling || prof_spans.empty()) return;
    cudaEventRecord(prof_spans.back().e1, s);
  }
  void clear_spans() {
    for (Span& sp : prof_spans) {
      if (sp.e0) cudaEventDestroy(sp.e0);
      if (sp.e1) cudaEventDestroy(sp.e1);
    }
    prof_spans.clear();
    for (TcSpan& t : tc_spans)
      for (cudaEvent_t e : t.e)
        if (e) cudaEventDestroy(e);
    tc_spans.clear();
  }
  ~scann_treeah() {
    clear_spans();
    if (stream) cudaStreamDestroy(stream);
  }
};

namespace scann {

constexpr size_t kScanSmemMax = 227 * 1024;  // dynamic shared memory a CTA may opt in to

// A persistent scan kernel of kScanWarps warps per CTA with smem bytes of dynamic shared memory, on as many CTAs as
// the device holds at once
template <typename... Params, typename... Args>
static scann_status launch_scan_kernel(void (*kern)(Params...), size_t smem, int sms, cudaStream_t s, Args... args) {
  SCANN_REQUIRE(smem <= kScanSmemMax, SCANN_RESOURCE_EXHAUSTED, "scan kernel needs %zu B of shared memory (R too large)",
                smem);
  SCANN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  int occ = 0;
  SCANN_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kScanWarps * 32, smem));
  if (occ < 1) occ = 1;
  kern<<<sms * occ, kScanWarps * 32, smem, s>>>(args...);
  SCANN_CUDA(cudaGetLastError());
  return SCANN_OK;
}

// The scan kernel of the handle's code format with G queries per work item: the register-LUT scan of nibble codes
// (lut16_scan_kernel.cuh) in the accumulation mode of S, or the f32-table scan of byte codes (lut_f32_scan_kernel.cuh).
// The restrict filter is a template flag so the unfiltered kernels carry none of it.
template <int G>
static scann_status launch_scan_g(const scann_treeah* h, ScanArgs a, cudaStream_t s) {
  a.cap = scan_list_cap(a.R);
  const bool filt = a.allow != nullptr;
  if (h->f32lut) {
    const int C = static_cast<int>(h->C);
    return launch_scan_kernel(filt ? lut_f32_scan_kernel<G, true> : lut_f32_scan_kernel<G, false>,
                              lut_f32_scan_smem_bytes(G, a.S, C, a.dim, a.cap), h->sms, s, a, C);
  }
  auto kern = filt ? lut16_scan_kernel<G, 2, true> : lut16_scan_kernel<G, 2, false>;
  if (scan_acc_mode(a.S) == 3) kern = filt ? lut16_scan_kernel<G, 3, true> : lut16_scan_kernel<G, 3, false>;
  return launch_scan_kernel(kern, scan_smem_bytes(G, a.SG * 4, a.dim, a.cap, filt), h->sms, s, a);
}

static scann_status launch_handle_scan(const scann_treeah* h, int G, const ScanArgs& a, cudaStream_t s) {
  switch (G) {
    case 8: return launch_scan_g<8>(h, a, s);
    case 4: return launch_scan_g<4>(h, a, s);
    case 2: return launch_scan_g<2>(h, a, s);
    default: return launch_scan_g<1>(h, a, s);
  }
}

// blocks of each closest leaf the probe launch scans: 16 x 256 = 4096 points (scann_b200.h)
constexpr int kProbeBlocks = 16;

// shared memory of one scan CTA of the handle's code format with G queries per work item
static size_t scan_cta_bytes(const scann_treeah* h, int G, int cap, bool filt) {
  if (h->f32lut)
    return lut_f32_scan_smem_bytes(G, static_cast<int>(h->S), static_cast<int>(h->C), static_cast<int>(h->dim), cap);
  return scan_smem_bytes(G, static_cast<int>(h->SG) * 4, static_cast<int>(h->dim), cap, filt);
}

// Worklist of the register-LUT scan over `tokens` (buffers in h->ck): count -> scans -> scatter -> items.  with_stats:
// add the batch's algorithmic scan bytes / pairs to h->stats.
static scann_status treeah_worklist(scann_treeah* h, const uint32_t* tokens, size_t nq, size_t L, bool first,
                                    cudaStream_t s) {
  const size_t K = h->K, P = nq * L;
  const int G = h->ck.G;
  const uint32_t T = static_cast<uint32_t>(h->ck.T);
  const bool with_stats = first;
  uint32_t* leaf_cnt = h->ck.leaf_cnt;                 // [2K] dense counts, then two padded arrays of 2K counters
  uint32_t* pad_cnt = leaf_cnt + 2 * K;                // [2K * kWlPad] counters of the count pass
  uint32_t* cursor = pad_cnt + 2 * K * kWlPad;         // [2K * kWlPad] cursors of the scatter pass
  SCANN_CUDA(cudaMemsetAsync(pad_cnt, 0, 4 * K * kWlPad * sizeof(uint32_t), s));
  // the rebuilt worklist (flagged queries after a tensor-core scan) keeps the per-pair lists of the class-A ranks
  if (first) SCANN_CUDA(cudaMemsetAsync(h->ck.cand_cnt, 0, P * sizeof(uint32_t), s));
  unsigned pb = static_cast<unsigned>((P + 255) / 256);
  wl_count_kernel<<<pb, 256, 0, s>>>(tokens, P, static_cast<uint32_t>(K), static_cast<uint32_t>(L), T, h->pt_off.p,
                                     pad_cnt);
  wl_unpad_kernel<<<static_cast<unsigned>((2 * K + 255) / 256), 256, 0, s>>>(pad_cnt, static_cast<uint32_t>(2 * K), leaf_cnt);
  // code bytes per point: ceil(S/2) nibble-packed, S as byte codes
  const uint32_t nwb = static_cast<uint32_t>((2 * K + kWlBlock - 1) / kWlBlock),
                 bpp32 = static_cast<uint32_t>(h->f32lut ? h->S : (h->S + 1) / 2);
  wl_reduce_kernel<<<nwb, kWlBlock, 0, s>>>(leaf_cnt, static_cast<uint32_t>(K), G, h->leaf_perm.p, h->pt_off.p, bpp32,
                                            h->ck.wl_blk_pair, h->ck.wl_blk_item, h->ck.wl_blk_bytes);
  wl_scan_blocks_kernel<<<1, 1024, 0, s>>>(h->ck.wl_blk_pair, h->ck.wl_blk_item, h->ck.wl_blk_bytes, nwb, h->ck.counters,
                                           with_stats ? h->stats.p : nullptr);
  wl_offsets_kernel<<<nwb, kWlBlock, 0, s>>>(leaf_cnt, static_cast<uint32_t>(K), G, h->leaf_perm.p, h->pt_off.p, bpp32,
                                             h->ck.wl_blk_pair, h->ck.wl_blk_item, h->ck.pair_start, h->ck.item_start,
                                             h->ck.counters);
  wl_scatter_kernel<<<pb, 256, 0, s>>>(tokens, P, static_cast<uint32_t>(K), static_cast<uint32_t>(L), T, h->pt_off.p,
                                       h->ck.pair_start, cursor, h->ck.sorted_pairs);
  wl_items_kernel<<<static_cast<unsigned>((2 * K + 255) / 256), 256, 0, s>>>(leaf_cnt, static_cast<uint32_t>(K), G,
                                                                            h->ck.pair_start, h->ck.item_start,
                                                                            h->ck.items);
  SCANN_CUDA(cudaGetLastError());
  return SCANN_OK;
}

// candidate list capacity per query of the tensor-core scan
static size_t tc_qcap(size_t R) { return std::min<size_t>(16384, std::max<size_t>(2048, 64 * R)); }

// tensor-core scan for this chunk?  tc_env = SCANN_SCAN_TC, read once per call: 0 never, 1 whenever the index supports
// it, default: when a leaf is probed by enough queries of the batch to fill the 128-wide query tiles
static bool treeah_use_tc(const scann_treeah* h, size_t nq, size_t L, size_t R, const char* tc_env) {
  if (!h->tc_ok || h->packed_rm.p == nullptr || L > 1024 || R < 1) return false;
  if (tc_env && tc_env[0] == '0') return false;
  if (tc_env && tc_env[0] == '1') return true;
  const size_t P = nq * L;
  return static_cast<double>(P) / static_cast<double>(std::min<size_t>(h->K, P)) >= 12.0;
}

// ranks (closest leaves of every query) the register-LUT kernel scans in full before the tensor-core pass: their exact
// per-leaf top-R lists give the bound tau_q the tensor-core pass filters with.  SCANN_TC_RANKS overrides (tuning).
static size_t tc_ranks(size_t L) {
  const char* e = getenv("SCANN_TC_RANKS");
  size_t v = e ? static_cast<size_t>(atoi(e)) : 2;
  if (v < 1) v = 1;
  return std::min(v, L);
}

// The restrict filters of one chunk: F rows of one byte per (block, lane) in scan order (build_allow_kernel) and the row
// of every query of the chunk.  allow == nullptr: no filter.
struct ChunkFilter {
  const uint8_t* allow = nullptr;
  size_t stride = 0;               // bytes per row (blocks * 32)
  uint32_t F = 0;                  // rows; a query whose row is >= F is allowed nothing
  const uint32_t* qfilt = nullptr; // [nq of the chunk]; nullptr = row 0 for every query
};

// the handle-wide filter of scann_treeah_set_filter: one row shared by every query
static ChunkFilter handle_filter(const scann_treeah* h) {
  ChunkFilter f;
  if (h->filter_on) {
    f.allow = h->allow_blk.p;
    f.stride = h->num_blocks * 32;
    f.F = 1;
  }
  return f;
}

// The per-query L / R / k of one chunk (scann_treeah_search_with_params: device arrays, nullptr = the scalar) and the
// caller's L, the bound of every L_q (the L of the search is clamped to K).
struct ChunkParams {
  const uint32_t *L = nullptr, *R = nullptr, *k = nullptr;
  size_t L_call = 0;
};

// The decisions a chunk of nq queries runs with, written into ck; the counting pass of the reservation and the run
// both take them from here.  partition: the chunk partitions its queries (else the caller passed tokens); filtered: a
// restrict filter applies; params: per-query R / k.
static void treeah_plan(const scann_treeah* h, size_t nq, size_t L, size_t R, const char* tc_env, bool partition,
                        bool filtered, bool params, scann_treeah::Chunk& ck) {
  const size_t P = nq * L;
  // group size: how many queries share a leaf on average
  const double avg = static_cast<double>(P) / static_cast<double>(std::min<size_t>(h->K, P));
  int G = avg >= 6.0 ? 8 : (avg >= 3.0 ? 4 : (avg >= 1.5 ? 2 : 1));
  // the scan CTA holds G queries' residuals, tables and candidate buffers: smaller groups where they do not fit (each
  // pair's per-leaf top-R does not depend on which queries share its item, so results stay the same)
  const int cap = scan_list_cap(static_cast<int>(R));
  while (G > 1 && scan_cta_bytes(h, G, cap, filtered) > kScanSmemMax) G /= 2;
  ck.nq = nq;
  ck.L = L;
  ck.R = R;
  ck.G = G;
  ck.use_tc = treeah_use_tc(h, nq, L, R, tc_env);  // then the chunk runs in two phases: the probe gives the bounds
  ck.T = ck.use_tc ? static_cast<int>(tc_ranks(L)) : 1;
  ck.partition = partition;
  ck.params = params;
}

// The buffers of a chunk planned into ck, written there.  The partition's scratch is taken by CentreScorer::select.
static void treeah_take_chunk(const scann_treeah* h, Workspace& ws, scann_treeah::Chunk& ck) {
  const size_t K = h->K, nq = ck.nq, P = nq * ck.L;
  if (ck.partition) ck.tokens = ws.take<uint32_t>(P);
  ck.leaf_cnt = ws.take<uint32_t>(2 * K + 4 * K * kWlPad);  // counts of the 2K virtual leaves + padded counters / cursors
  ck.pair_start = ws.take<uint32_t>(2 * K + 1);
  ck.item_start = ws.take<uint32_t>(2 * K + 1);
  ck.counters = ws.take<uint32_t>(4);
  const size_t nwl = (2 * K + kWlBlock - 1) / kWlBlock;
  ck.wl_blk_pair = ws.take<uint32_t>(nwl);
  ck.wl_blk_item = ws.take<uint32_t>(nwl);
  ck.wl_blk_bytes = ws.take<unsigned long long>(nwl);
  ck.sorted_pairs = ws.take<uint32_t>(P);
  ck.items = ws.take<uint4>(P / ck.G + 2 * std::min<size_t>(K, P) + 1);
  ck.cand = ws.take<uint2>(P * ck.R);
  ck.cand_cnt = ws.take<uint32_t>(P);
  ck.qthr = ws.take<uint32_t>(nq);
  ck.qR = ck.params ? ws.take<uint32_t>(nq) : nullptr;
  ck.qk = ck.params ? ws.take<uint32_t>(nq) : nullptr;
}

// Workspace bytes of a chunk planned into `plan`: treeah_take_chunk in phase 1, the partition's scratch and, in
// phase 2, the tensor-core scan
static size_t treeah_count_chunk(const scann_treeah* h, scann_treeah::Chunk plan) {
  return Workspace::count([&](Workspace& w) {
    treeah_take_chunk(h, w, plan);
    if (plan.partition) h->part.take_scratch(w, plan.nq);
    if (plan.use_tc) take_tc_scan(w, plan.nq, plan.L, h->K, h->S, h->max_leaf, tc_qcap(plan.R));
  });
}

// Phase 1 of a chunk planned into h->ck: partition -> worklist -> (two_phase: scan of the class-A items, i.e. every
// query's closest leaf on this shard; tau_out receives the bounds they prove).  State for phase 2 stays in h->ck / the
// workspace.
static scann_status treeah_phase1(scann_treeah* h, const float* dq, size_t k, bool two_phase, float* tau_out,
                                  const uint32_t* tokens_in, const ChunkFilter& filt, const ChunkParams& cp,
                                  cudaStream_t s) {
  scann_treeah::Chunk& ck = h->ck;
  const size_t nq = ck.nq, L = ck.L, R = ck.R, P = nq * L;
  treeah_take_chunk(h, h->ws, ck);
  SCANN_TRY(h->ws.check("Tree-AH chunk"));
  if (!ck.partition) ck.tokens = const_cast<uint32_t*>(tokens_in);  // the caller keeps the array alive
  ck.dq = dq;
  ck.k = k;

  // 1. partition (K == 1 still goes through it: one centre, token 0)
  h->span_begin(0, s);
  if (ck.partition) SCANN_TRY(h->part.select(dq, nq, L, ck.tokens, nullptr, h->ws, s));
  if (ck.params) {  // per-query parameters: the ranks a query does not search leave the batch here
    query_params_kernel<<<static_cast<unsigned>((P + 255) / 256), 256, 0, s>>>(
        ck.tokens, P, static_cast<uint32_t>(L), static_cast<uint32_t>(cp.L_call), static_cast<uint32_t>(R),
        static_cast<uint32_t>(k), cp.L, cp.R, cp.k, ck.qR, ck.qk);
    SCANN_CUDA(cudaGetLastError());
    h->prof_launches += 1;
  }
  h->span_end(s);
  // 2. worklist
  h->span_begin(1, s);
  SCANN_CUDA(cudaMemsetAsync(ck.qthr, 0xFF, nq * sizeof(uint32_t), s));
  SCANN_TRY(treeah_worklist(h, ck.tokens, nq, L, true, s));
  h->span_end(s);
  ScanArgs& a = ck.a;
  a.codes = reinterpret_cast<const uint4*>(h->codes.p);
  a.blk_off = h->blk_off.p;
  a.pt_off = h->pt_off.p;
  a.centers = h->part.centers();
  a.codebook = h->codebook.p;
  a.queries = dq;
  a.items = ck.items;
  a.sorted_pairs = ck.sorted_pairs;
  a.counters = ck.counters;
  a.end_idx = 0;
  a.max_blocks = 0;
  a.allow = filt.allow;
  a.allow_stride = filt.stride;
  a.qfilt = filt.qfilt;
  a.num_filters = filt.F;
  a.qR = ck.qR;
  a.sentinel = 255u * static_cast<uint32_t>(h->S) + 1u;
  a.cand = ck.cand;
  a.cand_cnt = ck.cand_cnt;
  a.qthr = ck.qthr;
  a.mul.one = 1u;
  a.mul.w15 = 0x80000001u;
  a.dim = static_cast<int>(h->dim);
  a.S = static_cast<int>(h->S);
  a.ds = static_cast<int>(h->ds);
  a.SG = static_cast<int>(h->SG);
  a.L = static_cast<int>(L);
  a.R = static_cast<int>(R);
  a.cap = 0;  // set per CTA shape in launch_scan_g
  a.pos_bits = h->pos_bits;
  a.use_residuals = h->use_residuals;
  h->prof_launches += (ck.partition ? h->part.launches() : 0) + 7;  // partition + 7 worklist kernels
  if (two_phase) {
    // 3a. probe of the class-A items: the first kProbeBlocks blocks of every query's closest leaf prove a bound in
    // bounded time (a full scan of the largest leaves would serialise on a few CTAs); phase 2 scans them in full
    h->span_begin(2, s);
    a.end_idx = 2;
    // tensor-core mode: the class-A ranks are scanned in full here (their per-leaf lists are final, phase 2 does not
    // come back to them); otherwise a bounded probe of the closest leaf
    a.max_blocks = ck.use_tc ? 0 : kProbeBlocks;
    SCANN_TRY(launch_handle_scan(h, ck.G, a, s));
    h->prof_launches += 1;
    if (ck.use_tc) {  // the class-A lists are final: their union bounds the tensor-core pass
      union_bound_kernel<<<static_cast<unsigned>((nq + 7) / 8), 256, 0, s>>>(
          ck.cand, ck.cand_cnt, nq, static_cast<uint32_t>(L), static_cast<uint32_t>(ck.T), static_cast<uint32_t>(R),
          ck.qR, ck.qthr);
      h->prof_launches += 1;
    }
    if (tau_out) {
      tau_out_kernel<<<static_cast<unsigned>((nq + 255) / 256), 256, 0, s>>>(ck.qthr, nq, tau_out);
      h->prof_launches += 1;
    }
    SCANN_CUDA(cudaGetLastError());
    h->span_end(s);
  }
  return SCANN_OK;
}

// Phase 2: scan of the remaining items (all of them when phase 1 did not scan) with the optional global bounds
// tau_in (device [nq]), then merge + exact reorder.
static scann_status treeah_phase2(scann_treeah* h, bool two_phase, const float* tau_in, uint32_t* d_ids, float* d_dists,
                                  uint32_t* d_counts, uint32_t* d_cand_ids, float* d_cand_dists,
                                  uint32_t* d_cand_counts, cudaStream_t s) {
  const size_t K = h->K, nq = h->ck.nq, L = h->ck.L, R = h->ck.R, k = h->ck.k;
  ScanArgs& a = h->ck.a;
  h->span_begin(2, s);
  if (two_phase) {
    SCANN_CUDA(cudaMemsetAsync(h->ck.counters + 1, 0, sizeof(uint32_t), s));  // restart the item counter
    if (tau_in) tau_in_kernel<<<static_cast<unsigned>((nq + 255) / 256), 256, 0, s>>>(tau_in, nq, h->ck.qthr);
  }
  TcScanOut tco{nullptr, nullptr, nullptr, nullptr};
  (h->ck.use_tc ? h->stat_tc : h->stat_lut) += 1;
  if (h->ck.use_tc) {
    // 3b. tensor-core scan (tcscan.cu) under the bounds of the probe: per-query candidate lists; the queries it flags
    // (no bound, list overflow) are re-done by the register-LUT kernel over a worklist of their tokens only
    TcScanParams tp;
    tp.tokens = h->ck.tokens;
    tp.nq = nq;
    tp.L = L;
    tp.T = static_cast<size_t>(h->ck.T);
    tp.K = K;
    tp.dim = h->dim;
    tp.S = h->S;
    tp.pt_off = h->pt_off.p;
    tp.leaf_perm = h->leaf_perm.p;
    tp.codes_rm = h->packed_rm.p;
    tp.queries = h->ck.dq;
    tp.centers = h->part.centers();
    tp.codebook = h->codebook.p;
    tp.qthr = h->ck.qthr;
    tp.use_residuals = h->use_residuals;
    tp.max_leaf = h->max_leaf;
    tp.qcap = tc_qcap(R);
    tp.sms = h->sms;
    tp.pair_points = h->stats.p + 2;
    // class B of the chunk's worklist (pairs of rank >= T, grouped by leaf) is exactly what the tensor-core scan groups
    tp.wl_cnt = h->ck.leaf_cnt + K;
    tp.wl_pair_start = h->ck.pair_start + K;
    tp.wl_sorted_pairs = h->ck.sorted_pairs;
    // restrict filters: survivors a query's filter does not allow are dropped before they take a list slot
    tp.allow = a.allow;
    tp.allow_stride = a.allow_stride;
    tp.qfilt = a.qfilt;
    tp.num_filters = a.num_filters;
    tp.blk_off = h->blk_off.p;
    if (h->profiling) {
      scann_treeah::TcSpan sp{{nullptr, nullptr, nullptr}};
      bool ok = true;
      for (auto& e : sp.e) ok = ok && cudaEventCreate(&e) == cudaSuccess;
      if (ok) {
        for (int i = 0; i < 3; ++i) tp.ev[i] = sp.e[i];
        h->tc_spans.push_back(sp);
      }
    }
    SCANN_TRY(launch_tc_scan(tp, h->ws, &tco, s));
    SCANN_TRY(treeah_worklist(h, tco.fb_tokens, nq, L, false, s));
    h->prof_launches += kTcScanLaunches + 7;
  }
  a.end_idx = 0;
  a.max_blocks = 0;
  SCANN_TRY(launch_handle_scan(h, h->ck.G, a, s));
  h->span_end(s);
  // 4. merge + reorder
  h->span_begin(3, s);
  MergeArgs m;
  m.qcand = tco.qcand;
  m.qcnt = tco.qcnt;
  m.qflag = tco.qflag;
  m.qcap = h->ck.use_tc ? static_cast<uint32_t>(tc_qcap(R)) : 0u;
  m.qR = h->ck.qR;
  m.qk = h->ck.qk;
  m.cand = h->ck.cand;
  m.cand_cnt = h->ck.cand_cnt;
  m.tokens = h->ck.tokens;
  m.pt_off = h->pt_off.p;
  m.ids = h->ids.p;
  m.raw = h->reorder_on ? h->raw_p : nullptr;
  m.stride = h->stride;
  m.num_raw = h->num_raw;
  m.raw_by_pos = h->raw_by_pos ? 1 : 0;
  m.queries = h->ck.dq;
  m.dim = static_cast<int>(h->dim);
  m.L = static_cast<int>(L);
  m.R = static_cast<int>(R);
  m.k = static_cast<int>(k);
  m.measure = h->reorder_measure;
  m.K = static_cast<uint32_t>(K);
  m.out_ids = d_ids;
  m.out_dists = d_dists;
  m.out_counts = d_counts;
  m.cand_ids = d_cand_ids;
  m.cand_dists = d_cand_dists;
  m.cand_counts = d_cand_counts;
  // candidates per query after pruning are few: 128 threads per query keep more queries in flight per SM; after a
  // tensor-core scan the smaller streaming chunk makes the CTA 8 KB instead of 20 KB (the kernel is latency-bound: 16
  // instead of 11 resident queries per SM)
  const bool small = h->ck.use_tc;
  size_t msm = merge_smem_bytes(static_cast<int>(R), static_cast<int>(L), static_cast<int>(h->dim),
                                small ? kMergeChunkSmall : kMergeChunk);
  const bool pq = m.qR != nullptr;
  auto kern = small ? (pq ? merge_reorder_kernel<kMergeThreads, kMergeChunkSmall, true>
                          : merge_reorder_kernel<kMergeThreads, kMergeChunkSmall, false>)
                    : (pq ? merge_reorder_kernel<kMergeThreads, kMergeChunk, true>
                          : merge_reorder_kernel<kMergeThreads, kMergeChunk, false>);
  SCANN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(msm)));
  kern<<<static_cast<unsigned>(nq), kMergeThreads, msm, s>>>(m);
  SCANN_CUDA(cudaGetLastError());
  h->span_end(s);
  h->prof_launches += two_phase && tau_in ? 3 : 2;  // (tau_in) + lut16_scan + merge_reorder
  return SCANN_OK;
}

// Per-call restrict filters of scann_treeah_search_filtered (the caller's arrays): F = num_filters rows of
// ceil(num_ids / 8) bytes, the row of every query.
struct FilterTable {
  const uint8_t* allow;
  size_t F, num_ids;
  const uint32_t* filter_of_query;
};

// Per-query L / R / k of scann_treeah_search_with_params (the caller's arrays; nullptr = the scalar for every query).
struct ParamTable {
  const uint32_t *L, *R, *k;
};

// What a call takes once for its whole batch of nq queries: (ft) the filters in block order and, on SCANN_HOST, the
// uploaded bitmaps and rows; (pt, SCANN_HOST) the uploaded per-query L / R / k.  Every chunk reads its slice.
struct CallBufs {
  uint8_t* table = nullptr;
  uint8_t* allow = nullptr;
  uint32_t* qf = nullptr;
  uint32_t* params[3] = {};  // L, R, k
};
static CallBufs treeah_take_call(const scann_treeah* h, Workspace& ws, size_t nq, int memspace, const FilterTable* ft,
                                 const ParamTable* pt) {
  CallBufs b;
  const bool host = memspace == SCANN_HOST;
  if (ft) {
    b.table = ws.take<uint8_t>(ft->F * h->num_blocks * 32);
    if (host) {
      b.allow = ws.take<uint8_t>(ft->F * ((ft->num_ids + 7) / 8));
      b.qf = ws.take<uint32_t>(nq);
    }
  }
  if (pt && host) {
    const uint32_t* src[3] = {pt->L, pt->R, pt->k};
    for (int i = 0; i < 3; ++i)
      if (src[i]) b.params[i] = ws.take<uint32_t>(nq);
  }
  return b;
}

// scann_treeah_search, scann_treeah_search_filtered (ft != nullptr: per-query filters of this call only) and
// scann_treeah_search_with_params (pt != nullptr: per-query L / R / k of this call only)
static scann_status treeah_search(scann_treeah* h, const float* queries, size_t nq, size_t qdim, size_t L, size_t R,
                                  size_t k, uint32_t* ids, float* dists, uint32_t* counts, uint32_t* cand_ids,
                                  float* cand_dists, uint32_t* cand_counts, int memspace, void* stream,
                                  const FilterTable* ft, const ParamTable* pt = nullptr) {
  SCANN_REQUIRE(h != nullptr, SCANN_FAILED_PRECONDITION, "searcher not built");
  if (nq == 0) return SCANN_OK;  // empty batch -> Ok(vec![])
  SCANN_REQUIRE(queries && ids && dists && counts, SCANN_INVALID_ARGUMENT, "NULL buffer");
  SCANN_REQUIRE(qdim == h->dim, SCANN_INVALID_ARGUMENT, "Query dimensionality mismatch");  // tree_x_hybrid/mod.rs:251-253
  SCANN_REQUIRE(L >= 1 && L <= 1024, SCANN_INVALID_ARGUMENT, "partitions_to_search %zu outside 1..1024", L);
  SCANN_REQUIRE(R <= 2048, SCANN_INVALID_ARGUMENT, "pre_reorder_k %zu > 2048 unsupported", R);
  SCANN_REQUIRE(k >= 1, SCANN_INVALID_ARGUMENT, "k must be >= 1");
  SCANN_REQUIRE((cand_ids == nullptr) == (cand_dists == nullptr), SCANN_INVALID_ARGUMENT,
                "cand_ids and cand_dists go together");
  if (ft) {
    SCANN_REQUIRE(ft->F >= 1, SCANN_INVALID_ARGUMENT, "num_filters is 0");
    SCANN_REQUIRE(ft->F <= 0xFFFFFFFFull, SCANN_INVALID_ARGUMENT, "num_filters %zu does not fit 32 bits", ft->F);
    SCANN_REQUIRE(ft->allow && ft->filter_of_query, SCANN_INVALID_ARGUMENT, "NULL allow or filter_of_query");
    if (memspace == SCANN_HOST)  // the device path cannot check without a synchronisation: there such a query gets nothing
      for (size_t q = 0; q < nq; ++q)
        SCANN_REQUIRE(ft->filter_of_query[q] < ft->F, SCANN_INVALID_ARGUMENT,
                      "filter_of_query[%zu] = %u >= num_filters %zu", q, ft->filter_of_query[q], ft->F);
  }
  // the device path cannot check without a synchronisation: there such a query gets nothing (query_params_kernel)
  if (pt && memspace == SCANN_HOST) {
    for (size_t q = 0; q < nq; ++q) {
      SCANN_REQUIRE(!pt->L || (pt->L[q] >= 1 && pt->L[q] <= L), SCANN_INVALID_ARGUMENT,
                    "L_of_query[%zu] = %u outside 1..%zu", q, pt->L[q], L);
      SCANN_REQUIRE(!pt->R || pt->R[q] <= R, SCANN_INVALID_ARGUMENT, "R_of_query[%zu] = %u > R %zu", q, pt->R[q], R);
      SCANN_REQUIRE(!pt->k || (pt->k[q] >= 1 && pt->k[q] <= k), SCANN_INVALID_ARGUMENT,
                    "k_of_query[%zu] = %u outside 1..%zu", q, pt->k[q], k);
    }
  }
  std::lock_guard<std::mutex> lock(h->mu);
  SCANN_REQUIRE(!h->split_active, SCANN_FAILED_PRECONDITION, "a split search is in flight on this handle");
  SCANN_REQUIRE(!(ft && h->filter_on), SCANN_FAILED_PRECONDITION,
                "a handle-wide filter is set (scann_treeah_set_filter): clear it before a filtered search");
  CallScope call(h->device, h->order, memspace, stream, h->stream);
  const cudaStream_t s = call.s;
  const size_t L_call = L;
  if (L > h->K) L = h->K;  // partition() returns min(L, K) tokens (tree_partitioner.rs:214)
  const size_t Reff = R < 1 ? 1 : R;  // R == 0 (k*multiplier < 1) -> no candidates
  // chunk the batch so that the candidate buffer stays <= 1 GiB and the centre-distance scratch <= 512 MiB
  size_t chunk = nq;
  chunk = std::min(chunk, std::max<size_t>(1, (size_t(1) << 30) / (L * Reff * 8)));
  chunk = std::min(chunk, std::max<size_t>(1, (size_t(512) << 20) / (h->K * 4)));
  const QueryOut outs[] = {{ids, k * 4}, {dists, k * 4}, {counts, 4},
                           {cand_ids, R * 4}, {cand_dists, R * 4}, {cand_counts, 4}};
  const char* tc_env = getenv("SCANN_SCAN_TC");
  const bool filtered = ft != nullptr || h->filter_on, params = pt && (pt->L || pt->R || pt->k);
  // One chunk's carve is reserved for the largest of the distinct chunk sizes (a full chunk and the last one): G grows
  // with a chunk's queries, so the items P / G + ... of a short last chunk can outnumber those of a full chunk.
  size_t chunk_bytes = 0;
  for (const size_t nqc : {chunk, nq % chunk}) {
    if (nqc == 0) continue;
    scann_treeah::Chunk plan;
    treeah_plan(h, nqc, L, R, tc_env, true, filtered, params, plan);
    chunk_bytes = std::max(chunk_bytes, treeah_count_chunk(h, plan));
  }
  SCANN_TRY(h->ws.reserve(chunk_bytes + Workspace::count([&](Workspace& w) {
                            treeah_take_call(h, w, nq, memspace, ft, pt);
                            take_staging(w, memspace, chunk, h->dim, outs);
                          })));
  SCANN_CUDA(cudaMemsetAsync(h->stats.p, 0, 4 * sizeof(unsigned long long), s));
  // below the staging of run_query_chunks
  const CallBufs cb = treeah_take_call(h, h->ws, nq, memspace, ft, pt);
  SCANN_TRY(h->ws.check("Tree-AH call"));
  ChunkFilter filt = handle_filter(h);
  if (ft) {
    const size_t total = h->num_blocks * 32, row_bytes = (ft->num_ids + 7) / 8;
    const uint8_t* src = ft->allow;
    const uint32_t* qf = ft->filter_of_query;
    if (memspace == SCANN_HOST) {
      if (ft->F * row_bytes > 0)
        SCANN_CUDA(cudaMemcpyAsync(cb.allow, src, ft->F * row_bytes, cudaMemcpyHostToDevice, s));
      SCANN_CUDA(cudaMemcpyAsync(cb.qf, qf, nq * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
      src = cb.allow;
      qf = cb.qf;
    }
    if (total > 0) {
      build_allow_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, s>>>(
          src, row_bytes, ft->F, ft->num_ids, h->blk_leaf.p, h->blk_off.p, h->pt_off.p, h->ids.p, total, cb.table);
      SCANN_CUDA(cudaGetLastError());
    }
    filt.allow = cb.table;
    filt.stride = total;
    filt.F = static_cast<uint32_t>(ft->F);
    filt.qfilt = qf;
  }
  ParamTable dp{nullptr, nullptr, nullptr};
  if (pt) {
    dp = *pt;
    const uint32_t** a[3] = {&dp.L, &dp.R, &dp.k};
    for (int i = 0; i < 3; ++i)
      if (cb.params[i]) {
        SCANN_CUDA(cudaMemcpyAsync(cb.params[i], *a[i], nq * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
        *a[i] = cb.params[i];
      }
  }
  return run_query_chunks(h->ws, memspace, s, queries, nq, h->dim, chunk, outs,
                          [&](const float* dq, size_t q0, size_t nqc, void* const* o) -> scann_status {
    uint32_t* d_ids = static_cast<uint32_t*>(o[0]);
    float* d_dists = static_cast<float*>(o[1]);
    uint32_t* d_counts = static_cast<uint32_t*>(o[2]);
    uint32_t* d_cc = static_cast<uint32_t*>(o[5]);
    if (R == 0) {
      // (k as f32 * multiplier) as usize == 0: FastTopNeighbors(0) keeps nothing -> empty results
      SCANN_CUDA(cudaMemsetAsync(d_ids, 0xFF, nqc * k * 4, s));
      SCANN_CUDA(cudaMemsetAsync(d_dists, 0x7F, nqc * k * 4, s));  // 0x7F7F7F7F = 3.39e38: padding, never uninitialised
      SCANN_CUDA(cudaMemsetAsync(d_counts, 0, nqc * 4, s));
      if (d_cc) SCANN_CUDA(cudaMemsetAsync(d_cc, 0, nqc * 4, s));
      return SCANN_OK;
    }
    ChunkFilter cf = filt;
    if (cf.qfilt) cf.qfilt += q0;
    ChunkParams cp;
    if (pt) {
      cp.L = dp.L ? dp.L + q0 : nullptr;
      cp.R = dp.R ? dp.R + q0 : nullptr;
      cp.k = dp.k ? dp.k + q0 : nullptr;
      cp.L_call = L_call;
    }
    treeah_plan(h, nqc, L, R, tc_env, true, filtered, params, h->ck);
    // with the tensor-core scan the chunk runs as probe (bounds from every query's closest leaf) + bulk scan
    const bool two_phase = h->ck.use_tc;
    SCANN_TRY(treeah_phase1(h, dq, k, two_phase, nullptr, nullptr, cf, cp, s));
    return treeah_phase2(h, two_phase, nullptr, d_ids, d_dists, d_counts, static_cast<uint32_t*>(o[3]),
                         static_cast<float*>(o[4]), d_cc, s);
  });
}

// scann_treeah_create_ex (bytes = false: `packed` holds PackedCodes4Bit rows, C = 16) and scann_treeah_create_lut_f32
// (bytes = true: `packed` holds byte codes [n][S], C codes per subspace)
static scann_status treeah_create(const float* centers, size_t K, size_t dim, const float* codebook, size_t S,
                                  size_t C, bool bytes, const uint8_t* packed, const uint32_t* ids,
                                  const uint64_t* part_offsets, size_t n, const float* raw, size_t num_raw,
                                  size_t stride, int use_residuals, int reorder_measure, uint32_t flags, int device,
                                  int memspace, scann_treeah** out) {
  SCANN_REQUIRE((flags & ~(SCANN_TREEAH_RAW_BY_POSITION | SCANN_TREEAH_BORROW_RAW)) == 0, SCANN_INVALID_ARGUMENT,
                "unknown flags 0x%x", flags);
  SCANN_REQUIRE(!(flags & SCANN_TREEAH_BORROW_RAW) || memspace == SCANN_DEVICE, SCANN_INVALID_ARGUMENT,
                "SCANN_TREEAH_BORROW_RAW needs device-resident arrays");
  SCANN_REQUIRE(!(flags & SCANN_TREEAH_RAW_BY_POSITION) || raw == nullptr || num_raw == n, SCANN_INVALID_ARGUMENT,
                "SCANN_TREEAH_RAW_BY_POSITION: raw must hold one row per index row (num_raw %zu != n %zu)", num_raw, n);
  SCANN_REQUIRE(out != nullptr, SCANN_INVALID_ARGUMENT, "out is NULL");
  *out = nullptr;
  SCANN_REQUIRE(n > 0 && K > 0, SCANN_INVALID_ARGUMENT, "Cannot build from empty dataset");  // tree_x_hybrid/mod.rs:132-134
  SCANN_REQUIRE(centers && codebook && packed && ids && part_offsets, SCANN_INVALID_ARGUMENT, "NULL index array");
  SCANN_REQUIRE(S >= 1 && S <= 256, SCANN_INVALID_ARGUMENT, "num_subspaces %zu outside 1..256", S);
  SCANN_REQUIRE(dim > 0 && dim % S == 0, SCANN_INVALID_ARGUMENT,
                "Dimensionality %zu must be divisible by num_subspaces %zu", dim, S);  // codebook.rs:154-159
  SCANN_REQUIRE(reorder_measure == SCANN_SQL2 || reorder_measure == SCANN_L2 || reorder_measure == SCANN_DOT,
                SCANN_INVALID_ARGUMENT, "unsupported reorder measure %d", reorder_measure);
  SCANN_REQUIRE(raw == nullptr || stride >= dim, SCANN_INVALID_ARGUMENT, "stride %zu < dim %zu", stride, dim);
  SCANN_REQUIRE(K < 0xFFFFFFFFull && n < 0xFFFFFFFFull, SCANN_INVALID_ARGUMENT, "index too large for u32 ids");
  if (bytes) {
    SCANN_REQUIRE(C >= 1 && C <= 256, SCANN_INVALID_ARGUMENT, "num_codes %zu outside 1..256", C);
    // the scan CTA holds one query's S x C table: a geometry that does not fit with one query and R = 1 cannot be searched
    const size_t smem = lut_f32_scan_smem_bytes(1, static_cast<int>(S), static_cast<int>(C), static_cast<int>(dim),
                                                scan_list_cap(1));
    SCANN_REQUIRE(smem <= kScanSmemMax, SCANN_OUT_OF_RANGE,
                  "S=%zu x C=%zu f32 lookup table: the scan needs %zu B of shared memory per query (> %zu)", S, C, smem,
                  kScanSmemMax);
  }
  SCANN_TRY(check_device(device));
  DeviceGuard g(device);

  scann_treeah* h = new scann_treeah();
  h->f32lut = bytes;
  h->C = C;
  h->device = device;
  h->K = K;
  h->dim = dim;
  h->S = S;
  h->ds = dim / S;
  h->SG = (S + 3) / 4;
  h->n = n;
  h->num_raw = raw ? num_raw : 0;
  h->stride = stride;
  h->use_residuals = use_residuals ? 1 : 0;
  h->reorder_measure = reorder_measure;
  h->sms = sm_count(device);
  int sum_bits = 1;
  while ((1u << sum_bits) <= 255u * S + 1u) ++sum_bits;  // scores 0..255*S plus the filter sentinel 255*S + 1
  h->pos_bits = 32 - sum_bits;
  // f32 distances carry no integer sum: the position keeps the 22 bits of the merge key (distance, leaf rank, position)
  if (h->pos_bits > 22 || bytes) h->pos_bits = 22;

  scann_status st = SCANN_OK;
  do {
    if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) {
      st = cuda_fail(cudaGetLastError(), "cudaStreamCreate", __FILE__, __LINE__);
      break;
    }
    cudaStream_t s = h->stream;
    // partition offsets on the host (block table is built there)
    std::vector<uint64_t> off(K + 1);
    if (cudaMemcpy(off.data(), part_offsets, (K + 1) * sizeof(uint64_t),
                   memspace == SCANN_DEVICE ? cudaMemcpyDeviceToHost : cudaMemcpyHostToHost) != cudaSuccess) {
      st = cuda_fail(cudaGetLastError(), "copy part_offsets", __FILE__, __LINE__);
      break;
    }
    bool ok = off[0] == 0 && off[K] == n;
    for (size_t l = 0; l < K && ok; ++l) ok = off[l] <= off[l + 1];
    if (!ok) {
      set_error("part_offsets must be non-decreasing with part_offsets[0]=0 and part_offsets[K]=n");
      st = SCANN_INVALID_ARGUMENT;
      break;
    }
    std::vector<uint32_t> blk_off(K + 1), blk_leaf;
    uint64_t nb = 0, max_leaf = 0;
    for (size_t l = 0; l < K; ++l) {
      blk_off[l] = static_cast<uint32_t>(nb);
      uint64_t sz = off[l + 1] - off[l];
      max_leaf = std::max(max_leaf, sz);
      nb += (sz + kBlockPts - 1) / kBlockPts;
    }
    blk_off[K] = static_cast<uint32_t>(nb);
    if (max_leaf >= (1ull << h->pos_bits)) {
      set_error("partition with %llu points exceeds the %d-bit in-leaf position limit for S=%zu",
                static_cast<unsigned long long>(max_leaf), h->pos_bits, S);
      st = SCANN_OUT_OF_RANGE;
      break;
    }
    h->max_leaf = static_cast<uint32_t>(max_leaf);
    blk_leaf.resize(nb);
    for (size_t l = 0; l < K; ++l)
      for (uint32_t b = blk_off[l]; b < blk_off[l + 1]; ++b) blk_leaf[b] = static_cast<uint32_t>(l);

    DevBuf<uint8_t> d_packed;
    DevBuf<uint32_t>& d_blk_leaf = h->blk_leaf;
    h->num_blocks = nb;
    size_t bpp = bytes ? S : (S + 1) / 2;
    if ((st = h->part.set(centers, K, dim, memspace, s)) != SCANN_OK) break;
    if ((st = h->codebook.upload(codebook, S * C * h->ds, memspace, s)) != SCANN_OK) break;
    if ((st = h->ids.upload(ids, n, memspace, s)) != SCANN_OK) break;
    if ((st = h->pt_off.upload(off.data(), K + 1, SCANN_HOST, s)) != SCANN_OK) break;
    if ((st = h->blk_off.upload(blk_off.data(), K + 1, SCANN_HOST, s)) != SCANN_OK) break;
    std::vector<uint32_t> perm(K);
    for (size_t l = 0; l < K; ++l) perm[l] = static_cast<uint32_t>(l);
    std::stable_sort(perm.begin(), perm.end(),
                     [&](uint32_t x, uint32_t y) { return off[x + 1] - off[x] > off[y + 1] - off[y]; });
    if ((st = h->leaf_perm.upload(perm.data(), K, SCANN_HOST, s)) != SCANN_OK) break;
    if ((st = d_blk_leaf.upload(blk_leaf.data(), nb, SCANN_HOST, s)) != SCANN_OK) break;
    if ((st = d_packed.upload(packed, n * bpp, memspace, s)) != SCANN_OK) break;
    if (bytes) {
      const size_t words = static_cast<size_t>(nb) * S * (kBlockPts / 4);
      if ((st = h->codes.alloc(words > 0 ? words : 4)) != SCANN_OK) break;
      DevBuf<uint32_t> bad;
      if ((st = bad.alloc(1)) != SCANN_OK) break;
      cudaMemsetAsync(bad.p, 0, 4, s);
      if (words > 0)
        repack_bytes_kernel<<<static_cast<unsigned>((words + 255) / 256), 256, 0, s>>>(
            d_packed.p, d_blk_leaf.p, h->blk_off.p, h->pt_off.p, static_cast<int>(S), static_cast<uint32_t>(C), words,
            h->codes.p, bad.p);
      uint32_t nbad = 0;
      if (cudaMemcpyAsync(&nbad, bad.p, 4, cudaMemcpyDeviceToHost, s) != cudaSuccess ||
          cudaStreamSynchronize(s) != cudaSuccess) {
        st = cuda_fail(cudaGetLastError(), "treeah_create code check", __FILE__, __LINE__);
        break;
      }
      if (nbad != 0) {
        set_error("%u codes are >= num_codes %zu", nbad, C);
        st = SCANN_INVALID_ARGUMENT;
        break;
      }
    }
    h->tc_ok = !bytes && tc_scan_supported(S, dim);
    size_t words = bytes ? 0 : static_cast<size_t>(nb) * h->SG * 128;
    if (!bytes && (st = h->codes.alloc(words > 0 ? words : 4)) != SCANN_OK) break;
    if (words > 0) {
      repack_blocked_kernel<<<static_cast<unsigned>((words + 255) / 256), 256, 0, s>>>(
          d_packed.p, d_blk_leaf.p, h->blk_off.p, h->pt_off.p, static_cast<int>(S), static_cast<int>(h->SG), words,
          h->codes.p);
    }
    if (h->tc_ok) {  // the tensor-core scan reads the row-major PackedCodes4Bit rows (one point per thread)
      cudaStreamSynchronize(s);  // the repack kernel has read d_packed
      h->packed_rm = std::move(d_packed);
    }
    h->raw_by_pos = raw != nullptr && (flags & SCANN_TREEAH_RAW_BY_POSITION) != 0;
    if (raw && (flags & SCANN_TREEAH_BORROW_RAW)) {
      h->raw_p = raw;  // the caller keeps the device array alive for the life of the handle
    } else if (raw) {
      if ((st = h->raw.upload(raw, num_raw * stride, memspace, s)) != SCANN_OK) break;
      h->raw_p = h->raw.p;
    }
    if ((st = h->stats.alloc(4)) != SCANN_OK) break;
    cudaMemsetAsync(h->stats.p, 0, 4 * sizeof(unsigned long long), s);
    if (cudaStreamSynchronize(s) != cudaSuccess || cudaGetLastError() != cudaSuccess) {
      st = cuda_fail(cudaGetLastError(), "treeah_create sync", __FILE__, __LINE__);
      break;
    }
  } while (0);
  if (st != SCANN_OK) {
    scann_treeah_destroy(h);
    return st;
  }
  *out = h;
  return SCANN_OK;
}

}  // namespace scann

extern "C" {

scann_status scann_treeah_create(const float* centers, size_t K, size_t dim, const float* codebook, size_t S,
                                 const uint8_t* packed, const uint32_t* ids, const uint64_t* part_offsets,
                                 size_t n, const float* raw, size_t num_raw, size_t stride, int use_residuals,
                                 int reorder_measure, int device, int memspace, scann_treeah** out) {
  return scann_treeah_create_ex(centers, K, dim, codebook, S, packed, ids, part_offsets, n, raw, num_raw, stride,
                                use_residuals, reorder_measure, 0u, device, memspace, out);
}

scann_status scann_treeah_create_ex(const float* centers, size_t K, size_t dim, const float* codebook, size_t S,
                                    const uint8_t* packed, const uint32_t* ids, const uint64_t* part_offsets,
                                    size_t n, const float* raw, size_t num_raw, size_t stride, int use_residuals,
                                    int reorder_measure, uint32_t flags, int device, int memspace,
                                    scann_treeah** out) {
  return scann::treeah_create(centers, K, dim, codebook, S, 16, false, packed, ids, part_offsets, n, raw, num_raw,
                              stride, use_residuals, reorder_measure, flags, device, memspace, out);
}

scann_status scann_treeah_create_lut_f32(const float* centers, size_t K, size_t dim, const float* codebook, size_t S,
                                         size_t C, const uint8_t* codes, const uint32_t* ids,
                                         const uint64_t* part_offsets, size_t n, const float* raw, size_t num_raw,
                                         size_t stride, int use_residuals, int reorder_measure, uint32_t flags,
                                         int device, int memspace, scann_treeah** out) {
  return scann::treeah_create(centers, K, dim, codebook, S, C, true, codes, ids, part_offsets, n, raw, num_raw, stride,
                              use_residuals, reorder_measure, flags, device, memspace, out);
}

scann_status scann_treeah_search(scann_treeah* h, const float* queries, size_t nq, size_t qdim, size_t L, size_t R,
                                 size_t k, uint32_t* ids, float* dists, uint32_t* counts, uint32_t* cand_ids,
                                 float* cand_dists, uint32_t* cand_counts, int memspace, void* stream) {
  return scann::treeah_search(h, queries, nq, qdim, L, R, k, ids, dists, counts, cand_ids, cand_dists, cand_counts,
                              memspace, stream, nullptr);
}

scann_status scann_treeah_search_filtered(scann_treeah* h, const float* queries, size_t nq, size_t qdim, size_t L,
                                          size_t R, size_t k, const uint8_t* allow, size_t num_filters, size_t num_ids,
                                          const uint32_t* filter_of_query, uint32_t* ids, float* dists,
                                          uint32_t* counts, uint32_t* cand_ids, float* cand_dists,
                                          uint32_t* cand_counts, int memspace, void* stream) {
  const scann::FilterTable ft{allow, num_filters, num_ids, filter_of_query};
  return scann::treeah_search(h, queries, nq, qdim, L, R, k, ids, dists, counts, cand_ids, cand_dists, cand_counts,
                              memspace, stream, &ft);
}

scann_status scann_treeah_search_with_params(scann_treeah* h, const float* queries, size_t nq, size_t qdim, size_t L,
                                             size_t R, size_t k, const uint32_t* L_of_query, const uint32_t* R_of_query,
                                             const uint32_t* k_of_query, uint32_t* ids, float* dists, uint32_t* counts,
                                             uint32_t* cand_ids, float* cand_dists, uint32_t* cand_counts, int memspace,
                                             void* stream) {
  const scann::ParamTable pt{L_of_query, R_of_query, k_of_query};
  return scann::treeah_search(h, queries, nq, qdim, L, R, k, ids, dists, counts, cand_ids, cand_dists, cand_counts,
                              memspace, stream, nullptr, &pt);
}

scann_status scann_treeah_last_scan_bytes(scann_treeah* h, uint64_t* bytes, uint64_t* pairs) {
  using namespace scann;
  SCANN_REQUIRE(h != nullptr, SCANN_FAILED_PRECONDITION, "searcher not built");
  DeviceGuard g(h->device);
  unsigned long long v[2] = {0, 0};
  SCANN_CUDA(cudaDeviceSynchronize());
  SCANN_CUDA(cudaMemcpy(v, h->stats.p, sizeof(v), cudaMemcpyDeviceToHost));
  if (bytes) *bytes = v[0];
  if (pairs) *pairs = v[1];
  return SCANN_OK;
}

// ---- split search for a sharded index (SURVEY §8e): begin = partition + worklist + scan of every query's closest
// leaf on this shard -> tau_out; the caller min-reduces tau over the shards; end = scan of the rest under the global
// bounds + merge + exact reorder.  Device pointers only; one chunk (the whole batch) per begin/end pair.
// TreePartitioner::partition of the handle's own centres for a slice of the batch (device pointers): lets a sharded
// deployment partition nq/world queries per GPU and all-gather the tokens instead of repeating the stage on every GPU.
scann_status scann_treeah_partition(scann_treeah* h, const float* queries, size_t nq, size_t qdim, size_t L,
                                    uint32_t* tokens, void* stream) {
  using namespace scann;
  SCANN_REQUIRE(h != nullptr, SCANN_FAILED_PRECONDITION, "searcher not built");
  if (nq == 0) return SCANN_OK;
  SCANN_REQUIRE(queries && tokens, SCANN_INVALID_ARGUMENT, "NULL buffer");
  SCANN_REQUIRE(qdim == h->dim, SCANN_INVALID_ARGUMENT, "Query dimensionality mismatch");
  SCANN_REQUIRE(L >= 1 && L <= 1024, SCANN_INVALID_ARGUMENT, "partitions_to_search %zu outside 1..1024", L);
  SCANN_REQUIRE(!h->split_active, SCANN_FAILED_PRECONDITION, "a split search is in flight on this handle");
  std::lock_guard<std::mutex> lock(h->mu);
  SCANN_REQUIRE(!h->split_active, SCANN_FAILED_PRECONDITION, "a split search is in flight on this handle");
  CallScope call(h->device, h->order, SCANN_DEVICE, stream, h->stream);
  const size_t K = h->K;
  const size_t Leff = std::min(L, K);
  SCANN_REQUIRE(Leff == L, SCANN_INVALID_ARGUMENT, "partitions_to_search %zu > %zu partitions", L, K);
  SCANN_TRY(h->ws.reserve(Workspace::count([&](Workspace& w) { h->part.take_scratch(w, nq); })));
  h->prof_launches += h->part.launches();
  return h->part.select(queries, nq, L, tokens, nullptr, h->ws, call.s);
}

scann_status scann_treeah_search_begin(scann_treeah* h, const float* queries, size_t nq, size_t qdim, size_t L,
                                       size_t R, size_t k, const uint32_t* tokens, float* tau_out, void* stream) {
  using namespace scann;
  SCANN_REQUIRE(h != nullptr, SCANN_FAILED_PRECONDITION, "searcher not built");
  SCANN_REQUIRE(!h->f32lut, SCANN_UNIMPLEMENTED, "the split search serves nibble-code (LUT16) handles only");
  SCANN_REQUIRE(!h->split_active, SCANN_FAILED_PRECONDITION, "scann_treeah_search_begin called twice without _end");
  SCANN_REQUIRE(queries && tau_out && nq >= 1, SCANN_INVALID_ARGUMENT, "NULL buffer or empty batch");
  SCANN_REQUIRE(qdim == h->dim, SCANN_INVALID_ARGUMENT, "Query dimensionality mismatch");
  SCANN_REQUIRE(L >= 1 && L <= 1024, SCANN_INVALID_ARGUMENT, "partitions_to_search %zu outside 1..1024", L);
  SCANN_REQUIRE(R >= 1 && R <= 2048, SCANN_INVALID_ARGUMENT, "pre_reorder_k %zu outside 1..2048", R);
  SCANN_REQUIRE(k >= 1, SCANN_INVALID_ARGUMENT, "k must be >= 1");
  if (L > h->K) L = h->K;
  SCANN_REQUIRE(nq * L * R * 8 <= (size_t(2) << 30) && (tokens != nullptr || nq * h->K * 4 <= (size_t(512) << 20)),
                SCANN_INVALID_ARGUMENT, "batch of %zu queries is too large for the split search (split it)", nq);
  std::lock_guard<std::mutex> lock(h->mu);
  SCANN_REQUIRE(!h->split_active, SCANN_FAILED_PRECONDITION, "scann_treeah_search_begin called twice without _end");
  {
    CallScope call(h->device, h->order, SCANN_DEVICE, stream, h->stream);
    // the reservation covers _end's tensor-core scan too: _end takes it from above phase 1's buffers
    treeah_plan(h, nq, L, R, getenv("SCANN_SCAN_TC"), tokens == nullptr, h->filter_on, false, h->ck);
    SCANN_TRY(h->ws.reserve(treeah_count_chunk(h, h->ck)));
    cudaMemsetAsync(h->stats.p, 0, 4 * sizeof(unsigned long long), call.s);
    SCANN_TRY(treeah_phase1(h, queries, k, true, tau_out, tokens, handle_filter(h), ChunkParams(), call.s));
  }
  // The handle is marked busy, not locked: every other entry point answers FAILED_PRECONDITION until _end (or _abort),
  // so nothing can be left locked by a caller that fails between the two calls.
  h->split_active = true;
  return SCANN_OK;
}

scann_status scann_treeah_search_abort(scann_treeah* h) {
  using namespace scann;
  SCANN_REQUIRE(h != nullptr, SCANN_FAILED_PRECONDITION, "searcher not built");
  std::lock_guard<std::mutex> lock(h->mu);
  h->split_active = false;
  return SCANN_OK;
}

scann_status scann_treeah_search_end(scann_treeah* h, const float* tau_in, uint32_t* ids, float* dists,
                                     uint32_t* counts, void* stream) {
  using namespace scann;
  SCANN_REQUIRE(h != nullptr, SCANN_FAILED_PRECONDITION, "searcher not built");
  SCANN_REQUIRE(!h->f32lut, SCANN_UNIMPLEMENTED, "the split search serves nibble-code (LUT16) handles only");
  std::lock_guard<std::mutex> lock(h->mu);
  SCANN_REQUIRE(h->split_active, SCANN_FAILED_PRECONDITION, "scann_treeah_search_end without _begin");
  scann_status st = SCANN_OK;
  if (!(ids && dists && counts)) {
    set_error("NULL buffer");
    st = SCANN_INVALID_ARGUMENT;
  } else {
    CallScope call(h->device, h->order, SCANN_DEVICE, stream, h->stream);
    st = treeah_phase2(h, true, tau_in, ids, dists, counts, nullptr, nullptr, nullptr, call.s);
  }
  h->split_active = false;
  return st;
}

// RestrictFilter for the following searches (TreeXHybridSearcher::search_with_filter, tree_x_hybrid/mod.rs:245-250,
// 327-332): allow_by_id = bitmap over datapoint ids (bit i of byte i/8, LSB first; ids >= num_ids are not allowed);
// NULL clears the filter.
scann_status scann_treeah_set_filter(scann_treeah* h, const uint8_t* allow_by_id, size_t num_ids, int memspace) {
  using namespace scann;
  SCANN_REQUIRE(h != nullptr, SCANN_FAILED_PRECONDITION, "searcher not built");
  SCANN_REQUIRE(!h->split_active, SCANN_FAILED_PRECONDITION, "a split search is in flight on this handle");
  std::lock_guard<std::mutex> lock(h->mu);
  DeviceGuard g(h->device);
  if (allow_by_id == nullptr) {
    SCANN_CUDA(cudaDeviceSynchronize());
    h->filter_on = false;
    return SCANN_OK;
  }
  const size_t total = h->num_blocks * 32;
  if (total == 0) return SCANN_OK;
  DevBuf<uint8_t> tmp;
  const uint8_t* src = allow_by_id;
  if (memspace == SCANN_HOST) {
    SCANN_TRY(tmp.upload(allow_by_id, (num_ids + 7) / 8, SCANN_HOST, h->stream));
    src = tmp.p;
  }
  SCANN_CUDA(cudaDeviceSynchronize());  // no search may be reading the previous filter
  if (h->allow_blk.n != total) SCANN_TRY(h->allow_blk.alloc(total));
  build_allow_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, h->stream>>>(
      src, (num_ids + 7) / 8, 1, num_ids, h->blk_leaf.p, h->blk_off.p, h->pt_off.p, h->ids.p, total, h->allow_blk.p);
  SCANN_CUDA(cudaGetLastError());
  SCANN_CUDA(cudaStreamSynchronize(h->stream));
  h->filter_on = true;
  return SCANN_OK;
}

scann_status scann_treeah_path_stats(scann_treeah* h, uint64_t* tc_chunks, uint64_t* lut_chunks) {
  using namespace scann;
  SCANN_REQUIRE(h != nullptr, SCANN_FAILED_PRECONDITION, "searcher not built");
  if (tc_chunks) *tc_chunks = h->stat_tc;
  if (lut_chunks) *lut_chunks = h->stat_lut;
  return SCANN_OK;
}

scann_status scann_treeah_set_profiling(scann_treeah* h, int enable) {
  using namespace scann;
  SCANN_REQUIRE(h != nullptr, SCANN_FAILED_PRECONDITION, "searcher not built");
  std::lock_guard<std::mutex> lock(h->mu);
  DeviceGuard g(h->device);
  cudaDeviceSynchronize();
  h->clear_spans();
  h->prof_launches = 0;
  h->profiling = enable != 0;
  return SCANN_OK;
}

scann_status scann_treeah_get_profile(scann_treeah* h, double* ms4, uint64_t* kernel_launches) {
  using namespace scann;
  SCANN_REQUIRE(h != nullptr && ms4 != nullptr, SCANN_INVALID_ARGUMENT, "NULL argument");
  std::lock_guard<std::mutex> lock(h->mu);
  DeviceGuard g(h->device);
  SCANN_CUDA(cudaDeviceSynchronize());
  for (int i = 0; i < 4; ++i) ms4[i] = 0.0;
  for (const scann_treeah::Span& sp : h->prof_spans) {
    float ms = 0.0f;
    if (sp.stage >= 0 && sp.stage < 4 && cudaEventElapsedTime(&ms, sp.e0, sp.e1) == cudaSuccess) ms4[sp.stage] += ms;
  }
  h->clear_spans();
  if (kernel_launches) *kernel_launches = h->prof_launches;
  h->prof_launches = 0;
  return SCANN_OK;
}

scann_status scann_treeah_tc_profile(scann_treeah* h, double* lut_ms, double* scan_ms, uint64_t* launches,
                                     uint64_t* pair_points) {
  using namespace scann;
  SCANN_REQUIRE(h != nullptr, SCANN_FAILED_PRECONDITION, "searcher not built");
  std::lock_guard<std::mutex> lock(h->mu);
  DeviceGuard g(h->device);
  SCANN_CUDA(cudaDeviceSynchronize());
  double a = 0.0, b = 0.0;
  for (const scann_treeah::TcSpan& t : h->tc_spans) {
    float ms = 0.0f;
    if (cudaEventElapsedTime(&ms, t.e[0], t.e[1]) == cudaSuccess) a += ms;
    if (cudaEventElapsedTime(&ms, t.e[1], t.e[2]) == cudaSuccess) b += ms;
  }
  if (lut_ms) *lut_ms = a;
  if (scan_ms) *scan_ms = b;
  if (launches) *launches = h->tc_spans.size();
  if (pair_points) {
    unsigned long long v = 0;
    SCANN_CUDA(cudaMemcpy(&v, h->stats.p + 2, sizeof(v), cudaMemcpyDeviceToHost));
    *pair_points = v;
  }
  return SCANN_OK;
}

scann_status scann_treeah_set_reorder(scann_treeah* h, int enable) {
  SCANN_REQUIRE(h != nullptr, SCANN_INVALID_ARGUMENT, "NULL handle");
  std::lock_guard<std::mutex> lk(h->mu);
  h->reorder_on = enable != 0;
  return SCANN_OK;
}

void scann_treeah_destroy(scann_treeah* h) {
  if (!h) return;
  scann::DeviceGuard g(h->device);
  cudaDeviceSynchronize();
  delete h;
}

}  // extern "C"
