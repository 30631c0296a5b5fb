// Tensor-core LUT16 scan (sm_100a, tcgen05.mma kind::i8): the same integers as the register-LUT scan of
// lut16_scan_kernel.cuh — the u32 sums of src/simd/dispatch.rs:259-295 over the u8 tables of
// src/hashes/lut16_simd.rs:39-90 — computed as an integer matrix product.
//
//   sum(q, p) = Σ_s LUT_q[s][code_p[s]] = < LUT_q (S*16 u8) , onehot(code_p) (S*16 {0,1}) >
//
// u8 x u8 products accumulated in s32 are exact, so the accumulators are bit-identical to the reference's u32 sums.
// The register-LUT kernel spends ~1.25 ALU instructions per (query, point, subspace) lookup and is ALU-pipe bound with
// the tensor pipe idle; here a 128-point x 128-query tile costs 24 (S = 48) tcgen05.mma instructions of 64 cycles.
//
// Per batch (launch_tc_scan, after the probe of every query's closest leaf has produced the bounds tau_q):
//   tcwl_*           pairs (query, rank) grouped BY LEAF; a group = one leaf + up to 128 of its pairs; an item = one
//                    group x a run of <= 32 point tiles (128 points each) of the leaf
//   tc_lut_kernel    one warp per (group, pair): residual LUT16 table (bit-exact quantiser, lut16_device.cuh) written as
//                    one K-major u8 row of the group's LUT tile, followed by two "threshold digits" (below)
//   tc_scan_kernel   persistent, one CTA per SM, warp-specialised:
//       warp 0       TMA: the item's LUT tile (128 rows x (S*16 + 32) bytes, 128-byte swizzle) -> shared memory (B operand)
//       warp 1       one lane issues tcgen05.mma.kind::i8, M = 128 points, N = 16..128 queries, K = 32 bytes; the A
//                    operand is read from TENSOR MEMORY, the accumulator (s32) is double-buffered in TMEM
//       warps 2-9    expanders: thread = one point; turn its packed 4-bit codes into one-hot bytes in registers, 8
//                    subspaces (128 K-bytes) at a time, and tcgen05.st them into a ring of A slots in TMEM
//       warps 10-13  epilogue: tcgen05.ld the accumulator (thread = one point, columns = queries), threshold, append the
//                    survivors (approx distance key | leaf rank | position) to per-query candidate lists
//   Threshold without a per-column compare: the LUT row of (query, leaf) carries two extra bytes (d0, d1) with
//   d0 + 255 d1 = BIG - smax, smax = the largest integer score whose dequantised distance is <= tau_q, and every point
//   row carries the constant bytes (1, 255) in the same K positions, so the accumulator is sum + BIG - smax and
//   "sum <= smax" is "acc <= BIG" for every column: one min tree per 32 accumulators.
//   Queries without a bound, and queries whose list overflows, are flagged and re-done by the register-LUT kernel
//   (treeah.cu), so the result does not depend on the list capacity.
// The candidates of a query are exactly { points of its probed leaves with approx distance <= tau_q }, a superset of
// its global top-R by (distance, leaf rank, position); merge_reorder_kernel selects the top-R from it, so results are
// identical to the register-LUT path.
#include <cuda.h>

#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "kernels.h"
#include "lut16_scan_kernel.cuh"
#include "tcscan.h"

namespace scann {

namespace {

// warp 0 TMA, 1-2 MMA issuers, 3 TMEM owner, then 4 * EG expander warps, then 8 epilogue warps
constexpr int ts_threads(int EG) { return 32 * (4 + 4 * EG + 8); }
constexpr int kTsRing = 8;            // A slots of 32 TMEM columns (128 K-bytes per point row)
constexpr int kTsHalf = kTsRing / 2;  // each expander group owns half of the ring: every use of a slot is by the same
                                      // group, so a waiter is never more than one mbarrier phase ahead
constexpr int kTsAcol = 256;          // first TMEM column of the A ring (accumulators: 2 x 128 columns before it)
constexpr int kTsAtom = 128 * 128;    // bytes of one (128 rows x 128 B) swizzle atom tile
constexpr uint32_t kTsBig = 32768;    // > 255 * 64: accumulator threshold
constexpr uint32_t kNoKey = 0xFFFFFFFFu;

// ---- PTX wrappers (same conventions as tc_gemm.cu) ------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// Bounded wait: a protocol error becomes a trap (reported as a CUDA error by the next API call) instead of a hang.
// g_tcs_dbg (host-mapped, optional): where the wait that timed out was — {1, barrier smem address, parity, tag}.
__device__ volatile uint32_t* g_tcs_dbg = nullptr;
__device__ __forceinline__ void dbg_mark(int idx, uint32_t v) {
  volatile uint32_t* d = g_tcs_dbg;
  if (d != nullptr && blockIdx.x == 0) d[8 + idx] = v;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, uint32_t tag = 0) {
  uint32_t ok = 0;
  for (uint32_t it = 0; !ok; ++it) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    if (!ok && it > (1u << 22)) {
      volatile uint32_t* d = g_tcs_dbg;
      if (d != nullptr && atomicCAS(const_cast<uint32_t*>(d), 0u, 1u) == 0u) {
        d[1] = bar;
        d[2] = parity;
        d[3] = tag;
        d[4] = blockIdx.x;
        d[5] = threadIdx.x;
        __threadfence_system();
      }
      __trap();
    }
  }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem desc], u8 x u8 -> s32
__device__ __forceinline__ void mma_i8_ts(uint32_t d, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d),
      "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tc_ld32_nowait(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_st32(uint32_t taddr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
      "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]),
      "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]),
      "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
      : "memory");
}
__device__ __forceinline__ void tc_st8(uint32_t taddr, uint32_t v0) {
  const uint32_t z = 0;
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(v0),
               "r"(z), "r"(z), "r"(z), "r"(z), "r"(z), "r"(z), "r"(z)
               : "memory");
}
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// K-major operand tile, canonical 128-byte-swizzle layout (rows of 128 B, 8-row groups 1024 B apart), sm_100 version
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr) {
  return static_cast<uint64_t>((saddr >> 4) & 0x3FFFu) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ uint32_t elect_one() {  // one lane of the (converged) warp
  uint32_t pred;
  asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xFFFFFFFF;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(pred));
  return pred;
}
__device__ __forceinline__ uint32_t shl_clamp(uint32_t v, uint32_t sh) {  // PTX shl: shift amounts > 31 give 0
  uint32_t r;
  asm("shl.b32 %0, %1, %2;" : "=r"(r) : "r"(v), "r"(sh));
  return r;
}

// One word of packed codes = the 4-bit codes of 8 consecutive subspaces of one point -> 8 x 16 one-hot bytes (K order:
// subspace-major, code-minor = the byte order of a LUT row).  Byte (s, c) is 1 iff code_s == c.
// Pipe balance: the expansion is the ALU-pipe load of the kernel (~5 nibbles per clock per SM at full tensor rate), so
// the nibble extraction and the three "- 32 k" run as integer multiply-adds on the FMA pipe; the multipliers come from
// kernel parameters (xm.sh[i] = 1 << (28 - 4 i), xm.eight = 8) so that the compiler cannot turn them back into shifts.
struct ExpandMul {
  uint32_t sh[8];
  uint32_t eight;
};
__device__ __forceinline__ void expand_onehot(uint32_t C, uint32_t (&r)[32], const ExpandMul& xm) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    uint32_t x, t, t1, t2, t3;
    asm("mul.lo.u32 %0, %1, %2;" : "=r"(x) : "r"(C), "r"(xm.sh[i]));  // nibble i -> bits 28..31 (lower nibbles below it)
    const uint32_t nib = x >> 28;                                         // the code, 0..15
    asm("mul.lo.u32 %0, %1, %2;" : "=r"(t) : "r"(nib), "r"(xm.eight));                // 8 * code: bit position of the 1
    asm("mad.lo.u32 %0, %1, %2, 0xFFFFFFE0;" : "=r"(t1) : "r"(nib), "r"(xm.eight));  // - 32
    asm("mad.lo.u32 %0, %1, %2, 0xFFFFFFC0;" : "=r"(t2) : "r"(nib), "r"(xm.eight));  // - 64
    asm("mad.lo.u32 %0, %1, %2, 0xFFFFFFA0;" : "=r"(t3) : "r"(nib), "r"(xm.eight));  // - 96
    r[4 * i + 0] = shl_clamp(1u, t);
    r[4 * i + 1] = shl_clamp(1u, t1);
    r[4 * i + 2] = shl_clamp(1u, t2);
    r[4 * i + 3] = shl_clamp(1u, t3);
  }
}

// largest integer score s (0 <= s <= smax_all) with dequant(s) <= tau; -1 when even 0 is above tau; -2 when the search
// does not settle (treated as "no bound").  dequant is monotone non-decreasing in s.
__device__ __forceinline__ int score_bound_from_tau(float tau, float mult, float biasS, int smax_all) {
  const float est = __fdiv_rn(__fsub_rn(tau, biasS), mult);
  long long s;
  if (!(est == est)) return -2;
  if (est < -1.0f) s = -1;
  else if (est > static_cast<float>(smax_all)) s = smax_all;
  else s = static_cast<long long>(floorf(est));
  for (int it = 0; it < 8 && s < smax_all && lut16_dequant(static_cast<uint32_t>(s + 1), mult, biasS) <= tau; ++it) ++s;
  for (int it = 0; it < 8 && s >= 0 && lut16_dequant(static_cast<uint32_t>(s), mult, biasS) > tau; --s, ++it) {
  }
  if (s >= 0 && lut16_dequant(static_cast<uint32_t>(s), mult, biasS) > tau) return -2;
  if (s < smax_all && lut16_dequant(static_cast<uint32_t>(s + 1), mult, biasS) <= tau) return -2;
  return static_cast<int>(s);
}

// ------------------------------------------------------------------------------------------------ worklist
// pairs of rank < T (the query's T closest leaves) are not part of this scan: the register-LUT kernel has scanned them
__global__ void tcwl_count_kernel(const uint32_t* __restrict__ tokens, size_t P, uint32_t K, uint32_t L, uint32_t T,
                                  const uint64_t* __restrict__ pt_off, uint32_t* __restrict__ leaf_cnt) {
  const size_t p = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (p >= P || static_cast<uint32_t>(p) % L < T) return;  // 32-bit: see wl_virtual_leaf (treeah.cu)
  const uint32_t leaf = tokens[p];
  if (leaf < K && pt_off[leaf + 1] > pt_off[leaf]) atomicAdd(&leaf_cnt[leaf], 1u);
}

__device__ __forceinline__ void tcwl_entry(uint32_t leaf, const uint32_t* __restrict__ leaf_cnt,
                                           const uint64_t* __restrict__ pt_off, uint32_t& pc, uint32_t& groups,
                                           uint32_t& chunks) {
  pc = leaf_cnt[leaf];
  groups = (pc + kTcsGroup - 1) / kTcsGroup;
  const uint32_t tiles = static_cast<uint32_t>((pt_off[leaf + 1] - pt_off[leaf] + kTcsTile - 1) / kTcsTile);
  chunks = pc ? (tiles + kTcsItemTiles - 1) / kTcsItemTiles : 0u;
}

// One CTA: exclusive scans over the leaves in `perm` order (largest leaves first, so the statically dealt items end on
// the small ones) of pairs / groups / items.  counters: [0] items, [1] groups.
__global__ void __launch_bounds__(1024) tcwl_scan_kernel(const uint32_t* __restrict__ leaf_cnt, uint32_t K,
                                                         const uint32_t* __restrict__ perm,
                                                         const uint64_t* __restrict__ pt_off,
                                                         uint32_t* __restrict__ pair_start,
                                                         uint32_t* __restrict__ group_start,
                                                         uint32_t* __restrict__ item_start,
                                                         uint32_t* __restrict__ counters,
                                                         unsigned long long* __restrict__ pair_points) {
  __shared__ uint32_t s_p[1024], s_g[1024], s_i[1024];
  unsigned long long pp_local = 0;
  const uint32_t per = (K + 1023) / 1024;
  const uint32_t b = threadIdx.x * per, e = min(K, b + per);
  uint32_t sp = 0, sg = 0, si = 0;
  for (uint32_t i = b; i < e; ++i) {
    uint32_t pc, g, c;
    tcwl_entry(perm[i], leaf_cnt, pt_off, pc, g, c);
    sp += pc;
    sg += g;
    si += g * c;
    pp_local += static_cast<unsigned long long>(pc) * (pt_off[perm[i] + 1] - pt_off[perm[i]]);
  }
  if (pair_points && pp_local) atomicAdd(pair_points, pp_local);
  s_p[threadIdx.x] = sp;
  s_g[threadIdx.x] = sg;
  s_i[threadIdx.x] = si;
  __syncthreads();
  for (int o = 1; o < 1024; o <<= 1) {
    uint32_t vp = 0, vg = 0, vi = 0;
    if (threadIdx.x >= o) {
      vp = s_p[threadIdx.x - o];
      vg = s_g[threadIdx.x - o];
      vi = s_i[threadIdx.x - o];
    }
    __syncthreads();
    s_p[threadIdx.x] += vp;
    s_g[threadIdx.x] += vg;
    s_i[threadIdx.x] += vi;
    __syncthreads();
  }
  uint32_t rp = s_p[threadIdx.x] - sp, rg = s_g[threadIdx.x] - sg, ri = s_i[threadIdx.x] - si;
  for (uint32_t i = b; i < e; ++i) {
    const uint32_t leaf = perm[i];
    uint32_t pc, g, c;
    tcwl_entry(leaf, leaf_cnt, pt_off, pc, g, c);
    pair_start[leaf] = rp;
    group_start[leaf] = rg;
    item_start[leaf] = ri;
    rp += pc;
    rg += g;
    ri += g * c;
  }
  if (threadIdx.x == 1023) {
    counters[0] = s_i[1023];
    counters[1] = s_g[1023];
    counters[2] = 0;  // protocol-error counter of the scan
  }
}

__global__ void tcwl_scatter_kernel(const uint32_t* __restrict__ tokens, size_t P, uint32_t K, uint32_t L, uint32_t T,
                                    const uint64_t* __restrict__ pt_off, const uint32_t* __restrict__ pair_start,
                                    uint32_t* __restrict__ cursor, uint32_t* __restrict__ sorted_pairs) {
  const size_t p = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (p >= P || static_cast<uint32_t>(p) % L < T) return;  // 32-bit: see wl_virtual_leaf (treeah.cu)
  const uint32_t leaf = tokens[p];
  if (leaf < K && pt_off[leaf + 1] > pt_off[leaf])
    sorted_pairs[pair_start[leaf] + atomicAdd(&cursor[leaf], 1u)] = static_cast<uint32_t>(p);
}

// groups[g] = {leaf, first sorted pair, pairs in the group, 0}; items[i] = {group, first tile, end tile, leaf}
__global__ void tcwl_items_kernel(const uint32_t* __restrict__ leaf_cnt, uint32_t K,
                                  const uint64_t* __restrict__ pt_off, const uint32_t* __restrict__ pair_start,
                                  const uint32_t* __restrict__ group_start, const uint32_t* __restrict__ item_start,
                                  uint4* __restrict__ groups, uint4* __restrict__ items) {
  const uint32_t leaf = blockIdx.x * blockDim.x + threadIdx.x;
  if (leaf >= K) return;
  uint32_t pc, ng, nc;
  tcwl_entry(leaf, leaf_cnt, pt_off, pc, ng, nc);
  if (pc == 0) return;
  const uint32_t tiles = static_cast<uint32_t>((pt_off[leaf + 1] - pt_off[leaf] + kTcsTile - 1) / kTcsTile);
  const uint32_t per = (tiles + nc - 1) / nc;  // balanced runs of <= kTcsItemTiles tiles
  const uint32_t pb = pair_start[leaf], gb = group_start[leaf], ib = item_start[leaf];
  for (uint32_t g = 0; g < ng; ++g) {
    groups[gb + g] = make_uint4(leaf, pb + g * kTcsGroup, min(static_cast<uint32_t>(kTcsGroup), pc - g * kTcsGroup), 0u);
    for (uint32_t c = 0; c < nc; ++c)
      items[ib + g * nc + c] = make_uint4(gb + g, c * per, min(tiles, (c + 1) * per), leaf);
  }
}

// ------------------------------------------------------------------------------------------------ LUT tiles
struct LutArgs {
  const uint4* groups;
  const uint32_t* counters;      // [1] = groups
  const uint32_t* sorted_pairs;
  const float* queries;
  const float* centers;
  const float* codebook;
  const uint32_t* qthr;          // [nq] f32 key of tau_q (kNoKey = none)
  uint8_t* lut;                  // [groups * 128][row_bytes]
  uint4* meta;                   // [groups * 128] {mult, bias*S, BIG - smax, pair}
  uint32_t* qflag;               // [nq] set when a pair of the query has no usable bound
  int dim, S, ds, L, use_residuals, row_bytes;
};

// Persistent warps, one LUT row (one pair of one group) per warp iteration.  A lane owns the table entries
// e = 128 t + 4 lane + b (b < 4, t < S / 8): four consecutive codes of one subspace, so a row is written with S / 8
// coalesced 128-byte stores and the lane's codewords never change.  DS = dims per subspace when they fit in registers
// (1 or 2), 0 = any ds (codewords re-read through L1).  Same operations in the same order as warp_build_lut16
// (lut16_device.cuh): sequential un-fused sum of squares, global min/max, scale = 255 / range, round half away from
// zero (values are >= 0 here: floor + (fraction >= 0.5), which is what roundf does), saturate.
__device__ __forceinline__ uint32_t lut16_quantize_nonneg(float v, float mn, float scale) {
  const float y = __fmul_rn(__fsub_rn(v, mn), scale);  // >= 0, or NaN (-> 0 like Rust's `as u8`)
  uint32_t i = __float2uint_rd(y);
  i += __fsub_rn(y, __uint2float_rn(i)) >= 0.5f ? 1u : 0u;
  return min(i, 255u);
}

// The row loop is bound by the latency of its dependent global loads (group -> pair -> query / centre rows: ~2 us per row
// against ~0.9 us of arithmetic), i.e. by the number of resident warps.  The codewords therefore live in shared memory
// (a lane reads its 4 codes x DS floats with one or two conflict-free LDS.128 per step) instead of 64 registers, which
// takes the kernel from 128 to <= 64 registers and from 16 to 32 warps per SM.
template <int DS>
__global__ void __launch_bounds__(256, DS > 0 ? 4 : 2) tc_lut_kernel(const LutArgs a) {
  extern __shared__ __align__(16) uint8_t sm[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* qres = reinterpret_cast<float*>(sm) + warp * a.dim;
  const int nstep = a.S / 8;  // 128 table bytes per step (S is a multiple of 16)
  constexpr int kDs = DS > 0 ? DS : 1;
  float* cbs = reinterpret_cast<float*>(sm) + 8 * a.dim;  // [S * 16 * DS] codewords (DS > 0), 16-byte aligned (dim % 16 == 0)
  if (DS > 0) {
    for (int i = threadIdx.x; i < a.S * 16 * DS; i += blockDim.x) cbs[i] = __ldg(a.codebook + i);
    __syncthreads();
  }
  const uint32_t ngroups = a.counters[1];
  const uint32_t total = ngroups * kTcsGroup;
  for (uint32_t r = blockIdx.x * 8 + warp; r < total; r += gridDim.x * 8) {
    const uint32_t g = r / kTcsGroup, j = r % kTcsGroup;
    const uint4 G = a.groups[g];
    const uint32_t ncol = (G.z + 15u) & ~15u;  // the MMA's N: rows beyond it are never read
    if (j >= ncol) continue;
    uint8_t* out = a.lut + static_cast<size_t>(r) * a.row_bytes;
    uint32_t val = kTsBig + 1u;  // never hits
    float mult = 1.0f, biasS = 0.0f;
    uint32_t pair = kNoKey;
    if (j < G.z) {
      pair = a.sorted_pairs[G.y + j];
      const uint32_t q = pair / static_cast<uint32_t>(a.L);
      __syncwarp();
      for (int d = lane; d < a.dim; d += 32) {
        float v = a.queries[static_cast<size_t>(q) * a.dim + d];
        if (a.use_residuals) v = __fsub_rn(v, __ldg(a.centers + static_cast<size_t>(G.x) * a.dim + d));
        qres[d] = v;
      }
      __syncwarp();
      float vals[8][4];
      float mn = 3.402823466e+38f, mx = -3.402823466e+38f;
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        if (t < nstep) {
          const int s = 8 * t + (lane >> 2);  // subspace of this lane's four entries
          float cw[4 * kDs];  // this lane's 4 codes x DS floats of step t
          if (DS > 0) {
            const float4* c4 = reinterpret_cast<const float4*>(cbs + (128 * t + 4 * lane) * DS);
#pragma unroll
            for (int v = 0; v < kDs; ++v) {
              const float4 x = c4[v];
              cw[4 * v + 0] = x.x;
              cw[4 * v + 1] = x.y;
              cw[4 * v + 2] = x.z;
              cw[4 * v + 3] = x.w;
            }
          }
#pragma unroll
          for (int b = 0; b < 4; ++b) {
            float sum = 0.0f;
            if (DS > 0) {
#pragma unroll
              for (int jj = 0; jj < kDs; ++jj) {
                const float d = __fsub_rn(qres[s * DS + jj], cw[b * DS + jj]);
                sum = __fadd_rn(sum, __fmul_rn(d, d));
              }
            } else {
              sum = lut_entry(qres, a.codebook, 128 * t + 4 * lane + b, a.ds);
            }
            vals[t][b] = sum;
            mn = fminf(mn, sum);
            mx = fmaxf(mx, sum);
          }
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        mn = fminf(mn, __shfl_xor_sync(0xFFFFFFFFu, mn, o));
        mx = fmaxf(mx, __shfl_xor_sync(0xFFFFFFFFu, mx, o));
      }
      const float range = __fsub_rn(mx, mn);
      float scale = 1.0f;
      if (!(range < 1e-10f)) {
        scale = __fdiv_rn(255.0f, range);
        mult = __fdiv_rn(1.0f, scale);
      }
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        if (t < nstep) {
          const uint32_t w = lut16_quantize_nonneg(vals[t][0], mn, scale) | (lut16_quantize_nonneg(vals[t][1], mn, scale) << 8) |
                             (lut16_quantize_nonneg(vals[t][2], mn, scale) << 16) |
                             (lut16_quantize_nonneg(vals[t][3], mn, scale) << 24);
          reinterpret_cast<uint32_t*>(out)[32 * t + lane] = w;
        }
      }
      biasS = __fmul_rn(mn, static_cast<float>(a.S));  // bias * S, rounded once (lut16_simd.rs:137)
      const uint32_t tk = a.qthr[q];
      int sb = -2;
      if (tk != kNoKey) sb = score_bound_from_tau(key_f32(tk), mult, biasS, 255 * a.S);
      if (sb == -2) {
        if (lane == 0) a.qflag[q] = 1u;  // no usable bound: the register-LUT kernel re-does this query
      } else {
        val = kTsBig - static_cast<uint32_t>(sb);  // sb = -1 -> BIG + 1
      }
    } else {
      for (int v = lane; v < a.S; v += 32) reinterpret_cast<uint4*>(out)[v] = make_uint4(0, 0, 0, 0);
    }
    if (lane < 2) {  // the 32-byte tail: (d0, d1, 0, ...) with d0 + 255 * d1 = val
      uint4 t = make_uint4(0, 0, 0, 0);
      if (lane == 0) t.x = (val % 255u) | ((val / 255u) << 8);
      reinterpret_cast<uint4*>(out + a.S * 16)[lane] = t;
    }
    if (lane == 0) a.meta[r] = make_uint4(__float_as_uint(mult), __float_as_uint(biasS), val, pair);
  }
}

// ------------------------------------------------------------------------------------------------ the scan
struct TcsArgs {
  const uint8_t* codes_rm;   // [n][bpp] PackedCodes4Bit rows in leaf order
  const uint64_t* pt_off;
  const uint4* groups;
  const uint4* items;
  const uint32_t* counters;  // [0] = items
  const uint4* meta;
  unsigned long long* qcand; // [nq][qcap]
  uint32_t* qcnt;            // [nq]
  uint32_t* err;             // protocol-error counter (must stay 0)
  uint32_t qcap;
  uint32_t nq;
  ExpandMul xm;              // opaque multipliers of expand_onehot
  int KA;                    // S / 8: 128-byte K atoms of table bytes (the threshold atom follows)
  int bpp;                   // S / 2
  int L;
};

// restrict filters of the filtered instantiation (TcScanParams).  A kernel parameter of its own: widening TcsArgs alone
// made ptxas spill in the unfiltered EG = 4 kernel.
struct TcsFilter {
  const uint8_t* allow;
  size_t allow_stride;
  const uint32_t* qfilt;
  const uint32_t* blk_off;
  uint32_t num_filters;
};

// A survivor (LUT row = (group, query column), accumulator, position in the leaf) -> the query's candidate list.
// FILT: a point the query's filter row does not allow is dropped first, so filtered-out points cannot overflow a list.
template <bool FILT>
__device__ __forceinline__ void tcs_emit(const TcsArgs& a, const TcsFilter& f, uint32_t lut_row, uint32_t acc, uint32_t pos,
                                         uint32_t leaf) {
  const uint4 m = __ldg(a.meta + lut_row);
  const uint32_t q = m.w / static_cast<uint32_t>(a.L), rank = m.w - q * static_cast<uint32_t>(a.L);
  if (m.w == kNoKey || q >= a.nq) {  // a padding row can never pass the threshold: protocol error, counted
    atomicAdd(a.err, 1u);
    return;
  }
  if (FILT) {  // bit pos % 8 of byte (block blk_off[leaf] + pos / 256, lane (pos % 256) / 8) of the query's row
    const uint32_t row = f.qfilt ? __ldg(f.qfilt + q) : 0u;
    if (row >= f.num_filters) return;
    const size_t at = row * f.allow_stride + (static_cast<size_t>(__ldg(f.blk_off + leaf)) + (pos >> 8)) * 32 +
                      ((pos & 255u) >> 3);
    if (!((__ldg(f.allow + at) >> (pos & 7u)) & 1u)) return;
  }
  const uint32_t sum = acc - m.z;  // acc = sum + (BIG - smax)
  const float dist = lut16_dequant(sum, __uint_as_float(m.x), __uint_as_float(m.y));
  const uint32_t slot = atomicAdd(a.qcnt + q, 1u);
  if (slot < a.qcap)
    a.qcand[static_cast<size_t>(q) * a.qcap + slot] =
        (static_cast<unsigned long long>(f32_key(dist)) << 32) | (static_cast<unsigned long long>(rank) << 22) | pos;
}

constexpr int kWqCap = 320;    // entries of one epilogue warp's survivor queue (uint4 {lut_row, acc, pos, leaf (FILT)})
constexpr int kWqStep = 256;   // most entries one filter step (32 lanes x 8 columns) can add

// EG: expander groups, 2 (one per pipeline) or 4 (two per pipeline, alternate chunks); FILT: restrict filters (a template
// flag, so the unfiltered kernel carries none of it)
template <int EG, bool FILT>
__global__ void __launch_bounds__(ts_threads(EG), 1) tc_scan_kernel(const __grid_constant__ CUtensorMap tmB, const TcsArgs a,
                                                                    const TcsFilter filt) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sB = smem;  // [KA + 1] atom tiles
  uint64_t* bars = reinterpret_cast<uint64_t*>(sB + (a.KA + 1) * kTsAtom);
  constexpr int kBFull = 0, kBEmpty = 1, kAFull = 2, kAEmpty = 2 + kTsRing, kTFull = 2 + 2 * kTsRing,
                kTEmpty = 4 + 2 * kTsRing, kNumBars = 6 + 2 * kTsRing;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + kNumBars);
  uint4* wq_base = reinterpret_cast<uint4*>(tmem_slot + 4);         // [8][kWqCap] survivor queues of the epilogue warps
  uint32_t* wq_cnt_base = reinterpret_cast<uint32_t*>(wq_base + 8 * kWqCap);  // [8]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t bar0 = smem_u32(bars);
  auto bar = [&](int i) { return bar0 + 8u * static_cast<uint32_t>(i); };

  if (warp == 0 && lane == 0) asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
  if (warp == 1 && lane == 0) {
    mbar_init(bar(kBFull), 1);
    mbar_init(bar(kBEmpty), 2);     // both MMA warps commit
    for (int i = 0; i < kTsRing; ++i) {
      mbar_init(bar(kAFull + i), 4);   // the four expander warps of one group
      mbar_init(bar(kAEmpty + i), 1);  // tcgen05.commit
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar(kTFull + i), 1);
      mbar_init(bar(kTEmpty + i), 8);  // the eight epilogue warps
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 3) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const uint32_t n_items = a.counters[0];
  const int nchunk = a.KA + 1;  // A chunks per point tile (the last one carries the threshold constants)

  if (warp == 0) {
    // ================================================================= TMA producer: the item's LUT tile
    if (lane == 0) {
      uint32_t it = 0;
      for (uint32_t item = blockIdx.x; item < n_items; item += gridDim.x, ++it) {
        const uint4 I = a.items[item];
        mbar_wait(bar(kBEmpty), (it & 1u) ^ 1u, 0x100u + it);  // the MMAs of the previous item have finished reading B
        mbar_expect_tx(bar(kBFull), static_cast<uint32_t>(nchunk) * kTsAtom);
        for (int c = 0; c < nchunk; ++c)
          tma_load_2d(smem_u32(sB + c * kTsAtom), &tmB, bar(kBFull), c * 128, static_cast<int>(I.x * kTcsGroup));
      }
    }
  } else if (warp == 1 || warp == 2) {
    // ================================================================= MMA issuers
    // Two issuing warps, one per accumulator / expander group ("pipeline" pp): a single thread needs ~200 cycles of
    // dependent instructions per tcgen05.mma when the operands have to be moved into uniform registers one by one,
    // which is 3-4x the 64 cycles the tensor core needs.  The whole warp runs the loop converged and one elected lane
    // issues, so the addresses stay warp-uniform; the two warps alternate tiles and share only the B tile.
    const uint32_t pp = warp == 1 ? 0u : 1u;
    if (elect_one()) {  // one lane runs the whole issue loop (elect.sync: the compiler knows it is a single thread)
      uint32_t it = 0, ts = 0;
      const uint64_t bd0 = umma_desc(smem_u32(sB));
      const uint32_t d = tmem + pp * kTcsGroup;
      const uint32_t a0 = tmem + kTsAcol + pp * kTsHalf * 32;
      for (uint32_t item = blockIdx.x; item < n_items; item += gridDim.x, ++it) {
        const uint4 I = a.items[item];
        const uint32_t ncol = (a.groups[I.x].z + 15u) & ~15u;
        const uint32_t idesc = (2u << 4) | ((ncol >> 3) << 17) | ((128u >> 4) << 24);  // s32 += u8 x u8, K-major both
        mbar_wait(bar(kBFull), it & 1u, 0x200u + it);
        for (uint32_t t = I.y; t < I.z; ++t, ++ts) {
          if ((ts & 1u) != pp) continue;
          const uint32_t k = ts >> 1;  // tiles of this pipeline so far
          mbar_wait(bar(kTEmpty + pp), (k & 1u) ^ 1u, 0x300000u + ts);  // the epilogue has drained this accumulator
          tc_fence_after();
          uint32_t m = k * static_cast<uint32_t>(nchunk);  // chunks of this pipeline so far
          for (int c = 0; c < a.KA; ++c, ++m) {
            const uint32_t sl = m % kTsHalf;
            mbar_wait(bar(kAFull + pp * kTsHalf + sl), (m / kTsHalf) & 1u, 0x400000u + m);
            tc_fence_after();
            const uint64_t bd = bd0 + static_cast<uint64_t>(c) * (kTsAtom >> 4);
            const uint32_t at = a0 + sl * 32;
            mma_i8_ts(d, at, bd, idesc, c != 0 ? 1u : 0u);
            mma_i8_ts(d, at + 8, bd + 2u, idesc, 1u);
            mma_i8_ts(d, at + 16, bd + 4u, idesc, 1u);
            mma_i8_ts(d, at + 24, bd + 6u, idesc, 1u);
            tc_commit(bar(kAEmpty + pp * kTsHalf + sl));  // the slot may be refilled once these MMAs retire
          }
          {  // the threshold atom holds 32 K-bytes
            const uint32_t sl = m % kTsHalf;
            mbar_wait(bar(kAFull + pp * kTsHalf + sl), (m / kTsHalf) & 1u, 0x400000u + m);
            tc_fence_after();
            mma_i8_ts(d, a0 + sl * 32, bd0 + static_cast<uint64_t>(a.KA) * (kTsAtom >> 4), idesc, 1u);
            tc_commit(bar(kAEmpty + pp * kTsHalf + sl));
            tc_commit(bar(kTFull + pp));
          }
        }
        tc_commit(bar(kBEmpty));  // this pipeline's MMAs on the B tile have retired
      }
    }
  } else if (warp >= 4 && warp < 4 + 4 * EG) {
    // ================================================================= expanders: codes -> one-hot A chunks in TMEM
    // Four groups of four warps (one warp per TMEM lane quadrant): pipeline pp = group / 2 takes the tiles of parity
    // pp, and inside a pipeline the two groups take alternate chunks (by the parity of the pipeline's running chunk
    // count m), so each A slot (m % 4) is always filled by the same group.
    const uint32_t gi = static_cast<uint32_t>(warp - 4) >> 2;
    const uint32_t pp = EG == 4 ? gi >> 1 : gi, sg = gi & 1u;
    const uint32_t quad = warp & 3;
    const uint32_t row = quad * 32 + lane;
    const uint32_t lane_addr = (quad * 32) << 16;
    uint32_t ts = 0;
    for (uint32_t item = blockIdx.x; item < n_items; item += gridDim.x) {
      const uint4 I = a.items[item];
      const uint64_t base = a.pt_off[I.w];
      const uint32_t leaf_n = static_cast<uint32_t>(a.pt_off[I.w + 1] - base);
      for (uint32_t t = I.y; t < I.z; ++t, ++ts) {
        if ((ts & 1u) != pp) continue;
        const uint32_t p = t * kTcsTile + row;
        uint32_t w[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) w[c] = 0;
        if (p < leaf_n) {
          const uint2* src = reinterpret_cast<const uint2*>(a.codes_rm + (base + p) * a.bpp);
#pragma unroll
          for (int c2 = 0; c2 < 4; ++c2)
            if (2 * c2 < a.KA) {
              const uint2 v = __ldg(src + c2);
              w[2 * c2] = v.x;
              w[2 * c2 + 1] = v.y;
            }
        }
        const uint32_t m0 = (ts >> 1) * static_cast<uint32_t>(nchunk);  // chunks of this pipeline before this tile
        // software pipeline: the tcgen05.st of a chunk is left in flight while this group's next chunk is expanded; its
        // completion (wait::st) and the hand-over to the MMA warp come right before the next store
        int prev_slot = -1;
        auto publish = [&]() {
          if (prev_slot >= 0) {
            tc_wait_st();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar(kAFull + prev_slot));
          }
        };
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const uint32_t m = m0 + c;
          if (c < a.KA && (EG == 2 || (m & 1u) == sg)) {
            const uint32_t slot = pp * kTsHalf + (m % kTsHalf);
            uint32_t r[32];
            expand_onehot(w[c], r, a.xm);  // rows past the end of the leaf expand code 0: the epilogue ignores them
            publish();
            mbar_wait(bar(kAEmpty + slot), ((m / kTsHalf) & 1u) ^ 1u, 0x500000u + m);
            tc_fence_after();
            tc_st32(tmem + lane_addr + kTsAcol + slot * 32, r);
            prev_slot = static_cast<int>(slot);
          }
        }
        {  // threshold chunk: K bytes (1, 255, 0, ...) against the LUT row's digits (d0, d1)
          const uint32_t m = m0 + static_cast<uint32_t>(a.KA);
          if (EG == 2 || (m & 1u) == sg) {
            const uint32_t slot = pp * kTsHalf + (m % kTsHalf);
            publish();
            mbar_wait(bar(kAEmpty + slot), ((m / kTsHalf) & 1u) ^ 1u, 0x600000u + m);
            tc_fence_after();
            tc_st8(tmem + lane_addr + kTsAcol + slot * 32, 0x0000FF01u);
            prev_slot = static_cast<int>(slot);
          }
          publish();
        }
      }
    }
  } else if (warp >= 4 + 4 * EG) {
    // ================================================================= epilogue: threshold + candidate append
    // Eight warps: two per TMEM lane quadrant, one for accumulator columns 0..63 and one for 64..127, so the
    // accumulator goes back to its MMA warp after ONE round of TMEM loads (a pipeline cannot start its next tile
    // before that).
    const uint32_t ew = static_cast<uint32_t>(warp - (4 + 4 * EG));  // 0..7
    const uint32_t half_id = ew >> 2;
    const uint32_t quad = warp & 3;
    const uint32_t row = quad * 32 + lane;
    const uint32_t lane_addr = (quad * 32) << 16;
    // survivors are queued in shared memory and written out 32 at a time, so that the L2 round trips of a flush
    // (meta load, list-slot atomic, store) overlap across lanes instead of serialising per hit
    uint4* const wq = wq_base + ew * kWqCap;
    volatile uint32_t* const wq_cnt = wq_cnt_base + ew;
    if (lane == 0) *wq_cnt = 0;
    __syncwarp();
    auto flush = [&]() {
      __syncwarp();
      const uint32_t nw = *wq_cnt;
      for (uint32_t i = lane; i < nw; i += 32) {
        const uint4 e = wq[i];
        tcs_emit<FILT>(a, filt, e.x, e.y, e.z, FILT ? e.w : 0u);
      }
      __syncwarp();
      if (lane == 0) *wq_cnt = 0;
      __syncwarp();
    };
    // threshold test of 32 accumulator columns starting at column c0 (nlive = 16 or 32 of them are real)
    // leaf: of the current item, carried in the queue entry for the restrict filter (FILT)
    auto filter32 = [&](const uint32_t (&v)[32], uint32_t c0, uint32_t nlive, bool valid, uint32_t lut_row0, uint32_t p,
                        uint32_t leaf) {
      uint32_t m8[4];
#pragma unroll
      for (int g8 = 0; g8 < 4; ++g8) {
        uint32_t m = v[8 * g8];
#pragma unroll
        for (int j = 1; j < 8; ++j) m = min(m, v[8 * g8 + j]);
        m8[g8] = m;
      }
      if (nlive < 32) m8[2] = m8[3] = kNoKey;
      const uint32_t mall = min(min(m8[0], m8[1]), min(m8[2], m8[3]));
      if (__any_sync(0xFFFFFFFFu, valid && mall <= kTsBig)) {
#pragma unroll
        for (int g8 = 0; g8 < 4; ++g8) {
          const bool hit = valid && m8[g8] <= kTsBig;
          if (__any_sync(0xFFFFFFFFu, hit)) {  // warp-uniform: the room check and the flush are collective
            if (*wq_cnt > kWqCap - kWqStep) flush();
            if (hit) {
#pragma unroll
              for (int j = 0; j < 8; ++j)
                if (v[8 * g8 + j] <= kTsBig)
                  wq[atomicAdd(const_cast<uint32_t*>(wq_cnt), 1u)] =
                      make_uint4(lut_row0 + c0 + 8 * g8 + j, v[8 * g8 + j], p, FILT ? leaf : 0u);
            }
            __syncwarp();
          }
        }
      }
    };
    uint32_t ts = 0;
    for (uint32_t item = blockIdx.x; item < n_items; item += gridDim.x) {
      const uint4 I = a.items[item];
      const uint32_t ncol = (a.groups[I.x].z + 15u) & ~15u;
      const uint32_t leaf_n = static_cast<uint32_t>(a.pt_off[I.w + 1] - a.pt_off[I.w]);
      const uint32_t lut_row0 = I.x * kTcsGroup;
      const uint32_t cb = half_id * 64;                                  // first column of this warp
      const uint32_t nmine = ncol > cb ? min(64u, ncol - cb) : 0u;       // live columns of this warp: 0, 16, .., 64
      for (uint32_t t = I.y; t < I.z; ++t, ++ts) {
        const uint32_t as = ts & 1u;
        const uint32_t p = t * kTcsTile + row;
        const bool valid = p < leaf_n;
        mbar_wait(bar(kTFull + as), (ts >> 1) & 1u, 0x700000u + ts);
        tc_fence_after();
        const uint32_t taddr = tmem + lane_addr + as * kTcsGroup + cb;
        uint32_t v0[32];
        if (nmine > 0) {
          tc_ld32_nowait(taddr, v0);
          tc_wait_ld();
        }
        if (nmine <= 32) {  // this warp's part of the accumulator is in registers: hand it back to the MMA warp
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(bar(kTEmpty + as));
        }
        if (nmine > 0) filter32(v0, cb, min(32u, nmine), valid, lut_row0, p, I.w);
        if (nmine > 32) {
          tc_ld32_nowait(taddr + 32, v0);
          tc_wait_ld();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(bar(kTEmpty + as));
          filter32(v0, cb + 32, nmine - 32, valid, lut_row0, p, I.w);
        }
      }
    }
    flush();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 3) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512) : "memory");
  }
}

// flags the queries the register-LUT kernel has to re-do (no bound / list overflow) and masks the tokens of all others
__global__ void tcs_flag_kernel(const uint32_t* __restrict__ tokens, size_t P, uint32_t L, uint32_t T,
                                const uint32_t* __restrict__ qcnt, uint32_t qcap, uint32_t* __restrict__ qflag,
                                uint32_t* __restrict__ fb_tokens) {
  const size_t p = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (p >= P) return;
  const uint32_t p32 = static_cast<uint32_t>(p);
  const uint32_t q = p32 / L, rank = p32 - q * L;
  const bool f = qflag[q] != 0u || qcnt[q] > qcap;
  fb_tokens[p] = (f && rank >= T) ? tokens[p] : kNoKey;  // ranks < T were scanned before the tensor-core pass
  if (f && rank == 0) qflag[q] = 1u;
}

// SCANN_TC_DEBUG=1: per-launch stage times and list statistics on stderr (synchronises; tuning only)
__global__ void tcs_debug_kernel(const uint32_t* __restrict__ qcnt, const uint32_t* __restrict__ qflag, size_t nq,
                                 uint32_t qcap, unsigned long long* __restrict__ out /* sum, max, flagged, overflowed */) {
  const size_t q = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (q >= nq) return;
  atomicAdd(&out[0], static_cast<unsigned long long>(qcnt[q]));
  atomicMax(&out[1], static_cast<unsigned long long>(qcnt[q]));
  if (qflag[q]) atomicAdd(&out[2], 1ull);
  if (qcnt[q] > qcap) atomicAdd(&out[3], 1ull);
}

}  // namespace

// ------------------------------------------------------------------------------------------------ host side
bool tc_scan_supported(size_t S, size_t dim) {
  return S >= 8 && S <= 64 && S % 8 == 0 && (S / 8) % 2 == 0 && dim % S == 0 && dim * 4 * 8 + S * 16 * 8 <= 48 * 1024;
}

size_t tc_scan_max_groups(size_t P, size_t K) { return P / kTcsGroup + std::min(K, P) + 1; }

size_t tc_scan_max_items(size_t P, size_t K, size_t max_leaf) {
  const size_t tiles = (max_leaf + kTcsTile - 1) / kTcsTile;
  return tc_scan_max_groups(P, K) * std::max<size_t>(1, (tiles + kTcsItemTiles - 1) / kTcsItemTiles);
}

size_t tc_scan_workspace_bytes(size_t nq, size_t L, size_t K, size_t S, size_t max_leaf, size_t qcap) {
  const size_t P = nq * L, G = tc_scan_max_groups(P, K);
  size_t b = 0;
  auto add = [&](size_t bytes) { b += Workspace::padded(bytes); };
  add(2 * K * 4);                       // leaf_cnt + cursor
  add(3 * (K + 1) * 4);                 // pair / group / item starts
  add(16);                              // counters
  add(P * 4);                           // sorted pairs
  add(G * 16);                          // groups
  add(tc_scan_max_items(P, K, max_leaf) * 16);
  add(G * kTcsGroup * (S * 16 + 32));   // LUT tiles
  add(G * kTcsGroup * 16);              // meta
  add(nq * qcap * 8);                   // candidate lists
  add(nq * 4);                          // counts
  add(nq * 4);                          // flags
  add(P * 4);                           // masked tokens
  return b + 4096;
}

scann_status launch_tc_scan(const TcScanParams& p, Workspace& ws, TcScanOut* out, cudaStream_t s) {
  const size_t K = p.K, P = p.nq * p.L, S = p.S;
  const size_t G = tc_scan_max_groups(P, K), I = tc_scan_max_items(P, K, p.max_leaf);
  const int row_bytes = static_cast<int>(S * 16 + 32);
  uint32_t* leaf_cnt = ws.take<uint32_t>(2 * K);
  uint32_t* cursor = leaf_cnt + K;
  uint32_t* starts = ws.take<uint32_t>(3 * (K + 1));
  uint32_t *pair_start = starts, *group_start = starts + (K + 1), *item_start = starts + 2 * (K + 1);
  uint32_t* counters = ws.take<uint32_t>(4);
  uint32_t* sorted_pairs = ws.take<uint32_t>(P);
  uint4* groups = ws.take<uint4>(G);
  uint4* items = ws.take<uint4>(I);
  uint8_t* lut = ws.take<uint8_t>(G * kTcsGroup * row_bytes);
  uint4* meta = ws.take<uint4>(G * kTcsGroup);
  unsigned long long* qcand = ws.take<unsigned long long>(p.nq * p.qcap);
  uint32_t* qcnt = ws.take<uint32_t>(p.nq);
  uint32_t* qflag = ws.take<uint32_t>(p.nq);
  uint32_t* fb_tokens = ws.take<uint32_t>(P);

  const char* dbg_env = getenv("SCANN_TC_DEBUG");
  const bool dbg = dbg_env && dbg_env[0] == '1';
  cudaEvent_t ev[5];
  if (dbg)
    for (auto& e : ev) cudaEventCreate(&e);
  if (dbg) cudaEventRecord(ev[0], s);
  SCANN_CUDA(cudaMemsetAsync(qcnt, 0, p.nq * 4, s));
  SCANN_CUDA(cudaMemsetAsync(qflag, 0, p.nq * 4, s));
  const unsigned pb = static_cast<unsigned>((P + 255) / 256);
  // The count and scatter passes are atomics on 4-byte counters (8 per 32-byte sector: ~1300 serialised updates per
  // sector at C3, 0.09 ms each).  The caller's worklist has usually grouped the same pairs already (class B of
  // treeah.cu's build_worklist): then only the group / item tables are built here.
  const bool reuse = p.wl_cnt != nullptr && p.wl_pair_start != nullptr && p.wl_sorted_pairs != nullptr;
  const uint32_t* cnt_in = leaf_cnt;
  const uint32_t* pairs_in = sorted_pairs;
  if (reuse) {
    cnt_in = p.wl_cnt;
    pairs_in = p.wl_sorted_pairs;
  } else {
    SCANN_CUDA(cudaMemsetAsync(leaf_cnt, 0, 2 * K * 4, s));
    tcwl_count_kernel<<<pb, 256, 0, s>>>(p.tokens, P, static_cast<uint32_t>(K), static_cast<uint32_t>(p.L),
                                         static_cast<uint32_t>(p.T), p.pt_off, leaf_cnt);
  }
  tcwl_scan_kernel<<<1, 1024, 0, s>>>(cnt_in, static_cast<uint32_t>(K), p.leaf_perm, p.pt_off, pair_start, group_start,
                                      item_start, counters, p.pair_points);
  if (!reuse)
    tcwl_scatter_kernel<<<pb, 256, 0, s>>>(p.tokens, P, static_cast<uint32_t>(K), static_cast<uint32_t>(p.L),
                                           static_cast<uint32_t>(p.T), p.pt_off, pair_start, cursor, sorted_pairs);
  tcwl_items_kernel<<<static_cast<unsigned>((K + 127) / 128), 128, 0, s>>>(cnt_in, static_cast<uint32_t>(K), p.pt_off,
                                                                          reuse ? p.wl_pair_start : pair_start,
                                                                          group_start, item_start, groups, items);
  if (dbg) cudaEventRecord(ev[1], s);
  if (p.ev[0]) cudaEventRecord(p.ev[0], s);
  LutArgs la;
  la.groups = groups;
  la.counters = counters;
  la.sorted_pairs = pairs_in;
  la.queries = p.queries;
  la.centers = p.centers;
  la.codebook = p.codebook;
  la.qthr = p.qthr;
  la.lut = lut;
  la.meta = meta;
  la.qflag = qflag;
  la.dim = static_cast<int>(p.dim);
  la.S = static_cast<int>(S);
  la.ds = static_cast<int>(p.dim / S);
  la.L = static_cast<int>(p.L);
  la.use_residuals = p.use_residuals;
  la.row_bytes = row_bytes;
  const size_t lsm = 8 * p.dim * sizeof(float) + (la.ds <= 2 ? S * 16 * la.ds * sizeof(float) : 0);
  const unsigned lgrid = static_cast<unsigned>(p.sms * (la.ds <= 2 ? 4 : 2));  // = the resident CTAs (persistent row loop)
  if (la.ds == 1) tc_lut_kernel<1><<<lgrid, 256, lsm, s>>>(la);
  else if (la.ds == 2) tc_lut_kernel<2><<<lgrid, 256, lsm, s>>>(la);
  else tc_lut_kernel<0><<<lgrid, 256, lsm, s>>>(la);
  SCANN_CUDA(cudaGetLastError());

  if (dbg) cudaEventRecord(ev[2], s);
  if (p.ev[1]) cudaEventRecord(p.ev[1], s);
  alignas(64) CUtensorMap tmB;
  SCANN_TRY(tc_make_map_u8(&tmB, lut, G * kTcsGroup, static_cast<size_t>(row_bytes)));
  TcsArgs a;
  a.codes_rm = p.codes_rm;
  a.pt_off = p.pt_off;
  a.groups = groups;
  a.items = items;
  a.counters = counters;
  a.meta = meta;
  a.qcand = qcand;
  a.qcnt = qcnt;
  a.qcap = static_cast<uint32_t>(p.qcap);
  a.nq = static_cast<uint32_t>(p.nq);
  a.err = counters + 2;
  for (int i = 0; i < 8; ++i) a.xm.sh[i] = 1u << (28 - 4 * i);
  a.xm.eight = 8u;
  a.KA = static_cast<int>(S / 8);
  a.bpp = static_cast<int>(S / 2);
  a.L = static_cast<int>(p.L);
  TcsFilter tf;
  tf.allow = p.allow;
  tf.allow_stride = p.allow_stride;
  tf.qfilt = p.qfilt;
  tf.blk_off = p.blk_off;
  tf.num_filters = p.num_filters;
  const bool filt = p.allow != nullptr;
  // >= 120 KB keeps it at one CTA per SM for every S (a second resident CTA would block in tcgen05.alloc)
  const size_t smem = std::max<size_t>(120 * 1024, 1024 + static_cast<size_t>(a.KA + 1) * kTsAtom + 32 * 8 + 64 +
                                                       8 * kWqCap * 16 + 64);
  const char* eg_env = getenv("SCANN_TC_EXP");
  const bool eg4 = eg_env && eg_env[0] == '4';
  auto kern = eg4 ? (filt ? tc_scan_kernel<4, true> : tc_scan_kernel<4, false>)
                  : (filt ? tc_scan_kernel<2, true> : tc_scan_kernel<2, false>);
  SCANN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  static uint32_t* h_dbg = nullptr;
  if (dbg && h_dbg == nullptr) {
    uint32_t* d_dbg = nullptr;
    if (cudaHostAlloc(&h_dbg, 64 * 4, cudaHostAllocMapped) == cudaSuccess &&
        cudaHostGetDevicePointer(&d_dbg, h_dbg, 0) == cudaSuccess) {
      memset(h_dbg, 0, 64 * 4);
      cudaMemcpyToSymbol(g_tcs_dbg, &d_dbg, sizeof(d_dbg));
    }
  }
  kern<<<p.sms, ts_threads(eg4 ? 4 : 2), smem, s>>>(tmB, a, tf);
  SCANN_CUDA(cudaGetLastError());
  if (dbg) {
    cudaError_t e = cudaStreamSynchronize(s);
    if (e != cudaSuccess && h_dbg)
    {
      fprintf(stderr, "[tcscan] scan kernel failed (%s): timed-out wait = %u, barrier smem 0x%x, parity %u, tag 0x%x, cta %u, thread %u\n",
              cudaGetErrorString(e), h_dbg[0], h_dbg[1], h_dbg[2], h_dbg[3], h_dbg[4], h_dbg[5]);
      fprintf(stderr, "[tcscan] cta 0 progress marks (warp: value):");
      for (int w = 0; w < 14; ++w) fprintf(stderr, " %d:0x%x", w, h_dbg[8 + w]);
      fprintf(stderr, "\n");
    }
  }
  if (dbg) cudaEventRecord(ev[3], s);
  if (p.ev[2]) cudaEventRecord(p.ev[2], s);
  tcs_flag_kernel<<<pb, 256, 0, s>>>(p.tokens, P, static_cast<uint32_t>(p.L), static_cast<uint32_t>(p.T), qcnt,
                                     static_cast<uint32_t>(p.qcap), qflag, fb_tokens);
  SCANN_CUDA(cudaGetLastError());
  if (dbg) {
    cudaEventRecord(ev[4], s);
    unsigned long long* d_st = nullptr;
    unsigned long long st[4] = {0, 0, 0, 0};
    uint32_t cnt[3] = {0, 0, 0};
    cudaMalloc(&d_st, sizeof(st));
    cudaMemsetAsync(d_st, 0, sizeof(st), s);
    tcs_debug_kernel<<<static_cast<unsigned>((p.nq + 255) / 256), 256, 0, s>>>(qcnt, qflag, p.nq,
                                                                              static_cast<uint32_t>(p.qcap), d_st);
    cudaStreamSynchronize(s);
    cudaMemcpy(st, d_st, sizeof(st), cudaMemcpyDeviceToHost);
    cudaMemcpy(cnt, counters, sizeof(cnt), cudaMemcpyDeviceToHost);
    cudaFree(d_st);
    float t[4];
    for (int i = 0; i < 4; ++i) cudaEventElapsedTime(&t[i], ev[i], ev[i + 1]);
    fprintf(stderr,
            "[tcscan] nq=%zu L=%zu items=%u groups=%u | worklist %.3f ms, lut %.3f ms, scan %.3f ms, flag %.3f ms | "
            "candidates/query mean %.1f max %llu (cap %zu), flagged %llu, overflowed %llu, errors %u\n",
            p.nq, p.L, cnt[0], cnt[1], t[0], t[1], t[2], t[3], static_cast<double>(st[0]) / static_cast<double>(p.nq), st[1],
            p.qcap, st[2], st[3], cnt[2]);
    for (auto& e : ev) cudaEventDestroy(e);
  }
  out->qcand = qcand;
  out->qcnt = qcnt;
  out->qflag = qflag;
  out->fb_tokens = fb_tokens;
  out->launches = reuse ? 5 : 7;  // kernels of this function (memsets are not counted)
  return SCANN_OK;
}

}  // namespace scann
