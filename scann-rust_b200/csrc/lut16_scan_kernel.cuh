// The Tree-AH hot kernel: persistent LUT16 scan over (leaf, <=G queries) work items.
//
// Per work item a CTA of kScanWarps = 8 warps
//   (1) stages the G query residuals q - centroid(leaf) in shared memory,
//   (2) builds the G residual LUT16 tables (warp g builds table g; bit-exact quantiser, lut16_device.cuh),
//   (3) turns the batch-wide upper bound tau_q of every query (see below) into an integer score bound
//       for THIS leaf's quantisation,
//   (4) streams the leaf's blocked 4-bit codes once for all G queries — one 256-point block per warp per
//       tile, register-LUT PRMT lookups on the ALU pipe, integer accumulation on the FMA pipe,
//   (5) keeps an exact running top-R per query: packed-min prefilter -> exact key filter -> append to a
//       shared-memory buffer -> warp radix select when the buffer could overflow,
//   (6) writes the <= R survivors (approx distance, position) of every (query, leaf) pair.
//
// tau_q (qthr[]): a per-query upper bound on the R-th smallest approximate distance over ALL probed
// leaves, shared through global memory.  Whenever a leaf has produced R candidates for a query, the
// distance of its R-th best is a valid bound (that leaf alone already holds R points at or below it) and
// is published with atomicMin.  Work items that run later drop everything above the bound up front.
// The bound only removes points that cannot be among the global top-R by (distance, leaf rank, position),
// so the final result is independent of the order in which work items happen to run.
#pragma once

#include "lut16_device.cuh"

namespace scann {

struct ScanArgs {
  const uint4* codes;
  const uint32_t* blk_off;
  const uint64_t* pt_off;
  const float* centers;
  const float* codebook;
  const float* queries;
  const uint4* items;
  const uint32_t* sorted_pairs;
  uint32_t* counters;  // [0] total items, [1] next item, [2] class-A items (closest-leaf pairs, scanned first)
  int end_idx;         // this launch stops at counters[end_idx]: 0 = every item, 2 = the class-A items only
  const uint8_t* allow;  // restrict filters (search_with_filter): [num_filters][total blocks * 32] bytes, bit i of byte
                         // (row, block, lane) = point lane*8+i of that block is allowed by filter `row`; nullptr = none
  uint32_t sentinel;     // 255*S + 1: the integer score given to filtered-out points (above every real score)
  int max_blocks;      // > 0: probe launch — scan only the first max_blocks 256-point blocks of each leaf and publish
                       // the bound they prove (any R points give a valid bound); candidates are not written
  uint32_t* qthr;      // [nq] f32_key of the best known bound on the R-th approx distance (0xFFFFFFFF = none)
  uint2* cand;         // [P][R] {approx distance bits, position in leaf}
  uint32_t* cand_cnt;  // [P]
  int dim, S, ds, SG, L, R, cap, pos_bits, use_residuals;
  AccMul mul;
  size_t allow_stride;    // bytes per filter row of `allow`
  const uint32_t* qfilt;  // [nq] filter row of every query of the chunk; nullptr = row 0 for every query
  uint32_t num_filters;   // rows of `allow`: a query whose row is >= num_filters is allowed nothing
  const uint32_t* qR;     // [nq] pre-reorder R of every query of the chunk (scann_treeah_search_with_params; a query
                          // with R_q == 0 has no pairs), read where it is used so that the shared-memory layout stays
                          // as it is; nullptr = R for every query.  The list stride and `cap` stay at R.
};

// largest integer score s with dequant(s) <= tau, as an exclusive key bound ((s+1) << pos_bits);
// 0 when even s = 0 is above tau.  dequant is monotone non-decreasing in s.
__device__ __forceinline__ uint32_t key_bound_from_tau(float tau, float mult, float biasS, int pos_bits) {
  const uint32_t smax_all = (pos_bits >= 32) ? 0u : ((0xFFFFFFFFu >> pos_bits) - 1u);  // keep (s+1)<<pos_bits in range
  float est = __fdiv_rn(__fsub_rn(tau, biasS), mult);
  long long s;
  if (!(est == est)) return 0xFFFFFFFFu;
  if (est < -1.0f) s = -1;
  else if (est > static_cast<float>(smax_all)) s = smax_all;
  else s = static_cast<long long>(floorf(est));
  for (int it = 0; it < 8 && s < static_cast<long long>(smax_all) &&
                   lut16_dequant(static_cast<uint32_t>(s + 1), mult, biasS) <= tau; ++it) ++s;
  for (int it = 0; it < 8 && s >= 0 && lut16_dequant(static_cast<uint32_t>(s), mult, biasS) > tau; ++it) --s;
  if (s >= 0 && lut16_dequant(static_cast<uint32_t>(s), mult, biasS) > tau) return 0xFFFFFFFFu;  // did not converge: no bound
  if (s < static_cast<long long>(smax_all) && lut16_dequant(static_cast<uint32_t>(s + 1), mult, biasS) <= tau)
    return 0xFFFFFFFFu;
  if (s < 0) return 0u;
  return static_cast<uint32_t>(s + 1) << pos_bits;
}

// 8 warps per scan CTA (2 CTAs/SM), for this kernel and lut_f32_scan_kernel.  Measured on B200 at C3: 8 warps 35.6 ms,
// 4 warps 35.8 ms, 2 warps 44.7 ms (profiles/r1_scan_kernel.md).
constexpr int kScanWarps = 8;

// MODE = scan_acc_mode(S) (lut16_device.cuh); FILT: restrict filters (a template flag, so the unfiltered kernel carries
// none of it)
template <int G, int MODE, bool FILT>
__global__ void __launch_bounds__(kScanWarps * 32, 16 / kScanWarps) lut16_scan_kernel(const ScanArgs a) {
  extern __shared__ __align__(16) uint8_t smem[];
  const int S4 = a.SG * 4;
  uint4* lut = reinterpret_cast<uint4*>(smem);                                  // [G][S4]
  float* qres = reinterpret_cast<float*>(lut + G * S4);                         // [G][dim]
  uint32_t* buf = reinterpret_cast<uint32_t*>(qres + ((G * a.dim + 3) & ~3));   // [G][cap], 16-B aligned
  uint32_t* hist = buf + static_cast<size_t>(G) * a.cap;                        // [kScanWarps][256]
  float* s_mult = reinterpret_cast<float*>(hist + kScanWarps * 256);
  float* s_bias = s_mult + G;
  uint32_t* s_thr = reinterpret_cast<uint32_t*>(s_bias + G);   // exclusive key bound per query
  uint32_t* s_cnt = s_thr + G;                                 // candidates buffered per query
  uint32_t* s_pair = s_cnt + G;                                // pair id (q * L + rank)
  uint32_t* s_tau = s_pair + G;                                // last tau key seen per query
  uint32_t* s_item = s_tau + G;
  uint32_t* s_row = s_item + 1;                                // FILT: filter row per query (0xFFFFFFFF = none allowed)

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t total_items = a.counters[a.end_idx];
  const uint32_t pos_mask = (1u << a.pos_bits) - 1u;

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
    int nblk = static_cast<int>(a.blk_off[leaf + 1] - blk0);
    uint32_t leaf_n = static_cast<uint32_t>(a.pt_off[leaf + 1] - a.pt_off[leaf]);
    if (a.max_blocks > 0 && nblk > a.max_blocks) {
      nblk = a.max_blocks;
      leaf_n = static_cast<uint32_t>(nblk) * kBlockPts;
    }

    // (1) query residuals: q - centroid (src/tree_x_hybrid/mod.rs:309-316)
    for (int idx = tid; idx < G * a.dim; idx += kScanWarps * 32) {
      int g = idx / a.dim, d = idx - g * a.dim;
      float v = 0.0f;
      if (g < ng) {
        uint32_t pair = a.sorted_pairs[pbeg + g];
        uint32_t q = pair / static_cast<uint32_t>(a.L);
        v = a.queries[static_cast<size_t>(q) * a.dim + d];
        if (a.use_residuals) v = __fsub_rn(v, __ldg(a.centers + static_cast<size_t>(leaf) * a.dim + d));
      }
      qres[idx] = v;
    }
    if (tid < G) s_pair[tid] = tid < ng ? a.sorted_pairs[pbeg + tid] : 0xFFFFFFFFu;
    if (FILT && tid < ng) {
      const uint32_t row = a.qfilt ? a.qfilt[a.sorted_pairs[pbeg + tid] / static_cast<uint32_t>(a.L)] : 0u;
      s_row[tid] = row < a.num_filters ? row : 0xFFFFFFFFu;
    }
    __syncthreads();

    // (2) LUT16 build (warp g builds query g's table) and (3) the bound for this leaf
    const int nfull0 = min(kScanWarps, static_cast<int>(leaf_n / kBlockPts));  // full blocks of tile 0
    for (int g = warp; g < G; g += kScanWarps) {
      uint8_t* l8 = reinterpret_cast<uint8_t*>(lut + g * S4);
      if (g < ng) {
        float mult, bias;
        warp_build_lut16(qres + g * a.dim, a.codebook, a.S, S4, a.ds, l8, &mult, &bias, lane);
        if (lane == 0) {
          const float biasS = __fmul_rn(bias, static_cast<float>(a.S));  // bias * S, rounded once (lut16_simd.rs:137)
          s_mult[g] = mult;
          s_bias[g] = biasS;
          const uint32_t q = s_pair[g] / static_cast<uint32_t>(a.L);
          const uint32_t tk = __ldcg(a.qthr + q);
          s_tau[g] = tk;
          uint32_t thr = 0xFFFFFFFFu;
          if (tk != 0xFFFFFFFFu) thr = key_bound_from_tau(key_f32(tk), mult, biasS, a.pos_bits);
          s_thr[g] = thr;
          // without a bound the full blocks of tile 0 are stored unfiltered at fixed slots
          s_cnt[g] = thr == 0xFFFFFFFFu ? static_cast<uint32_t>(nfull0) * kBlockPts : 0u;
        }
      } else {
        for (int e = lane; e < S4 * 16; e += 32) l8[e] = 0;
        if (lane == 0) {
          s_thr[g] = 0u;
          s_cnt[g] = 0u;
        }
      }
    }
    __syncthreads();

    // (4)+(5) stream the leaf, one 256-point block per warp per tile
    const int ntiles = (nblk + kScanWarps - 1) / kScanWarps;
    for (int t = 0; t < ntiles; ++t) {
      const int b = t * kScanWarps + warp;
      if (b < nblk) {
        PackedSums ps[G];
        {
          // remainder items carry fewer than G queries: the lookups of the unused tables are skipped by running the
          // narrower instantiation (the code-only work is per block either way)
          const uint4* cb = a.codes + (static_cast<size_t>(blk0) + b) * a.SG * 32;
          if (G >= 8 && ng <= 2) {
            PackedSums p2[2];
            scan_block<2, MODE>(cb, a.SG, lut, S4, lane, a.mul, p2);
            ps[0] = p2[0];
            ps[1] = p2[1];
          } else if (G >= 8 && ng <= 4) {
            PackedSums p4[4];
            scan_block<4, MODE>(cb, a.SG, lut, S4, lane, a.mul, p4);
#pragma unroll
            for (int g = 0; g < 4; ++g) ps[g] = p4[g];
          } else {
            scan_block<G, MODE>(cb, a.SG, lut, S4, lane, a.mul, ps);
          }
        }
        if (FILT) {
          // RestrictFilter::is_allowed (tree_x_hybrid/mod.rs:327-332): filtered-out points never enter a top-R; here
          // their score becomes the sentinel, which sorts after every real score and is dropped at the output.  Every
          // query of the item reads the byte of its own filter row.
          const size_t at = (static_cast<size_t>(blk0) + b) * 32 + lane;
#pragma unroll
          for (int g = 0; g < G; ++g) {
            if (g >= ng) continue;
            const uint32_t row = s_row[g];
            const uint32_t am = row == 0xFFFFFFFFu ? 0u : a.allow[row * a.allow_stride + at];
            if (am == 0xFFu) continue;
            const uint32_t lo = 0x0000FFFFu, hi = 0xFFFF0000u, sl = a.sentinel, sh = a.sentinel << 16;
            const uint32_t k_ea = ((am & 1u) ? lo : 0u) | ((am & 4u) ? hi : 0u), k_xa = ((am & 2u) ? lo : 0u) | ((am & 8u) ? hi : 0u);
            const uint32_t k_eb = ((am & 16u) ? lo : 0u) | ((am & 64u) ? hi : 0u), k_xb = ((am & 32u) ? lo : 0u) | ((am & 128u) ? hi : 0u);
            const uint32_t v_ea = ((am & 1u) ? 0u : sl) | ((am & 4u) ? 0u : sh), v_xa = ((am & 2u) ? 0u : sl) | ((am & 8u) ? 0u : sh);
            const uint32_t v_eb = ((am & 16u) ? 0u : sl) | ((am & 64u) ? 0u : sh), v_xb = ((am & 32u) ? 0u : sl) | ((am & 128u) ? 0u : sh);
            ps[g].ea = (ps[g].ea & k_ea) | v_ea;
            ps[g].xa = (ps[g].xa & k_xa) | v_xa;
            ps[g].eb = (ps[g].eb & k_eb) | v_eb;
            ps[g].xb = (ps[g].xb & k_xb) | v_xb;
          }
        }
        const uint32_t pos0 = static_cast<uint32_t>(b) * kBlockPts + lane * 8;
#pragma unroll
        for (int g = 0; g < G; ++g) {
          if (g >= ng) continue;
          const uint32_t thr = s_thr[g];
          uint32_t* bg = buf + static_cast<size_t>(g) * a.cap;
          if (thr == 0xFFFFFFFFu && t == 0 && b < nfull0) {
            uint32_t s[8];
            unpack_sums(ps[g], s);
            uint4* dst = reinterpret_cast<uint4*>(bg + pos0);
            dst[0] = make_uint4((s[0] << a.pos_bits) | (pos0 + 0), (s[1] << a.pos_bits) | (pos0 + 1),
                                (s[2] << a.pos_bits) | (pos0 + 2), (s[3] << a.pos_bits) | (pos0 + 3));
            dst[1] = make_uint4((s[4] << a.pos_bits) | (pos0 + 4), (s[5] << a.pos_bits) | (pos0 + 5),
                                (s[6] << a.pos_bits) | (pos0 + 6), (s[7] << a.pos_bits) | (pos0 + 7));
          } else if (min_sum(ps[g]) <= ((thr - 1u) >> a.pos_bits) && thr != 0u) {
            // some point of this lane may qualify: exact key test (sum, position) < bound
            uint32_t s[8];
            unpack_sums(ps[g], s);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const uint32_t pos = pos0 + i;
              const uint32_t key = (s[i] << a.pos_bits) | pos;
              if (pos < leaf_n && key < thr) {
                uint32_t slot = atomicAdd(&s_cnt[g], 1u);
                if (slot < static_cast<uint32_t>(a.cap)) bg[slot] = key;
              }
            }
          }
        }
      }
      __syncthreads();
      // exact compaction to the R best when the buffer could overflow in the next tile; refresh tau
      for (int g = warp; g < ng; g += kScanWarps) {
        int c = static_cast<int>(min(s_cnt[g], static_cast<uint32_t>(a.cap)));
        const uint32_t q = s_pair[g] / static_cast<uint32_t>(a.L);
        const int R = a.qR ? static_cast<int>(__ldg(a.qR + q)) : a.R;
        uint32_t thr = s_thr[g];
        if (c > R && (t == ntiles - 1 || c > 2 * R)) {
          thr = warp_select_u32(buf + static_cast<size_t>(g) * a.cap, c, R, hist + warp * 256, lane);
          c = R;
          if (lane == 0) {
            s_cnt[g] = static_cast<uint32_t>(R);
            // this leaf alone holds R points at or below dist(thr): publish the bound (unless the R-th entry is a
            // filtered-out point: then fewer than R allowed points were seen and nothing is proved)
            if (!FILT || (thr >> a.pos_bits) < a.sentinel) {
              const float dR = lut16_dequant(thr >> a.pos_bits, s_mult[g], s_bias[g]);
              atomicMin(a.qthr + q, f32_key(dR));
            }
          }
        }
        if (lane == 0 && t + 1 < ntiles) {
          const uint32_t tk = __ldcg(a.qthr + q);
          if (tk < s_tau[g]) {  // somebody tightened the batch-wide bound
            s_tau[g] = tk;
            const uint32_t tb = key_bound_from_tau(key_f32(tk), s_mult[g], s_bias[g], a.pos_bits);
            if (tb < thr) thr = tb;
          }
          s_thr[g] = thr;
        } else if (lane == 0) {
          s_thr[g] = thr;
        }
      }
      __syncthreads();
    }

    // (6) write this item's candidates: approx distance = sum*multiplier + bias*S (lut16_simd.rs:136-140)
    if (a.max_blocks > 0) continue;  // probe launch: only the bounds matter
    for (int g = warp; g < ng; g += kScanWarps) {
      const uint32_t R = a.qR ? __ldg(a.qR + s_pair[g] / static_cast<uint32_t>(a.L)) : static_cast<uint32_t>(a.R);
      const int c = static_cast<int>(min(s_cnt[g], R));
      const uint32_t pair = s_pair[g];
      const float mult = s_mult[g], biasS = s_bias[g];
      const uint32_t* bg = buf + static_cast<size_t>(g) * a.cap;
      uint2* out = a.cand + static_cast<size_t>(pair) * a.R;
      if (!FILT) {
        for (int i = lane; i < c; i += 32) {
          uint32_t key = bg[i];
          float dist = lut16_dequant(key >> a.pos_bits, mult, biasS);
          out[i] = make_uint2(__float_as_uint(dist), key & pos_mask);
        }
        if (lane == 0) a.cand_cnt[pair] = static_cast<uint32_t>(c);
      } else {  // drop the filtered-out points that were kept only because the leaf has fewer than R allowed ones
        int w = 0;
        for (int base = 0; base < c; base += 32) {
          const int i = base + lane;
          const uint32_t key = i < c ? bg[i] : 0xFFFFFFFFu;
          const bool ok = i < c && (key >> a.pos_bits) < a.sentinel;
          const uint32_t bal = __ballot_sync(0xFFFFFFFFu, ok);
          if (ok) {
            const float dist = lut16_dequant(key >> a.pos_bits, mult, biasS);
            out[w + __popc(bal & lanemask_lt())] = make_uint2(__float_as_uint(dist), key & pos_mask);
          }
          w += __popc(bal);
        }
        if (lane == 0) a.cand_cnt[pair] = static_cast<uint32_t>(w);
      }
    }
  }
}

// entries of a query's shared-memory candidate buffer: one tile of unfiltered points + 2R carried, in 32-entry rows
inline int scan_list_cap(int R) { return (kScanWarps * kBlockPts + 2 * R + 31) / 32 * 32; }

inline size_t scan_smem_bytes(int G, int S4, int dim, int cap, bool filt) {
  return static_cast<size_t>(G) * S4 * 16 + static_cast<size_t>((G * dim + 3) & ~3) * 4 +
         static_cast<size_t>(G) * cap * 4 + kScanWarps * 256 * 4 + static_cast<size_t>(G) * (filt ? 7 : 6) * 4 + 16;
}

}  // namespace scann
