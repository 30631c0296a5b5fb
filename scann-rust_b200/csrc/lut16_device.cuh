// LUT16 device functions: per-query u8 table build (bit-exact restatement of the reference's
// quantiser) and the register-LUT block scan.  Shared by the Tree-AH hot kernel (treeah.cu) and the
// parity taps (taps.cu) so the taps exercise the same arithmetic as the product path.
//
// Code layout in HBM ("blocked"): the rows of one leaf are cut into blocks of 256 points.  A block is
// SG = ceil(S/4) groups x 32 lanes x uint4.  Lane l's uint4 of group sg holds, for subspaces
// 4*sg+0..3 (one u32 each), the eight 4-bit codes of points l*8+0..7 (nibble i = point l*8+i).
// A warp therefore streams a block with SG fully coalesced 512-byte LDG.128 requests, and every
// register is "one subspace x eight points" — the shape the PRMT lookup wants.
//
// Lookup: a 16-entry u8 table is 4 registers T0..T3.  PRMT(T0,T1,sel) looks 4 codes up in entries
// 0..7, PRMT(T2,T3,sel) in entries 8..15, and a byte mask made from bit 3 of each code picks between
// them.  Selector/mask preparation depends only on the codes, so it is shared by all G queries that
// scan the block together; per query the cost is 4 PRMT + 2 LOP3 per 8 lookups.
//
// Accumulation without widening every byte: with r = b0|b1<<8|b2<<16|b3<<24 (four points' values),
//   accE += r & 0x00FF00FF   -> low half Σb0, high half Σb2          (each < 2^16 for S <= 256)
//   accX += r >> 8           -> Σb1 + 2^8 Σb2 + 2^16 Σb3             (< 2^32 for S <= 256)
// and Σb1, Σb3 are recovered exactly at the end from accX - (Σb2 << 8).
#pragma once

#include "common.cuh"

namespace scann {

constexpr int kBlockPts = 256;   // points per code block (32 lanes x 8 nibbles)

// Accumulation mode of scan_block() for a table of S subspaces: 3 (IDP.2A, measured best on B200) where the per-point
// sums fit its 15-bit fields (S <= 128: 128 * 255 = 32640 < 2^15), else 2.
constexpr int scan_acc_mode(int S) { return S <= 128 ? 3 : 2; }

#ifdef __CUDACC__

// One f32 LUT entry: Σ_j (qres[s*ds+j] - cb[e*ds+j])², sequential, never fused.
// (src/hashes/lut16.rs:246-255 squared_l2_distance_slice; codebook.rs:106-115)
__device__ __forceinline__ float lut_entry(const float* __restrict__ qres, const float* __restrict__ cb, int e,
                                           int ds) {
  int s = e >> 4;
  float sum = 0.0f;
  for (int j = 0; j < ds; ++j) {
    float d = __fsub_rn(qres[s * ds + j], __ldg(cb + e * ds + j));
    sum = __fadd_rn(sum, __fmul_rn(d, d));
  }
  return sum;
}

// Warp-cooperative LUT16 build for one query (already residual-subtracted, in shared or global
// memory).  Restates Lut16LookupTables::from_query (src/hashes/lut16.rs:151-173) followed by
// Lut16SimdTables::from_float_tables (src/hashes/lut16_simd.rs:39-90):
//   global min/max over all S*16 entries; range < 1e-10 -> scale 1 (multiplier 1);
//   else scale = 255/range, multiplier = 1/scale; q = round_half_away((v-min)*scale) saturated to u8.
// lut8 receives S4*16 bytes ([s][16], rows S..S4-1 zeroed).  Lane 0 returns multiplier/bias.
// The f32 entries are computed once and kept in registers between the min/max pass and the quantise
// pass when the table is small enough (S <= 64, 32 entries per lane); larger tables recompute.
__device__ __forceinline__ uint8_t lut16_quantize_entry(float v, float mn, float scale) {
  float r = roundf(__fmul_rn(__fsub_rn(v, mn), scale));
  if (!(r == r)) return 0;  // Rust `as u8`: NaN -> 0, saturating
  if (r <= 0.0f) return 0;
  if (r >= 255.0f) return 255;
  return static_cast<uint8_t>(r);
}

__device__ __forceinline__ void warp_build_lut16(const float* __restrict__ qres, const float* __restrict__ cb,
                                                 int S, int S4, int ds, uint8_t* lut8, float* mult_out,
                                                 float* bias_out, int lane) {
  const int nent = S * 16;
  const bool cached = nent <= 32 * 32;
  float vals[32];
  float mn = 3.402823466e+38f, mx = -3.402823466e+38f;
  if (cached) {
#pragma unroll
    for (int t = 0; t < 32; ++t) {
      const int e = lane + 32 * t;
      vals[t] = 0.0f;
      if (e < nent) {
        vals[t] = lut_entry(qres, cb, e, ds);
        mn = fminf(mn, vals[t]);
        mx = fmaxf(mx, vals[t]);
      }
    }
  } else {
    for (int e = lane; e < nent; e += 32) {
      float v = lut_entry(qres, cb, e, ds);
      mn = fminf(mn, v);
      mx = fmaxf(mx, v);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mn = fminf(mn, __shfl_xor_sync(0xFFFFFFFFu, mn, o));
    mx = fmaxf(mx, __shfl_xor_sync(0xFFFFFFFFu, mx, o));
  }
  float range = __fsub_rn(mx, mn);
  float scale = 1.0f, mult = 1.0f;
  if (!(range < 1e-10f)) {
    scale = __fdiv_rn(255.0f, range);
    mult = __fdiv_rn(1.0f, scale);
  }
  if (cached) {
#pragma unroll
    for (int t = 0; t < 32; ++t) {
      const int e = lane + 32 * t;
      if (e < S4 * 16) lut8[e] = e < nent ? lut16_quantize_entry(vals[t], mn, scale) : 0;
    }
  } else {
    for (int e = lane; e < S4 * 16; e += 32)
      lut8[e] = e < nent ? lut16_quantize_entry(lut_entry(qres, cb, e, ds), mn, scale) : 0;
  }
  if (lane == 0) {
    *mult_out = mult;
    *bias_out = mn;
  }
}

// Dequantisation of one u32 accumulator: sum as f32 * multiplier + bias * S
// (src/hashes/lut16_simd.rs:136-140; bias_total is rounded first, then mul and add unfused)
__device__ __forceinline__ float lut16_dequant(uint32_t sum, float mult, float bias_total) {
  return __fadd_rn(__fmul_rn(static_cast<float>(sum), mult), bias_total);
}

// Packed per-lane accumulators of one (query, block): u16 halves hold the sums of points
//   ea = (p0 | p2 << 16), xa = (p1 | p3 << 16), eb = (p4 | p6 << 16), xb = (p5 | p7 << 16)   (p_i = point lane*8+i)
struct PackedSums {
  uint32_t ea, xa, eb, xb;
};
__device__ __forceinline__ void unpack_sums(const PackedSums& p, uint32_t (&s)[8]) {
  s[0] = p.ea & 0xFFFFu;
  s[2] = p.ea >> 16;
  s[1] = p.xa & 0xFFFFu;
  s[3] = p.xa >> 16;
  s[4] = p.eb & 0xFFFFu;
  s[6] = p.eb >> 16;
  s[5] = p.xb & 0xFFFFu;
  s[7] = p.xb >> 16;
}
// smallest of the eight sums (two packed u16 minima, then the halves)
__device__ __forceinline__ uint32_t min_sum(const PackedSums& p) {
  uint32_t m = __vminu2(__vminu2(p.ea, p.xa), __vminu2(p.eb, p.xb));
  return min(m & 0xFFFFu, m >> 16);
}

// Pipe balancing: the PRMT/LOP3 lookups saturate the ALU pipe, so the accumulation is issued on the
// FMA pipe as integer multiply-adds.  The multipliers are kernel parameters so the compiler cannot
// strength-reduce them back into ALU-pipe adds.
struct AccMul {
  uint32_t one, w15;  // 1 (MODE 2), (1 | 2^15 << 16): the IDP.2A weight pair of MODE 3
};
// MODE 2: masked add on the FMA pipe (acc_e = (r & 0x00FF00FF) * one + acc_e, IMAD), shifted add on the ALU pipe
__device__ __forceinline__ void acc_add(uint32_t& acc_e, uint32_t& acc_x, uint32_t r, const AccMul& m) {
  const uint32_t e = r & 0x00FF00FFu;
  asm("mad.lo.u32 %0, %1, %2, %0;" : "+r"(acc_e) : "r"(e), "r"(m.one));
  acc_x += r >> 8;
}

// Scan one 256-point block for G queries.  lut: shared memory, [G][S4] uint4 (one 16-entry u8
// table per (query, subspace)).  On return out[g] holds the eight u32 accumulators of points
// lane*8+0..7 in packed form — the same integers src/simd/dispatch.rs:259-295 computes.
// MODE = scan_acc_mode(S).
//
// MODE 3 (S <= 128): the four bytes of a lookup result r are accumulated by two IDP.2A instructions on
// the FMA pipe with the constant weight pair w = (1, 2^15):
//   acc01 += b0 + 2^15 * b1      (dp2a.lo)        acc23 += b2 + 2^15 * b3      (dp2a.hi)
// Each per-point sum is < 2^15 for S <= 128 (128 * 255 = 32640), so the two 15-bit fields never carry
// into each other and the accumulators stay below 2^30.  No mask, no shift: the ALU pipe only carries
// the three lookup instructions (PRMT, PRMT, LOP3) per four lookups.
template <int G, int MODE>
__device__ __forceinline__ void scan_block(const uint4* __restrict__ blk, int SG, const uint4* __restrict__ lut,
                                           int S4, int lane, const AccMul mul, PackedSums (&out)[G]) {
  static_assert(MODE == 2 || MODE == 3, "accumulation mode");
  uint32_t accEA[G], accXA[G], accEB[G], accXB[G];
#pragma unroll
  for (int g = 0; g < G; ++g) accEA[g] = accXA[g] = accEB[g] = accXB[g] = 0;

  uint4 c = __ldg(blk + lane);
  for (int sg = 0; sg < SG; ++sg) {
    uint4 cn = make_uint4(0, 0, 0, 0);
    if (sg + 1 < SG) cn = __ldg(blk + (sg + 1) * 32 + lane);
    const uint32_t cw[4] = {c.x, c.y, c.z, c.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t C = cw[j];
      const uint32_t selA = C & 0x77777777u;
      const uint32_t selB = selA >> 16;
      const uint32_t tm = (C >> 3) & 0x11111111u;
      const uint32_t mA = __byte_perm(0x0000FF00u, 0u, tm);
      const uint32_t mB = __byte_perm(0x0000FF00u, 0u, tm >> 16);
      const int s = sg * 4 + j;
#pragma unroll
      for (int g = 0; g < G; ++g) {
        const uint4 T = lut[g * S4 + s];
        const uint32_t loA = __byte_perm(T.x, T.y, selA);
        const uint32_t hiA = __byte_perm(T.z, T.w, selA);
        const uint32_t rA = (loA & ~mA) | (hiA & mA);
        const uint32_t loB = __byte_perm(T.x, T.y, selB);
        const uint32_t hiB = __byte_perm(T.z, T.w, selB);
        const uint32_t rB = (loB & ~mB) | (hiB & mB);
        if (MODE == 3) {
          asm("dp2a.lo.u32.u32 %0, %1, %2, %0;" : "+r"(accEA[g]) : "r"(mul.w15), "r"(rA));
          asm("dp2a.hi.u32.u32 %0, %1, %2, %0;" : "+r"(accXA[g]) : "r"(mul.w15), "r"(rA));
          asm("dp2a.lo.u32.u32 %0, %1, %2, %0;" : "+r"(accEB[g]) : "r"(mul.w15), "r"(rB));
          asm("dp2a.hi.u32.u32 %0, %1, %2, %0;" : "+r"(accXB[g]) : "r"(mul.w15), "r"(rB));
        } else {
          acc_add(accEA[g], accXA[g], rA, mul);
          acc_add(accEB[g], accXB[g], rB, mul);
        }
      }
    }
    c = cn;
  }
#pragma unroll
  for (int g = 0; g < G; ++g) {
    if (MODE == 3) {  // (p0 | p1 << 15), (p2 | p3 << 15)  ->  (p0 | p2 << 16), (p1 | p3 << 16)
      out[g].ea = (accEA[g] & 0x7FFFu) | ((accXA[g] & 0x7FFFu) << 16);
      out[g].xa = (accEA[g] >> 15) | ((accXA[g] >> 15) << 16);
      out[g].eb = (accEB[g] & 0x7FFFu) | ((accXB[g] & 0x7FFFu) << 16);
      out[g].xb = (accEB[g] >> 15) | ((accXB[g] >> 15) << 16);
    } else {
      out[g].ea = accEA[g];
      out[g].xa = accXA[g] - ((accEA[g] >> 16) << 8);  // Σb1 + 2^16 Σb3
      out[g].eb = accEB[g];
      out[g].xb = accXB[g] - ((accEB[g] >> 16) << 8);
    }
  }
}

// ---- warp-level exact selection on u32 keys in shared memory -----------------------------------
// One radix digit: given a 256-bin histogram (shared memory of the warp) of the keys still in play and the rank
// need >= 1 among them, d = the bin that holds the need-th smallest and below = the keys in the bins before it.
__device__ __forceinline__ void warp_hist_digit(const uint32_t* hist, uint32_t need, int lane, uint32_t& d,
                                                uint32_t& below) {
  uint32_t h[8];
  uint32_t s = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    h[j] = hist[lane * 8 + j];
    s += h[j];
  }
  uint32_t incl = s;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
    if (lane >= o) incl += v;
  }
  uint32_t excl = incl - s;
  bool mine = (excl < need) && (need <= incl);
  d = 0;
  below = 0;
  if (mine) {
    uint32_t run = excl;
    bool found = false;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (!found && run + h[j] >= need) {
        d = lane * 8 + j;
        below = run;
        found = true;
      }
      if (!found) run += h[j];
    }
  }
  uint32_t owner = __ffs(__ballot_sync(0xFFFFFFFFu, mine)) - 1;
  d = __shfl_sync(0xFFFFFFFFu, d, owner);
  below = __shfl_sync(0xFFFFFFFFu, below, owner);
}

// Finds T = the R-th smallest of the c distinct keys in buf (1 <= R < c), compacts buf in place to the
// R keys <= T and returns T.  hist: 256 u32 of shared memory private to the warp.
__device__ __forceinline__ uint32_t warp_select_u32(uint32_t* buf, int c, int R, uint32_t* hist, int lane) {
  uint32_t prefix = 0, mask = 0;
  uint32_t need = static_cast<uint32_t>(R);
  for (int shift = 24; shift >= 0; shift -= 8) {
#pragma unroll
    for (int j = 0; j < 8; ++j) hist[lane + 32 * j] = 0;
    __syncwarp();
    for (int i = lane; i < c; i += 32) {
      uint32_t k = buf[i];
      if ((k & mask) == prefix) atomicAdd(&hist[(k >> shift) & 255u], 1u);
    }
    __syncwarp();
    uint32_t d, below;
    warp_hist_digit(hist, need, lane, d, below);
    need -= below;
    prefix |= d << shift;
    mask |= 0xFFu << shift;
    __syncwarp();
  }
  const uint32_t T = prefix;
  int write = 0;
  for (int base = 0; base < c; base += 32) {
    int i = base + lane;
    uint32_t k = i < c ? buf[i] : 0xFFFFFFFFu;
    bool keep = (i < c) && (k <= T);
    uint32_t b = __ballot_sync(0xFFFFFFFFu, keep);
    __syncwarp();
    if (keep) buf[write + __popc(b & lanemask_lt())] = k;
    write += __popc(b);
    __syncwarp();
  }
  return T;
}

#endif  // __CUDACC__

}  // namespace scann
