// Stand-alone probe for the tensor-core LUT16 scan (tcgen05.mma kind::i8 on sm_100a).  Answers, in one GPU run:
//   1. does kind::i8 (u8 x u8 -> s32) give exact sums with hand-written 128-byte-swizzled K-major smem operands (SS)?
//   2. does the A operand work from TMEM (TS), written by tcgen05.st 32x32b (lane = row, 4 K-bytes per 32-bit column)?
//   3. MMA issue rate: cycles per M=128 x N x K=32 instruction for N = 128 / 256, SS and TS.
// and, for the 2:4-sparse form tcgen05.mma.sp ... kind::i8 with the compressed A and its metadata both in TMEM:
//   4. read-out: B = identity (N = 64), so D is the decompressed A; one metadata nibble (column c, nibble b) at a time is
//      set to (2,3) and all others to (0,1), which shows which (TMEM column, nibble) drives which group of 4 K-bytes;
//   5. bit-exactness of 4 chained K = 64 sparse MMAs (dense K = 256) on random 2:4 operands and on the one-hot rows of
//      the scan's expansion (every code 0..15 in every subspace), N = 128 / 256, against a host reference;
//   6. cycles per sparse M=128 x N x K=64 instruction, back to back.
// Metadata hypothesis checked by 5: lane = row; MMA q reads columns meta + 2q (groups 0-7, 8-15 of its 64 K-bytes),
// group g in bits 4 (g % 8) .. 4 (g % 8) + 3; in a nibble bits 0-1 = index of the first kept byte, bits 2-3 = second.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o tools/tcscan_probe.bin tools/tcscan_probe.cu
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ bool mbar_try(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  for (long long it = 0; !mbar_try(bar, parity); ++it)
    if (it > 200000000LL) {
      printf("mbarrier timeout\n");
      __trap();
    }
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mma_i8_ss(uint32_t d, uint64_t ad, uint64_t bd, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}" ::"r"(d),
      "l"(ad), "l"(bd), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void mma_i8_ts(uint32_t d, uint32_t a_tmem, uint64_t bd, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d),
      "r"(a_tmem), "l"(bd), "r"(idesc), "r"(acc)
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
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
// K-major, 128-byte swizzle, 8-row groups 1024 B apart (same as the TMA SWIZZLE_128B image of a [rows][128 B] box)
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr) {
  return static_cast<uint64_t>((saddr >> 4) & 0x3FFFu) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ uint32_t swz(int row, int byte_col) {
  return static_cast<uint32_t>((row >> 3) * 1024 + (row & 7) * 128 + ((((byte_col >> 4) ^ (row & 7)) << 4) | (byte_col & 15)));
}

// A [128][128] u8, B [N][128] u8 (row-major).  D_ss / D_ts: [128][N] s32.  cyc: [0] SS loop, [1] TS loop cycles.
__global__ void __launch_bounds__(128, 1) probe_kernel(const uint8_t* __restrict__ A, const uint8_t* __restrict__ B, int N,
                                                       int32_t* __restrict__ D_ss, int32_t* __restrict__ D_ts,
                                                       long long* __restrict__ cyc, int reps) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;                 // 128 x 128 B
  uint8_t* sB = smem + 16384;         // N x 128 B
  uint64_t* bars = reinterpret_cast<uint64_t*>(sB + 256 * 128);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4);
  const int tid = threadIdx.x, warp = tid >> 5;
  if (tid == 0) {
    mbar_init(smem_u32(bars), 1);
    mbar_init(smem_u32(bars + 1), 1);
    mbar_init(smem_u32(bars + 2), 1);
    mbar_init(smem_u32(bars + 3), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  for (int i = tid; i < 128 * 128; i += 128) sA[swz(i >> 7, i & 127)] = A[i];
  for (int i = tid; i < N * 128; i += 128) sB[swz(i >> 7, i & 127)] = B[i];
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy smem writes -> async proxy (tensor core)
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const uint32_t idesc = (2u << 4) | (static_cast<uint32_t>(N >> 3) << 17) | ((128u >> 4) << 24);  // S32 acc, u8 x u8
  const uint32_t lane_base = static_cast<uint32_t>(warp * 32) << 16;

  // ---- 1. SS
  if (tid == 0) {
    const uint64_t ad = umma_desc(smem_u32(sA)), bd = umma_desc(smem_u32(sB));
    for (int k4 = 0; k4 < 4; ++k4) mma_i8_ss(tmem, ad + 2u * k4, bd + 2u * k4, idesc, k4 ? 1u : 0u);
    tc_commit(smem_u32(bars));
  }
  mbar_wait(smem_u32(bars), 0);
  tc_fence_after();
  for (int c = 0; c < N; c += 32) {
    uint32_t v[32];
    tc_ld32(tmem + lane_base + c, v);
    for (int j = 0; j < 32; ++j) D_ss[tid * N + c + j] = static_cast<int32_t>(v[j]);
  }
  tc_fence_before();
  __syncthreads();

  // ---- 2. TS: thread = row; 32 columns x 4 bytes = 128 K-bytes per row at TMEM columns [256, 288)
  {
    uint32_t a[32];
    for (int j = 0; j < 32; ++j) a[j] = reinterpret_cast<const uint32_t*>(A + tid * 128)[j];
    tc_st32(tmem + lane_base + 256, a);
  }
  tc_fence_before();
  __syncthreads();
  if (tid == 0) {
    tc_fence_after();
    const uint64_t bd = umma_desc(smem_u32(sB));
    for (int k4 = 0; k4 < 4; ++k4) mma_i8_ts(tmem, tmem + 256 + 8 * k4, bd + 2u * k4, idesc, k4 ? 1u : 0u);
    tc_commit(smem_u32(bars + 1));
  }
  mbar_wait(smem_u32(bars + 1), 0);
  tc_fence_after();
  for (int c = 0; c < N; c += 32) {
    uint32_t v[32];
    tc_ld32(tmem + lane_base + c, v);
    for (int j = 0; j < 32; ++j) D_ts[tid * N + c + j] = static_cast<int32_t>(v[j]);
  }
  tc_fence_before();
  __syncthreads();

  // ---- 3. issue-rate loops (results discarded)
  if (tid == 0) {
    tc_fence_after();
    const uint64_t ad = umma_desc(smem_u32(sA)), bd = umma_desc(smem_u32(sB));
    long long t0 = clock64();
    for (int r = 0; r < reps; ++r)
      for (int k4 = 0; k4 < 4; ++k4) mma_i8_ss(tmem, ad + 2u * k4, bd + 2u * k4, idesc, 1u);
    tc_commit(smem_u32(bars + 2));
    mbar_wait(smem_u32(bars + 2), 0);
    long long t1 = clock64();
    for (int r = 0; r < reps; ++r)
      for (int k4 = 0; k4 < 4; ++k4) mma_i8_ts(tmem, tmem + 256 + 8 * k4, bd + 2u * k4, idesc, 1u);
    tc_commit(smem_u32(bars + 3));
    mbar_wait(smem_u32(bars + 3), 0);
    long long t2 = clock64();
    cyc[0] = t1 - t0;
    cyc[1] = t2 - t1;
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------- sparse kind::i8
__device__ __forceinline__ void mma_i8_sp(uint32_t d, uint32_t a_tmem, uint64_t bd, uint32_t m_tmem, uint32_t idesc,
                                          uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %5, 0;\n\t"
      "tcgen05.mma.sp.cta_group::1.kind::i8 [%0], [%1], %2, [%3], %4, p;\n\t}" ::"r"(d),
      "r"(a_tmem), "l"(bd), "r"(m_tmem), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void tc_st8(uint32_t taddr, const uint32_t (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(v[0]),
               "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t shl_clamp(uint32_t v, uint32_t sh) {
  uint32_t r;
  asm("shl.b32 %0, %1, %2;" : "=r"(r) : "r"(v), "r"(sh));
  return r;
}
// The scan's expansion (csrc/tcscan.cu expand_sparse): one word of 8 codes -> 16 value columns + 4 metadata columns.
// Code c = 4 g + j: value byte c >> 1 of the subspace's 8 (group g, kept byte j >> 1) is 1, the others 0; every group
// of the subspace gets the nibble (0,2) when c is even and (1,3) when c is odd.
__device__ __forceinline__ void expand_sparse_ref(uint32_t C, uint32_t* v, uint32_t* mt) {
  for (int i = 0; i < 8; ++i) {
    const uint32_t c = (C >> (4 * i)) & 15u;
    v[2 * i] = shl_clamp(1u, 8u * (c >> 1));
    v[2 * i + 1] = shl_clamp(1u, 8u * (c >> 1) - 32u);
  }
  const uint32_t y = C << 7, z = C << 3;
  for (int k = 0; k < 4; ++k) {  // prmt with selector bit 3: the sign of the selected byte, replicated
    uint32_t s;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(s) : "r"(y), "r"(z), "r"(0xCC88u + 0x1111u * k));
    mt[k] = (s & 0x55555555u) | 0x88888888u;
  }
}

constexpr int kSpRuns = 64;  // read-out runs: metadata column c (0..7) x nibble b (0..7)
// TMEM map: D at columns 0..255, compressed A at 256..287 (4 MMAs x 8 columns), metadata at 320..327
// Ap: [128][32] u32 compressed A (4 MMAs x 32 bytes per row); Mp: [128][8] u32 metadata; codes: [128][2] u32 (mode 2)
// mode 0: read-out (B = identity [64][64 of 128 bytes]), D_ro [kSpRuns + 1][128][64]
// mode 1: random operands from Ap / Mp; mode 2: one-hot rows expanded on the device from codes.  Both: D [128][N].
__global__ void __launch_bounds__(128, 1) sparse_probe_kernel(int mode, const uint32_t* __restrict__ Ap,
                                                              const uint32_t* __restrict__ Mp,
                                                              const uint32_t* __restrict__ codes,
                                                              const uint8_t* __restrict__ B, int N,
                                                              int32_t* __restrict__ D, long long* __restrict__ cyc,
                                                              int reps) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sB = smem;  // 2 atoms of N x 128 B (K bytes 0..127, 128..255)
  uint64_t* bars = reinterpret_cast<uint64_t*>(sB + 2 * 256 * 128);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4);
  const int tid = threadIdx.x, warp = tid >> 5;
  if (tid == 0) {
    mbar_init(smem_u32(bars), 1);
    mbar_init(smem_u32(bars + 1), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  const int kb = mode == 0 ? 128 : 256;  // K bytes of B per row
  for (int i = tid; i < N * kb; i += 128) {
    const int n = i / kb, k = i % kb;
    sB[(k >> 7) * (N * 128) + swz(n, k & 127)] = B[i];
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const uint32_t idesc = (1u << 2) | (2u << 4) | (static_cast<uint32_t>(N >> 3) << 17) | ((128u >> 4) << 24);
  const uint32_t lane_base = static_cast<uint32_t>(warp * 32) << 16;
  const uint32_t aT = tmem + 256, mT = tmem + 320;
  const uint64_t bd = umma_desc(smem_u32(sB));
  const uint32_t atom16 = static_cast<uint32_t>(N * 128) >> 4;  // descriptor units between the two B atoms
  uint32_t phase = 0;

  {  // A operand
    uint32_t a[32];
    if (mode == 2) {
      uint32_t m8[8];
      expand_sparse_ref(codes[tid * 2], a, m8);
      expand_sparse_ref(codes[tid * 2 + 1], a + 16, m8 + 4);
      tc_st8(lane_base + mT, m8);
    } else {
      for (int j = 0; j < 32; ++j) a[j] = Ap[tid * 32 + j];
      if (mode == 1) {
        uint32_t m8[8];
        for (int j = 0; j < 8; ++j) m8[j] = Mp[tid * 8 + j];
        tc_st8(lane_base + mT, m8);
      }
    }
    tc_st32(lane_base + aT, a);
  }
  const int nruns = mode == 0 ? kSpRuns + 1 : 1;
  for (int run = 0; run < nruns; ++run) {
    if (mode == 0) {  // run r < 64: column r / 8, nibble r % 8 = (2,3); run 64: no mark
      uint32_t m8[8];
      for (int j = 0; j < 8; ++j) m8[j] = 0x44444444u;
      if (run < kSpRuns) m8[run >> 3] = (0x44444444u & ~(15u << (4 * (run & 7)))) | (0xEu << (4 * (run & 7)));
      tc_st8(lane_base + mT, m8);
    }
    tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc_fence_after();
      if (mode == 0) {
        mma_i8_sp(tmem, aT, bd, mT, idesc, 0u);
      } else {
        for (int q = 0; q < 4; ++q)
          mma_i8_sp(tmem, aT + 8 * q, bd + (q >> 1) * atom16 + (q & 1) * 4u, mT + 2 * q, idesc, q ? 1u : 0u);
      }
      tc_commit(smem_u32(bars));
    }
    mbar_wait(smem_u32(bars), phase);
    phase ^= 1u;
    tc_fence_after();
    for (int c = 0; c < N; c += 32) {
      uint32_t v[32];
      tc_ld32(tmem + lane_base + c, v);
      for (int j = 0; j < 32; ++j) D[(static_cast<size_t>(run) * 128 + tid) * N + c + j] = static_cast<int32_t>(v[j]);
    }
    tc_fence_before();
    __syncthreads();
  }
  if (mode != 0 && tid == 0) {  // issue rate, results discarded
    tc_fence_after();
    long long t0 = clock64();
    for (int r = 0; r < reps; ++r)
      for (int q = 0; q < 4; ++q)
        mma_i8_sp(tmem, aT + 8 * q, bd + (q >> 1) * atom16 + (q & 1) * 4u, mT + 2 * q, idesc, 1u);
    tc_commit(smem_u32(bars + 1));
    mbar_wait(smem_u32(bars + 1), 0);
    cyc[0] = clock64() - t0;
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512) : "memory");
  }
}

#define CK(x)                                                                      \
  do {                                                                             \
    cudaError_t e = (x);                                                           \
    if (e != cudaSuccess) {                                                        \
      printf("CUDA error %s at line %d: %s\n", #x, __LINE__, cudaGetErrorString(e)); \
      return 1;                                                                    \
    }                                                                              \
  } while (0)

static int sparse_main(int reps) {
  const int smem = 1024 + 2 * 256 * 128 + 64;
  CK(cudaFuncSetAttribute(sparse_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  uint32_t *dA, *dM, *dCodes;
  uint8_t* dB;
  int32_t* dD;
  long long* dC;
  CK(cudaMalloc(&dA, 128 * 32 * 4));
  CK(cudaMalloc(&dM, 128 * 8 * 4));
  CK(cudaMalloc(&dCodes, 128 * 2 * 4));
  CK(cudaMalloc(&dB, 256 * 256));
  CK(cudaMalloc(&dD, static_cast<size_t>(kSpRuns + 1) * 128 * 256 * 4));
  CK(cudaMalloc(&dC, 16));

  // ---- 4. read-out: compressed byte k' of every row = k' + 1, B = identity
  {
    std::vector<uint8_t> Ab(128 * 128, 0), B(64 * 128, 0);
    for (int m = 0; m < 128; ++m)
      for (int k = 0; k < 32; ++k) Ab[m * 128 + k] = static_cast<uint8_t>(k + 1);
    for (int n = 0; n < 64; ++n) B[n * 128 + n] = 1;
    CK(cudaMemcpy(dA, Ab.data(), Ab.size(), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dB, B.data(), B.size(), cudaMemcpyHostToDevice));
    sparse_probe_kernel<<<1, 128, smem>>>(0, dA, dM, dCodes, dB, 64, dD, dC, 0);
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    std::vector<int32_t> D(static_cast<size_t>(kSpRuns + 1) * 128 * 64);
    CK(cudaMemcpy(D.data(), dD, D.size() * 4, cudaMemcpyDeviceToHost));
    // group g of a row: 'n' = (2g+1, 2g+2, 0, 0) [nibble (0,1)], 'M' = (0, 0, 2g+1, 2g+2) [nibble (2,3)], '?' other
    auto classify = [&](int run, int m) {
      std::string s;
      const int32_t* r = D.data() + (static_cast<size_t>(run) * 128 + m) * 64;
      for (int g = 0; g < 16; ++g) {
        const int32_t a = 2 * g + 1, b = 2 * g + 2;
        const int32_t* x = r + 4 * g;
        s += (x[0] == a && x[1] == b && !x[2] && !x[3]) ? 'n' : (!x[0] && !x[1] && x[2] == a && x[3] == b) ? 'M' : '?';
      }
      return s;
    };
    printf("sparse read-out, no mark: row 0 groups %s, D[0][0..63] =", classify(kSpRuns, 0).c_str());
    for (int k = 0; k < 64; ++k) printf(" %d", D[static_cast<size_t>(kSpRuns) * 128 * 64 + k]);
    int agree = 0;
    for (int m = 0; m < 128; ++m) agree += classify(kSpRuns, m) == std::string(16, 'n');
    printf("\n  rows with every group (0,1): %d / 128\n", agree);
    for (int run = 0; run < kSpRuns; ++run) {
      const std::string r0 = classify(run, 0);
      int same = 0;
      for (int m = 1; m < 128; ++m) same += classify(run, m) == r0;
      printf("  mark column %d nibble %d: row 0 groups %s (rows 1..127 equal to row 0: %d)\n", run >> 3, run & 7,
             r0.c_str(), same);
    }
  }

  // ---- 5 / 6. chained sparse MMAs: random 2:4 operands (mode 1), the scan's one-hot rows (mode 2)
  const uint8_t valid_nib[6] = {0x4, 0x8, 0xC, 0x9, 0xD, 0xE};
  for (int mode = 1; mode <= 2; ++mode)
    for (int N : {128, 256}) {
      srand(777 + 10 * mode + N);
      std::vector<uint8_t> Ab(128 * 128, 0), B(N * 256);
      std::vector<uint32_t> Mw(128 * 8, 0), codes(128 * 2, 0);
      std::vector<int> dense(128 * 256, 0);
      for (auto& v : B) v = rand() & 255;
      for (int m = 0; m < 128; ++m) {
        if (mode == 1) {
          for (int q = 0; q < 4; ++q)
            for (int g = 0; g < 16; ++g) {
              const uint32_t nib = valid_nib[rand() % 6];
              Mw[m * 8 + 2 * q + g / 8] |= nib << (4 * (g % 8));
              const uint8_t v0 = rand() & 255, v1 = rand() & 255;
              Ab[m * 128 + 32 * q + 2 * g] = v0;
              Ab[m * 128 + 32 * q + 2 * g + 1] = v1;
              dense[m * 256 + 64 * q + 4 * g + (nib & 3)] = v0;
              dense[m * 256 + 64 * q + 4 * g + (nib >> 2)] = v1;
            }
        } else {
          for (int s = 0; s < 16; ++s) {
            const uint32_t c = (m + 5 * s) & 15u;  // every code in every subspace over the 128 rows
            codes[m * 2 + s / 8] |= c << (4 * (s % 8));
            dense[m * 256 + 16 * s + c] = 1;
          }
        }
      }
      CK(cudaMemcpy(dA, Ab.data(), Ab.size(), cudaMemcpyHostToDevice));
      CK(cudaMemcpy(dM, Mw.data(), Mw.size() * 4, cudaMemcpyHostToDevice));
      CK(cudaMemcpy(dCodes, codes.data(), codes.size() * 4, cudaMemcpyHostToDevice));
      CK(cudaMemcpy(dB, B.data(), B.size(), cudaMemcpyHostToDevice));
      CK(cudaMemset(dD, 0xFF, 128 * N * 4));
      sparse_probe_kernel<<<1, 128, smem>>>(mode, dA, dM, dCodes, dB, N, dD, dC, reps);
      CK(cudaGetLastError());
      CK(cudaDeviceSynchronize());
      std::vector<int32_t> D(128 * N);
      long long cyc = 0;
      CK(cudaMemcpy(D.data(), dD, D.size() * 4, cudaMemcpyDeviceToHost));
      CK(cudaMemcpy(&cyc, dC, 8, cudaMemcpyDeviceToHost));
      long bad = 0;
      int first = -1;
      for (int m = 0; m < 128; ++m)
        for (int n = 0; n < N; ++n) {
          int32_t ref = 0;
          for (int k = 0; k < 256; ++k) ref += dense[m * 256 + k] * int(B[n * 256 + k]);
          if (D[m * N + n] != ref) {
            ++bad;
            if (first < 0) {
              first = m * N + n;
              printf("  first mismatch m=%d n=%d: got %d, want %d\n", m, n, D[m * N + n], ref);
            }
          }
        }
      printf("sparse %s, N=%d, 4 x (M=128,K=64) chained: mismatches %ld / %d; %d x 4 back-to-back: %.1f cycles/MMA\n",
             mode == 1 ? "random 2:4" : "one-hot (all 16 codes)", N, bad, 128 * N, reps, double(cyc) / (reps * 4));
    }
  cudaFree(dA);
  cudaFree(dM);
  cudaFree(dCodes);
  cudaFree(dB);
  cudaFree(dD);
  cudaFree(dC);
  return 0;
}

int main() {
  const int reps = 2000;
  for (int N : {128, 256}) {
    std::vector<uint8_t> A(128 * 128), B(N * 128);
    srand(1234 + N);
    for (auto& v : A) v = rand() & 255;
    for (auto& v : B) v = rand() & 255;
    uint8_t *dA, *dB;
    int32_t *dS, *dT;
    long long* dC;
    CK(cudaMalloc(&dA, A.size()));
    CK(cudaMalloc(&dB, B.size()));
    CK(cudaMalloc(&dS, 128 * N * 4));
    CK(cudaMalloc(&dT, 128 * N * 4));
    CK(cudaMalloc(&dC, 16));
    CK(cudaMemcpy(dA, A.data(), A.size(), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dB, B.data(), B.size(), cudaMemcpyHostToDevice));
    CK(cudaMemset(dS, 0xFF, 128 * N * 4));
    CK(cudaMemset(dT, 0xFF, 128 * N * 4));
    const int smem = 1024 + 16384 + 256 * 128 + 64;
    CK(cudaFuncSetAttribute(probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    probe_kernel<<<1, 128, smem>>>(dA, dB, N, dS, dT, dC, reps);
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    std::vector<int32_t> S(128 * N), T(128 * N);
    long long cyc[2];
    CK(cudaMemcpy(S.data(), dS, S.size() * 4, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(T.data(), dT, T.size() * 4, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(cyc, dC, 16, cudaMemcpyDeviceToHost));
    long bad_s = 0, bad_t = 0, bad_t_swapped = 0;
    for (int m = 0; m < 128; ++m)
      for (int n = 0; n < N; ++n) {
        int32_t ref = 0, ref_sw = 0;
        for (int k = 0; k < 128; ++k) {
          ref += int(A[m * 128 + k]) * int(B[n * 128 + k]);
          ref_sw += int(A[m * 128 + (k ^ 3)]) * int(B[n * 128 + k]);  // A bytes big-endian inside a TMEM column?
        }
        bad_s += S[m * N + n] != ref;
        bad_t += T[m * N + n] != ref;
        bad_t_swapped += T[m * N + n] != ref_sw;
      }
    printf("N=%d: SS mismatches %ld / %d, TS mismatches %ld (byte-swapped hypothesis: %ld); D_ss[0..3] = %d %d %d %d, D_ts[0..3] = %d %d %d %d\n",
           N, bad_s, 128 * N, bad_t, bad_t_swapped, S[0], S[1], S[2], S[3], T[0], T[1], T[2], T[3]);
    printf("N=%d: %d x 4 MMAs (M=128,N=%d,K=32 u8): SS %.1f cycles/MMA, TS %.1f cycles/MMA\n", N, reps, N,
           double(cyc[0]) / (reps * 4), double(cyc[1]) / (reps * 4));
    cudaFree(dA);
    cudaFree(dB);
    cudaFree(dS);
    cudaFree(dT);
    cudaFree(dC);
  }
  return sparse_main(reps);
}
