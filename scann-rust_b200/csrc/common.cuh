// Shared host/device helpers of libscann_b200.so (sm_100a only; compiled with -fmad=false so that
// plain a*b+c never contracts — FMA appears only where fmaf() is written, mirroring the places the
// reference calls _mm256_fmadd_ps; SURVEY.md F8).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <mutex>
#include <vector>

#include "../../include/scann_b200.h"

namespace scann {

// ------------------------------------------------------------------------------------------ host
void set_error(const char* fmt, ...);
scann_status cuda_fail(cudaError_t e, const char* what, const char* file, int line);

#define SCANN_CUDA(expr)                                                  \
  do {                                                                    \
    cudaError_t _e = (expr);                                              \
    if (_e != cudaSuccess) return ::scann::cuda_fail(_e, #expr, __FILE__, __LINE__); \
  } while (0)

#define SCANN_TRY(expr)                 \
  do {                                  \
    scann_status _s = (expr);           \
    if (_s != SCANN_OK) return _s;      \
  } while (0)

#define SCANN_REQUIRE(cond, code, ...)  \
  do {                                  \
    if (!(cond)) {                      \
      ::scann::set_error(__VA_ARGS__);  \
      return (code);                    \
    }                                   \
  } while (0)

struct DeviceGuard {
  int prev = -1;
  bool ok = false;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) == cudaSuccess && cudaSetDevice(dev) == cudaSuccess) ok = true;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

scann_status check_device(int device);

// Orders the device work of successive calls on one handle ACROSS STREAMS.  A handle's workspace is shared by its calls
// and a SCANN_DEVICE call returns with its kernels only enqueued, so the next call — possibly on another stream — must
// not start before they have finished: every call waits on the event the previous one recorded.
struct StreamOrder {
  cudaEvent_t done = nullptr;
  void enter(cudaStream_t s) {
    if (done) cudaStreamWaitEvent(s, done, 0);
  }
  void leave(cudaStream_t s) {
    if (!done && cudaEventCreateWithFlags(&done, cudaEventDisableTiming) != cudaSuccess) done = nullptr;
    if (done) cudaEventRecord(done, s);
  }
  ~StreamOrder() {
    if (done) cudaEventDestroy(done);
  }
};

// The device, stream and stream order of one call on a handle; the caller holds the handle's lock.  A SCANN_DEVICE call
// runs on the caller's stream; a SCANN_HOST call on the caller's stream when one is given, else on the handle's own
// (scann_b200.h).
struct CallScope {
  DeviceGuard g;
  cudaStream_t s;
  StreamOrder& order;
  CallScope(int device, StreamOrder& o, int memspace, void* user_stream, cudaStream_t own)
      : g(device), s(memspace == SCANN_DEVICE || user_stream ? static_cast<cudaStream_t>(user_stream) : own), order(o) {
    order.enter(s);
  }
  ~CallScope() { order.leave(s); }
};

// Grow-only device arena; one per handle, guarded by the handle's mutex.  A list of buffers is one carve (a function
// that only calls take), run by count() in counting mode (take returns nullptr) to size the reservation, then for real:
// a take past the reservation returns nullptr, and check() after the carve reports it before any kernel runs.
struct Workspace {
  char* base = nullptr;
  size_t cap = 0;
  size_t used = 0;
  bool counting = false;
  bool overflow = false;
  Workspace() = default;
  Workspace(const Workspace&) = delete;
  Workspace& operator=(const Workspace&) = delete;
  ~Workspace() { release(); }
  scann_status reserve(size_t bytes);
  // bytes carve(Workspace&) takes
  template <class Carve>
  static size_t count(Carve carve) {
    Workspace w;
    w.counting = true;
    carve(w);
    return w.used;
  }
  template <class T>
  T* take(size_t count) {
    const size_t bytes = (count * sizeof(T) + 255) & ~size_t(255);
    if (!counting && bytes > cap - used) {
      overflow = true;
      return nullptr;
    }
    T* p = counting ? nullptr : reinterpret_cast<T*>(base + used);
    used += bytes;
    return p;
  }
  scann_status check(const char* carve) const;
  void release();
};

// device buffer owned by a handle
template <class T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  DevBuf(DevBuf&& o) noexcept : p(o.p), n(o.n) {
    o.p = nullptr;
    o.n = 0;
  }
  DevBuf& operator=(DevBuf&& o) noexcept {
    if (this != &o) {
      free_();
      p = o.p;
      n = o.n;
      o.p = nullptr;
      o.n = 0;
    }
    return *this;
  }
  scann_status alloc(size_t count) {
    free_();
    n = count;
    if (count == 0) return SCANN_OK;
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&p), count * sizeof(T));
    if (e != cudaSuccess) {
      p = nullptr;
      return cuda_fail(e, "cudaMalloc", __FILE__, __LINE__);
    }
    return SCANN_OK;
  }
  scann_status upload(const T* src, size_t count, int memspace, cudaStream_t s) {
    SCANN_TRY(alloc(count));
    if (count == 0) return SCANN_OK;
    SCANN_CUDA(cudaMemcpyAsync(p, src, count * sizeof(T),
                               memspace == SCANN_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, s));
    return SCANN_OK;
  }
  void free_() {
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
  }
  ~DevBuf() { free_(); }
};

inline cudaMemcpyKind in_kind(int memspace) {
  return memspace == SCANN_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
}
inline cudaMemcpyKind out_kind(int memspace) {
  return memspace == SCANN_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
}

// One output of a query-batched call: the caller's array, `bytes` per query; p == NULL: optional and not requested.
struct QueryOut {
  void* p;
  size_t bytes;
};

// The staging carve of run_query_chunks: on SCANN_HOST the chunk's queries and every requested output.
template <size_t N>
struct Staging {
  float* q = nullptr;
  void* out[N] = {};
};
template <size_t N>
Staging<N> take_staging(Workspace& ws, int memspace, size_t chunk, size_t dim, const QueryOut (&outs)[N]) {
  Staging<N> st;
  if (memspace != SCANN_HOST) return st;
  st.q = ws.take<float>(chunk * dim);
  for (size_t i = 0; i < N; ++i)
    if (outs[i].p) st.out[i] = ws.take<uint8_t>(chunk * outs[i].bytes);
  return st;
}

// Runs a batch of nq queries [nq][dim] in chunks of at most `chunk` queries as
//   run(const float* device_queries, size_t q0, size_t nqc, void* const* device_outs)  -> scann_status
// where device_outs[i] is outs[i] of the chunk (NULL when not requested).  SCANN_DEVICE: the caller's arrays at q0;
// nothing is copied or synchronised.  SCANN_HOST: staging buffers taken from `ws` once (the reservation counts
// take_staging); per chunk one copy of the queries in, one copy of every requested output out, one stream
// synchronisation.  The workspace is reset to the mark above the staging before every chunk: run takes its scratch
// from there.
template <size_t N, class Run>
scann_status run_query_chunks(Workspace& ws, int memspace, cudaStream_t s, const float* queries, size_t nq, size_t dim,
                              size_t chunk, const QueryOut (&outs)[N], Run run) {
  const bool host = memspace == SCANN_HOST;
  const Staging<N> st = take_staging(ws, memspace, chunk, dim, outs);
  SCANN_TRY(ws.check("query staging"));
  const size_t mark = ws.used;
  for (size_t q0 = 0; q0 < nq; q0 += chunk) {
    const size_t nqc = nq - q0 < chunk ? nq - q0 : chunk;
    ws.used = mark;
    if (!host) {
      void* dout[N];
      for (size_t i = 0; i < N; ++i) dout[i] = outs[i].p ? static_cast<char*>(outs[i].p) + q0 * outs[i].bytes : nullptr;
      SCANN_TRY(run(queries + q0 * dim, q0, nqc, dout));
      continue;
    }
    SCANN_CUDA(cudaMemcpyAsync(st.q, queries + q0 * dim, nqc * dim * sizeof(float), cudaMemcpyHostToDevice, s));
    SCANN_TRY(run(static_cast<const float*>(st.q), q0, nqc, st.out));
    for (size_t i = 0; i < N; ++i)
      if (outs[i].p)
        SCANN_CUDA(cudaMemcpyAsync(static_cast<char*>(outs[i].p) + q0 * outs[i].bytes, st.out[i], nqc * outs[i].bytes,
                                   cudaMemcpyDeviceToHost, s));
    SCANN_CUDA(cudaStreamSynchronize(s));
  }
  return SCANN_OK;
}

int sm_count(int device);

// shared kernels / launchers implemented in select.cu, used by several translation units
// Exact distance re-score + final order: see select.cu.
struct RescoreParams {
  const float* queries;    // [nq][dim]
  size_t dim;
  const float* raw;        // f32 rows (or nullptr)
  const int8_t* raw_i8;    // i8 rows (or nullptr); distance = q·((i8)x*scale) as the reference's AVX2 kernel
  float scale;
  size_t stride;           // row stride in elements
  int measure;
};

// ---------------------------------------------------------------------------------------- device
#ifdef __CUDACC__

__device__ __forceinline__ uint32_t f32_key(float f) {
  // monotone f32 -> u32 (partial_cmp order; -0.0 == +0.0; NaN sorts last = OrderedFloat "greatest")
  uint32_t u = __float_as_uint(f);
  if (u == 0x80000000u) u = 0;
  if ((u & 0x7F800000u) == 0x7F800000u && (u & 0x007FFFFFu)) return 0xFFFFFFFFu;  // NaN
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key_f32(uint32_t k) {
  uint32_t u = (k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k;
  return __uint_as_float(u);
}

__device__ __forceinline__ uint32_t lanemask_lt() {
  uint32_t m;
  asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
  return m;
}

// Exact single-pair distance in the reference's AVX2+FMA order, computed by a group of 8 adjacent
// lanes (sub = lane & 7 plays AVX lane `sub`).  All 8 lanes return the same value.
//   f32 rows : src/simd/x86.rs:72-96 (dot), :139-165 (sqL2), hsum :31-44
//   i8 rows  : src/distance_measures/one_to_many_asymmetric.rs:77-144, :207-261, hsum :383-399
// Both hsums reduce as ((a0+a4)+(a1+a5)) + ((a2+a6)+(a3+a7)); f32 add is commutative so xor-shuffles
// give every lane the identical bit pattern.
template <bool I8>
__device__ __forceinline__ float exact_pair_distance(const float* __restrict__ q, const void* __restrict__ row,
                                                     int dim, int measure, float scale, int sub) {
  const float* xf = reinterpret_cast<const float*>(row);
  const int8_t* xi = reinterpret_cast<const int8_t*>(row);
  int chunks = dim >> 3;
  float acc = 0.0f;
  for (int i = 0; i < chunks; ++i) {
    float a = q[i * 8 + sub];
    float b = I8 ? __fmul_rn(static_cast<float>(xi[i * 8 + sub]), scale) : xf[i * 8 + sub];
    if (measure == SCANN_DOT) {
      acc = fmaf(a, b, acc);
    } else {
      float d = __fsub_rn(a, b);
      acc = fmaf(d, d, acc);
    }
  }
  float t = __fadd_rn(acc, __shfl_xor_sync(0xFFFFFFFFu, acc, 4));
  float u = __fadd_rn(t, __shfl_xor_sync(0xFFFFFFFFu, t, 1));
  float r = __fadd_rn(u, __shfl_xor_sync(0xFFFFFFFFu, u, 2));
  for (int j = chunks * 8; j < dim; ++j) {  // scalar tail: mul then add, never fused
    float a = q[j];
    float b = I8 ? __fmul_rn(static_cast<float>(xi[j]), scale) : xf[j];
    if (measure == SCANN_DOT) {
      r = __fadd_rn(r, __fmul_rn(a, b));
    } else {
      float d = __fsub_rn(a, b);
      r = __fadd_rn(r, __fmul_rn(d, d));
    }
  }
  if (measure == SCANN_DOT) return -r;
  if (measure == SCANN_L2) return __fsqrt_rn(r);
  return r;
}

// ---- certified error bound of the bf16 tensor-core ranking score (tc_gemm.cu) ------------------------------------------
// |q~.x~ - q.x| with both operands rounded to bf16 (RN, 8 significant bits: unit roundoff u = 2^-8) is bounded by
// (2u + u^2) sum|q_j x_j| <= (2^-7 + 2^-16) |q||x| < 0.0079 |q||x|; when the rows are int8 they are exact in bf16 and
// only the query rounds: u |q||x| < 0.0040 |q||x|.  The second term covers the f32 accumulation of the tensor core, of
// hx and of the reference's own sum (all <= ~dim * 2^-23 relative).
__device__ __forceinline__ float tc_rank_eps(float nqr, float nx, bool rows_exact_in_bf16) {
  const float c = rows_exact_in_bf16 ? 0.0040f : 0.0079f;
  return c * nqr * nx + 1.6e-5f * (nqr + nx) * (nqr + nx);
}

// ---- block-level exact selection of the R smallest distinct u64 keys ---------------------------
// hist: 264 u32 of shared memory ([0..255] bins, [256] digit, [257] below, [258] counter)
template <int NT>
__device__ uint64_t block_radix_threshold(const uint64_t* buf, int c, int R, uint32_t* hist) {
  // returns the R-th smallest key (1 <= R <= c); all threads get the same value
  const int tid = threadIdx.x;
  uint64_t prefix = 0, mask = 0;
  int need = R;
  for (int shift = 56; shift >= 0; shift -= 8) {
    for (int i = tid; i < 256; i += NT) hist[i] = 0;
    __syncthreads();
    for (int i = tid; i < c; i += NT) {
      uint64_t k = buf[i];
      if ((k & mask) == prefix) atomicAdd(&hist[(k >> shift) & 255], 1u);
    }
    __syncthreads();
    if (tid < 32) {
      uint32_t h[8];
      uint32_t s = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        h[j] = hist[tid * 8 + j];
        s += h[j];
      }
      uint32_t incl = s;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (tid >= o) incl += v;
      }
      uint32_t excl = incl - s;
      if (excl < static_cast<uint32_t>(need) && static_cast<uint32_t>(need) <= incl) {
        uint32_t run = excl;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          if (run + h[j] >= static_cast<uint32_t>(need)) {
            hist[256] = tid * 8 + j;
            hist[257] = run;
            break;
          }
          run += h[j];
        }
      }
    }
    __syncthreads();
    uint32_t d = hist[256];
    need -= static_cast<int>(hist[257]);
    prefix |= static_cast<uint64_t>(d) << shift;
    mask |= 0xFFull << shift;
    __syncthreads();
  }
  return prefix;
}

template <int NT>
__device__ void block_bitonic_sort(uint64_t* s, int p2) {
  const int tid = threadIdx.x;
  for (int k = 2; k <= p2; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = tid; i < p2; i += NT) {
        int ixj = i ^ j;
        if (ixj > i) {
          bool asc = ((i & k) == 0);
          uint64_t a = s[i], b = s[ixj];
          if ((a > b) == asc) {
            s[i] = b;
            s[ixj] = a;
          }
        }
      }
      __syncthreads();
    }
  }
}

__host__ __device__ inline int next_pow2(int v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}

// Streaming top-R: gen(i) yields distinct u64 keys for i in [0, n).  On return out[0..m) holds the
// m = min(n, R) smallest keys in ascending order and out[m..p2) = ~0.  Shared memory needed:
// buf[R + CHUNK] u64, out[next_pow2(R)] u64, hist[264] u32.  All NT threads must call.
// thr_init: keys >= thr_init are dropped up front (pass ~0ull for "no bound").
template <int NT, int CHUNK, class Gen>
__device__ int block_topr_sorted(Gen gen, int n, int R, uint64_t* buf, uint64_t* out, uint32_t* hist,
                                 uint64_t thr_init = ~0ull) {
  const int tid = threadIdx.x;
  const int p2 = next_pow2(R < 1 ? 1 : R);
  if (tid == 0) hist[258] = 0;
  __syncthreads();
  uint64_t thr = thr_init;
  for (int base = 0; base < n; base += CHUNK) {
    int end = base + CHUNK < n ? base + CHUNK : n;
    for (int i = base + tid; i < end; i += NT) {
      uint64_t k = gen(i);
      if (k < thr) {
        uint32_t slot = atomicAdd(&hist[258], 1u);
        buf[slot] = k;
      }
    }
    __syncthreads();
    int c = static_cast<int>(hist[258]);
    __syncthreads();  // every thread has read c before the next chunk's appends can change hist[258]: c is block-uniform
    if (c > R && R > 0) {
      uint64_t T = block_radix_threshold<NT>(buf, c, R, hist);
      if (tid == 0) hist[258] = 0;
      __syncthreads();
      for (int i = tid; i < c; i += NT) {
        uint64_t k = buf[i];
        if (k <= T) out[atomicAdd(&hist[258], 1u)] = k;
      }
      __syncthreads();
      for (int i = tid; i < R; i += NT) buf[i] = out[i];
      thr = T;
      __syncthreads();
    }
  }
  int m = static_cast<int>(hist[258]);
  if (R <= 0) m = 0;
  for (int i = tid; i < p2; i += NT) out[i] = i < m ? buf[i] : ~0ull;
  __syncthreads();
  block_bitonic_sort<NT>(out, p2);
  return m;
}


// Grouped variant of block_topr_sorted: LANES adjacent lanes (a power of two <= 32) cooperate on one candidate.
// gen(i, sub) is called by all lanes of a group with the same i (and by every lane of the warp at the same time, so
// it may shuffle); the key it returns on sub == 0 is the one that is kept.  Same shared-memory needs and result.
template <int NT, int CHUNK, int LANES, class Gen>
__device__ int block_topr_sorted_grouped(Gen gen, int n, int R, uint64_t* buf, uint64_t* out, uint32_t* hist,
                                         uint64_t thr_init = ~0ull) {
  const int tid = threadIdx.x;
  const int p2 = next_pow2(R < 1 ? 1 : R);
  const int grp = tid / LANES, sub = tid % LANES;
  if (tid == 0) hist[258] = 0;
  __syncthreads();
  uint64_t thr = thr_init;
  for (int base = 0; base < n; base += CHUNK) {
    const int end = base + CHUNK < n ? base + CHUNK : n;
    for (int i0 = base; i0 < end; i0 += NT / LANES) {
      const int i = i0 + grp;
      const bool valid = i < end;
      const uint64_t k = gen(valid ? i : end - 1, sub);
      if (valid && sub == 0 && k < thr) {
        uint32_t slot = atomicAdd(&hist[258], 1u);
        buf[slot] = k;
      }
    }
    __syncthreads();
    int c = static_cast<int>(hist[258]);
    __syncthreads();  // every thread has read c before the next chunk's appends can change hist[258]: c is block-uniform
    if (c > R && R > 0) {
      uint64_t T = block_radix_threshold<NT>(buf, c, R, hist);
      if (tid == 0) hist[258] = 0;
      __syncthreads();
      for (int i = tid; i < c; i += NT) {
        uint64_t k = buf[i];
        if (k <= T) out[atomicAdd(&hist[258], 1u)] = k;
      }
      __syncthreads();
      for (int i = tid; i < R; i += NT) buf[i] = out[i];
      thr = T;
      __syncthreads();
    }
  }
  int m = static_cast<int>(hist[258]);
  if (R <= 0) m = 0;
  for (int i = tid; i < p2; i += NT) out[i] = i < m ? buf[i] : ~0ull;
  __syncthreads();
  block_bitonic_sort<NT>(out, p2);
  return m;
}

// ---- warp-level upper bound of the need-th smallest of row[0..n) ----------------------------------------------------
// One 256-bucket linear histogram over [min, max of the finite entries]: the bucket that holds the need-th smallest
// value ends at the returned edge (>= that value; the slack covers the rounding of the bucket arithmetic).  Entries
// that are NaN or +inf land in the last bucket; the result is +inf when the need-th smallest lies there.  Three passes
// over the row (L1/L2 resident), one of them with shared-memory atomics.  hist: 256 u32 private to the warp.
template <class Get>  // get(i) = the i-th value, i in [0, n)
__device__ __forceinline__ float warp_kth_upper_bound_of(Get get, int n, uint32_t need, uint32_t* hist, int lane) {
  const float inf = __int_as_float(0x7F800000);
  float mn = inf, mx = -inf;
  for (int i = lane; i < n; i += 32) {
    const float v = get(i);
    mn = fminf(mn, v);
    if (v < inf) mx = fmaxf(mx, v);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mn = fminf(mn, __shfl_xor_sync(0xFFFFFFFFu, mn, o));
    mx = fmaxf(mx, __shfl_xor_sync(0xFFFFFFFFu, mx, o));
  }
  if (!(mx >= mn)) return inf;  // no finite entry
  const float width = (mx - mn) * (1.0f / 255.0f);  // finite entries use buckets 0..254 (max lands on 255: clamped)
  const float scale = width > 0.0f ? 1.0f / width : 0.0f;
#pragma unroll
  for (int j = 0; j < 8; ++j) hist[lane + 32 * j] = 0;
  __syncwarp();
  for (int i = lane; i < n; i += 32) {
    const float v = get(i);
    int b = 255;
    if (v < inf) b = min(254, max(0, static_cast<int>((v - mn) * scale)));
    atomicAdd(&hist[b], 1u);
  }
  __syncwarp();
  uint32_t h[8], s = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    h[j] = hist[lane * 8 + j];
    s += h[j];
  }
  uint32_t incl = s;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
    if (lane >= o) incl += v;
  }
  const uint32_t excl = incl - s;
  const bool mine = (excl < need) && (need <= incl);
  int dg = 255;
  if (mine) {
    uint32_t run = excl;
    bool found = false;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (!found && run + h[j] >= need) {
        dg = lane * 8 + j;
        found = true;
      }
      if (!found) run += h[j];
    }
  }
  const uint32_t bal = __ballot_sync(0xFFFFFFFFu, mine);
  int bL = 255;
  if (bal) bL = __shfl_sync(0xFFFFFFFFu, dg, __ffs(bal) - 1);
  __syncwarp();
  if (bL >= 255) return inf;
  return mn + static_cast<float>(bL + 1) * width * 1.00001f + (fabsf(mn) + fabsf(mx)) * 1e-6f;
}
__device__ __forceinline__ float warp_kth_upper_bound(const float* __restrict__ row, int n, uint32_t need,
                                                      uint32_t* hist, int lane) {
  return warp_kth_upper_bound_of([&](int i) { return row[i]; }, n, need, hist, lane);
}

#endif  // __CUDACC__

}  // namespace scann
