// Host runtime pieces shared by every entry point: thread-local error text, CUDA error mapping,
// device checks, the grow-only workspace arena.
#include <stdarg.h>
#include <string.h>

#include "common.cuh"

namespace scann {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

scann_status cuda_fail(cudaError_t e, const char* what, const char* file, int line) {
  set_error("CUDA error %d (%s) at %s:%d: %s", static_cast<int>(e), cudaGetErrorString(e), file, line, what);
  switch (e) {
    case cudaErrorMemoryAllocation: return SCANN_RESOURCE_EXHAUSTED;
    case cudaErrorNoDevice:
    case cudaErrorInsufficientDriver:
    case cudaErrorInvalidDevice: return SCANN_UNAVAILABLE;
    default: return SCANN_INTERNAL;
  }
}

scann_status check_device(int device) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    cudaGetLastError();
    set_error("no CUDA device available (%s); libscann_b200 has no CPU fallback",
              e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    return SCANN_UNAVAILABLE;
  }
  if (device < 0 || device >= n) {
    set_error("device %d out of range (have %d)", device, n);
    return SCANN_INVALID_ARGUMENT;
  }
  return SCANN_OK;
}

int sm_count(int device) {
  int v = 0;
  if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || v <= 0) v = 148;
  return v;
}

scann_status Workspace::reserve(size_t bytes) {
  used = 0;
  overflow = false;
  if (bytes <= cap) return SCANN_OK;
  if (base) cudaFree(base);
  base = nullptr;
  cap = 0;
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&base), bytes);
  if (e != cudaSuccess) {
    base = nullptr;
    return cuda_fail(e, "workspace cudaMalloc", __FILE__, __LINE__);
  }
  cap = bytes;
  return SCANN_OK;
}

scann_status Workspace::check(const char* carve) const {
  SCANN_REQUIRE(!overflow, SCANN_INTERNAL, "workspace: the %s carve exceeds its reservation of %zu bytes", carve, cap);
  return SCANN_OK;
}

void Workspace::release() {
  if (base) cudaFree(base);
  base = nullptr;
  cap = used = 0;
}

}  // namespace scann

extern "C" {

const char* scann_last_error(void) { return scann::g_err; }

int scann_version(void) { return 100; }

scann_status scann_device_count(int* count) {
  if (!count) return SCANN_INVALID_ARGUMENT;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) {
    cudaGetLastError();
    *count = 0;
    scann::set_error("cudaGetDeviceCount: %s", cudaGetErrorString(e));
    return SCANN_UNAVAILABLE;
  }
  *count = n;
  return SCANN_OK;
}

}  // extern "C"
