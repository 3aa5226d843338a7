// libdnmf core: status, device info, split planning, workspace sizing.
#include <stdarg.h>

#include "common.cuh"
#include "tc_api.cuh"

namespace dnmf {

TlsState& tls() {
  static thread_local TlsState s = {{0}, 0, 0, 0, 0, 0};
  return s;
}

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(tls().msg, sizeof(tls().msg), fmt, ap);
  va_end(ap);
  return code;
}

int cuda_fail(cudaError_t e, const char* where) {
  snprintf(tls().msg, sizeof(tls().msg), "%s: CUDA error %d (%s)", where, (int)e, cudaGetErrorString(e));
  cudaGetLastError();  // clear the sticky-less error state
  return (int)e;
}

int sm_count() {
  static int cached = 0;
  if (cached) return cached;
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) == cudaSuccess &&
      cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0) {
    cached = n;
  } else {
    cudaGetLastError();
    cached = 148;  // B200; keeps workspace queries usable on a host without a GPU
  }
  return cached;
}

Split plan_split(int64_t outer, int64_t outer_tile, int64_t reduce_len, int64_t align, int64_t min_chunk) {
  Split s;
  s.blocks = ceil_div(outer > 0 ? outer : 1, outer_tile);
  int64_t target = (int64_t)sm_count() * 8;
  int64_t want = ceil_div(target, s.blocks);
  if (want < 1) want = 1;
  if (want > 64) want = 64;
  int64_t chunk = round_up(ceil_div(reduce_len > 0 ? reduce_len : 1, want), align);
  if (chunk < min_chunk) chunk = min_chunk;
  s.chunk = chunk;
  s.splits = ceil_div(reduce_len > 0 ? reduce_len : 1, chunk);
  return s;
}

}  // namespace dnmf

using namespace dnmf;

extern "C" {

const char* dnmf_version(void) { return "libdnmf 0.1 (sm_100a)"; }

const char* dnmf_last_error(void) { return tls().msg; }

int dnmf_last_path(void) { return tls().last_path; }

int64_t dnmf_launch_count(int reset) {
  int64_t v = tls().launches;
  if (reset) tls().launches = 0;
  return v;
}

int64_t dnmf_pass_count(int which, int reset) {
  int64_t& c = which ? tls().tc_passes : tls().generic_passes;
  const int64_t v = c;
  if (reset) c = 0;
  return v;
}

int dnmf_set_force_generic(int on) {
  tls().force_generic = on ? 1 : 0;
  return 0;
}

int dnmf_set_tc_min_elems(int64_t elems) {
  tc_set_min_elems(elems);
  return 0;
}

int dnmf_device_info(int* sms, int* cc_major, int* cc_minor) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return cuda_fail(e, "dnmf_device_info");
  int a = 0, b = 0, c = 0;
  cudaDeviceGetAttribute(&a, cudaDevAttrMultiProcessorCount, dev);
  cudaDeviceGetAttribute(&b, cudaDevAttrComputeCapabilityMajor, dev);
  cudaDeviceGetAttribute(&c, cudaDevAttrComputeCapabilityMinor, dev);
  if (sms) *sms = a;
  if (cc_major) *cc_major = b;
  if (cc_minor) *cc_minor = c;
  return 0;
}

}  // extern "C"
