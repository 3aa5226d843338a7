// Shared helpers for libdnmf (sm_100a).  See include/dnmf.h for the C-ABI.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/dnmf.h"

namespace dnmf {

// ---- thread-local status -------------------------------------------------------
struct TlsState {
  char msg[512];
  int last_path;
  int64_t launches;
  int force_generic;
  int64_t tc_passes;        // A-streaming passes routed to the tcgen05 kernels on this thread
  int64_t generic_passes;   // ... and to the generic CUDA-core kernels
};
TlsState& tls();

int fail(int code, const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* where);

#define DNMF_CHECK_ARG(cond, what) \
  do { if (!(cond)) return ::dnmf::fail(DNMF_E_ARG, "%s: bad argument: %s", __func__, what); } while (0)

#define DNMF_LAUNCH_CHECK(where)                                  \
  do {                                                            \
    ::dnmf::tls().launches++;                                     \
    cudaError_t _e = cudaPeekAtLastError();                       \
    if (_e != cudaSuccess) return ::dnmf::cuda_fail(_e, where);   \
  } while (0)

// Raise kernel KERN's dynamic shared-memory limit to `bytes`, once per kernel: on its first launch, which is eager (never
// during a stream capture).
template <auto KERN>
int smem_attr_once(int bytes, const char* where) {
  static bool done = false;
  if (!done) {
    cudaError_t e = cudaFuncSetAttribute(KERN, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e != cudaSuccess) return cuda_fail(e, where);
    done = true;
  }
  return 0;
}

int sm_count();

inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
inline int64_t round_up(int64_t a, int64_t b) { return ceil_div(a, b) * b; }

// padded factor width used as a template parameter
inline int padded_k(int64_t k) {
  if (k <= 4) return 4;
  if (k <= 8) return 8;
  if (k <= 16) return 16;
  if (k <= 32) return 32;
  return 64;
}

// ---- split planning (must be a pure function of the shape: the workspace query and the launch
//      agree, and the reduction order is fixed => deterministic results) ----------------------
struct Split {
  int64_t blocks;      // blocks along the streamed (non-reduced) dimension
  int64_t splits;      // chunks along the reduced dimension (partial buffers)
  int64_t chunk;       // elements of the reduced dimension per split (multiple of `align`)
};
Split plan_split(int64_t outer, int64_t outer_tile, int64_t reduce_len, int64_t align, int64_t min_chunk);

// ---- device helpers -----------------------------------------------------------
template <typename T> struct VecOf;
template <> struct VecOf<float> { using type = float4; static constexpr int N = 4; };
template <> struct VecOf<double> { using type = double2; static constexpr int N = 2; };

template <typename T>
__device__ __forceinline__ void vload(const T* p, T (&out)[VecOf<T>::N]) {
  using V = typename VecOf<T>::type;
  V v = *reinterpret_cast<const V*>(p);
  const T* q = reinterpret_cast<const T*>(&v);
#pragma unroll
  for (int i = 0; i < VecOf<T>::N; ++i) out[i] = q[i];
}

template <typename T>
__device__ __forceinline__ void vstore(T* p, const T (&in)[VecOf<T>::N]) {
  using V = typename VecOf<T>::type;
  V v;
  T* q = reinterpret_cast<T*>(&v);
#pragma unroll
  for (int i = 0; i < VecOf<T>::N; ++i) q[i] = in[i];
  *reinterpret_cast<V*>(p) = v;
}

// widening of an element of A (fp32 / fp64, or the 16-bit storage formats DNMF_A_F16 / DNMF_A_BF16)
template <typename T>
__device__ __forceinline__ double to_f64(T x) { return (double)x; }
__device__ __forceinline__ double to_f64(__half x) { return (double)__half2float(x); }
__device__ __forceinline__ double to_f64(__nv_bfloat16 x) { return (double)__bfloat162float(x); }

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// deterministic block-wide sum of doubles; result valid on thread 0
template <int NT>
__device__ __forceinline__ double block_sum(double v, double* red /* [NT/32] shared */) {
  v = warp_sum(v);
  int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) red[w] = v;
  __syncthreads();
  double r = 0.0;
  if (threadIdx.x == 0) {
#pragma unroll
    for (int i = 0; i < NT / 32; ++i) r += red[i];
  }
  __syncthreads();
  return r;
}

}  // namespace dnmf
