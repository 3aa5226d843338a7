// Host-side launchers for the generic A-streaming passes.  The kernels are instantiated in their own
// translation units (inst_row_*.cu / inst_col_*.cu) so the library builds in parallel.
#pragma once
#include "common.cuh"
#include "generic_passes.cuh"

namespace dnmf {

#define DNMF_DISPATCH_KP(KPV, ...)                     \
  switch (KPV) {                                  \
    case 4:  { constexpr int KP = 4;  __VA_ARGS__; } break;  \
    case 8:  { constexpr int KP = 8;  __VA_ARGS__; } break;  \
    case 16: { constexpr int KP = 16; __VA_ARGS__; } break;  \
    case 32: { constexpr int KP = 32; __VA_ARGS__; } break;  \
    default: { constexpr int KP = 64; __VA_ARGS__; } break;  \
  }

#define DNMF_DISPATCH_T(dtype, ...)                          \
  if ((dtype) == DNMF_F32) { using T = float; __VA_ARGS__; } \
  else { using T = double; __VA_ARGS__; }

template <typename T, int KP, bool KL>
Split row_pass_plan(int64_t m, int64_t n) {
  // (min chunk of 2 K-tiles: mid-sized shards such as 1024 x 256 still spread over many CTAs)
  return plan_split(m, RowPassCfg<T, KP, KL>::BM, n, kRowPassBK, 2 * kRowPassBK);
}
template <typename T, int KP, bool KL>
Split col_pass_plan(int64_t m, int64_t n) {
  return plan_split(n, (int64_t)kColPassThreads * ColPassCfg<T, KP, KL>::CPT, m, kColPassBR, kColPassBR);
}

// fixed-order sum of split partials with rows ldp apart (see reduce_partials_kernel)
template <typename T>
inline int launch_reduce(const T* P, int64_t split_stride, int splits, int64_t R, int64_t C, int64_t ldp, T* out,
                         int64_t so_r, int64_t so_c, cudaStream_t st) {
  const int64_t tot = R * C;
  if (tot == 0) return 0;
  reduce_partials_kernel<T><<<(unsigned)ceil_div(tot, 256), 256, 0, st>>>(P, split_stride, splits, R, C, out, so_r, so_c, ldp);
  DNMF_LAUNCH_CHECK("reduce_partials_kernel");
  return 0;
}

// V[m x k] = A H^T  or  (A/(WH+eps)) H^T   (A's elements of type TA are widened to T as they are staged)
template <typename T, int KP, bool KL, typename TA = T>
int run_row_pass(const TA* A, int64_t lda, const T* H, int64_t ldh, const T* W, int64_t ldw, T* V, int64_t ldv,
                 int64_t m, int64_t n, int k, T eps, void* ws, int64_t ws_bytes, cudaStream_t st) {
  using Cfg = RowPassCfg<T, KP, KL>;
  const Split sp = row_pass_plan<T, KP, KL>(m, n);
  const int vec_ok = (((uintptr_t)A % (Cfg::VN * sizeof(TA))) == 0) && (lda % Cfg::VN == 0);
  auto kern = row_pass_kernel<T, KP, KL, TA>;
  if (Cfg::smem_bytes > 48 * 1024)
    if (int rc = smem_attr_once<row_pass_kernel<T, KP, KL, TA>>((int)Cfg::smem_bytes, "row_pass smem attribute")) return rc;
  dim3 grid((unsigned)sp.blocks, (unsigned)sp.splits);
  if (sp.splits == 1) {
    kern<<<grid, kRowPassThreads, Cfg::smem_bytes, st>>>(A, lda, H, ldh, W, ldw, V, ldv, 0, m, n, k, sp.chunk, eps, vec_ok);
    DNMF_LAUNCH_CHECK("row_pass_kernel");
    return 0;
  }
  const int64_t need = sp.splits * m * k * (int64_t)sizeof(T);
  if (ws == nullptr || ws_bytes < need) return fail(DNMF_E_WORKSPACE, "row pass needs %lld workspace bytes, got %lld", (long long)need, (long long)ws_bytes);
  T* P = reinterpret_cast<T*>(ws);
  kern<<<grid, kRowPassThreads, Cfg::smem_bytes, st>>>(A, lda, H, ldh, W, ldw, P, k, m * k, m, n, k, sp.chunk, eps, vec_ok);
  DNMF_LAUNCH_CHECK("row_pass_kernel");
  return launch_reduce<T>(P, m * k, (int)sp.splits, m, k, k, V, ldv, 1, st);
}

// Y[k x n] = W^T A  or  W^T (A/(WH+eps));  transposed_out: Y^T [n x k]
template <typename T, int KP, bool KL, typename TA = T>
int run_col_pass(const TA* A, int64_t lda, const T* W, int64_t ldw, const T* H, int64_t ldh, T* Y, int64_t ldy,
                 int64_t m, int64_t n, int k, T eps, int transposed_out, void* ws, int64_t ws_bytes,
                 cudaStream_t st) {
  constexpr int CPT = ColPassCfg<T, KP, KL>::CPT;
  const Split sp = col_pass_plan<T, KP, KL>(m, n);
  const int vec_ok = (((uintptr_t)A % (CPT * sizeof(TA))) == 0) && (lda % CPT == 0);
  dim3 grid((unsigned)sp.blocks, (unsigned)sp.splits);
  if (sp.splits == 1 && !transposed_out) {
    col_pass_kernel<T, KP, KL, TA><<<grid, kColPassThreads, 0, st>>>(A, lda, W, ldw, H, ldh, Y, ldy, 0, m, n, k, sp.chunk, eps, vec_ok);
    DNMF_LAUNCH_CHECK("col_pass_kernel");
    return 0;
  }
  const int64_t need = sp.splits * (int64_t)k * n * (int64_t)sizeof(T);
  if (ws == nullptr || ws_bytes < need) return fail(DNMF_E_WORKSPACE, "col pass needs %lld workspace bytes, got %lld", (long long)need, (long long)ws_bytes);
  T* P = reinterpret_cast<T*>(ws);
  col_pass_kernel<T, KP, KL, TA><<<grid, kColPassThreads, 0, st>>>(A, lda, W, ldw, H, ldh, P, n, (int64_t)k * n, m, n, k, sp.chunk, eps, vec_ok);
  DNMF_LAUNCH_CHECK("col_pass_kernel");
  if (transposed_out) return launch_reduce<T>(P, (int64_t)k * n, (int)sp.splits, k, n, n, Y, 1, ldy, st);
  return launch_reduce<T>(P, (int64_t)k * n, (int)sp.splits, k, n, n, Y, ldy, 1, st);
}


template <typename T>
Split row_pass_plan_rt(int kp, bool kl, int64_t m, int64_t n) {
  Split sp;
  DNMF_DISPATCH_KP(kp, sp = kl ? row_pass_plan<T, KP, true>(m, n) : row_pass_plan<T, KP, false>(m, n));
  return sp;
}
template <typename T>
Split col_pass_plan_rt(int kp, bool kl, int64_t m, int64_t n) {
  Split sp;
  DNMF_DISPATCH_KP(kp, sp = kl ? col_pass_plan<T, KP, true>(m, n) : col_pass_plan<T, KP, false>(m, n));
  return sp;
}

// defined (explicitly instantiated) in inst_row_f32.cu / inst_row_f64.cu / inst_col_f32.cu / inst_col_f64.cu, and for
// 16-bit A with fp32 factors in inst_row_a16.cu / inst_col_a16.cu
template <typename T, typename TA = T>
int row_pass_dispatch(bool kl, const TA* A, int64_t lda, const T* H, int64_t ldh, const T* W, int64_t ldw, T* V,
                      int64_t ldv, int64_t m, int64_t n, int k, T eps, void* ws, int64_t ws_bytes, cudaStream_t st);
template <typename T, typename TA = T>
int col_pass_dispatch(bool kl, const TA* A, int64_t lda, const T* W, int64_t ldw, const T* H, int64_t ldh, T* Y,
                      int64_t ldy, int64_t m, int64_t n, int k, T eps, int transposed_out, void* ws,
                      int64_t ws_bytes, cudaStream_t st);

#ifdef DNMF_INSTANTIATE_ROW
template <typename T, typename TA>
int row_pass_dispatch(bool kl, const TA* A, int64_t lda, const T* H, int64_t ldh, const T* W, int64_t ldw, T* V,
                      int64_t ldv, int64_t m, int64_t n, int k, T eps, void* ws, int64_t ws_bytes, cudaStream_t st) {
  const int kp = padded_k(k);
  DNMF_DISPATCH_KP(kp, {
    if (kl) return run_row_pass<T, KP, true, TA>(A, lda, H, ldh, W, ldw, V, ldv, m, n, k, eps, ws, ws_bytes, st);
    return run_row_pass<T, KP, false, TA>(A, lda, H, ldh, W, ldw, V, ldv, m, n, k, eps, ws, ws_bytes, st);
  });
  return 0;
}
#endif
#ifdef DNMF_INSTANTIATE_COL
template <typename T, typename TA>
int col_pass_dispatch(bool kl, const TA* A, int64_t lda, const T* W, int64_t ldw, const T* H, int64_t ldh, T* Y,
                      int64_t ldy, int64_t m, int64_t n, int k, T eps, int transposed_out, void* ws,
                      int64_t ws_bytes, cudaStream_t st) {
  const int kp = padded_k(k);
  DNMF_DISPATCH_KP(kp, {
    if (kl) return run_col_pass<T, KP, true, TA>(A, lda, W, ldw, H, ldh, Y, ldy, m, n, k, eps, transposed_out, ws, ws_bytes, st);
    return run_col_pass<T, KP, false, TA>(A, lda, W, ldw, H, ldh, Y, ldy, m, n, k, eps, transposed_out, ws, ws_bytes, st);
  });
  return 0;
}
#endif

}  // namespace dnmf
