// Host-side launchers for the factor-sized kernels that are templated on the padded factor width.
// Instantiated per dtype in inst_small_f32.cu / inst_small_f64.cu.
#pragma once
#include "common.cuh"
#include "generic_small.cuh"
#include "launch_passes.cuh"

namespace dnmf {

struct GramPlan { int64_t blocks, rows_per_block; };
inline GramPlan gram_plan(int64_t rows) {
  GramPlan g;
  int64_t want = (int64_t)sm_count() * 4;
  int64_t tiles = ceil_div(rows > 0 ? rows : 1, kGramTR);
  int64_t nb = tiles < want ? tiles : want;
  g.rows_per_block = round_up(ceil_div(rows > 0 ? rows : 1, nb), kGramTR);
  g.blocks = ceil_div(rows > 0 ? rows : 1, g.rows_per_block);
  return g;
}

struct SumPlan { int64_t chunks, per_chunk; };
inline SumPlan sum_plan(int64_t len, int64_t gran, int64_t max_chunks) {
  SumPlan s;
  int64_t c = ceil_div(len > 0 ? len : 1, gran);
  if (c > max_chunks) c = max_chunks;
  s.per_chunk = round_up(ceil_div(len > 0 ? len : 1, c), gran);
  s.chunks = ceil_div(len > 0 ? len : 1, s.per_chunk);
  return s;
}

struct ResPlan { int64_t col_blocks, chunks, chunk; };
inline ResPlan residual_plan(int64_t m, int64_t n) {
  ResPlan r;
  r.col_blocks = ceil_div(n > 0 ? n : 1, kColPassThreads);
  int64_t want = ceil_div((int64_t)sm_count() * 8, r.col_blocks);
  if (want < 1) want = 1;
  if (want > 256) want = 256;
  r.chunk = round_up(ceil_div(m > 0 ? m : 1, want), kColPassBR);
  r.chunks = ceil_div(m > 0 ? m : 1, r.chunk);
  return r;
}

template <typename T>
int gram_dispatch(const T* X, int64_t ldx, int64_t rows, int k, int trans, T* G, T* ws, cudaStream_t st);
// mode 0: MU (p0 = eps), mode 1: BCD projected gradient (p0 = Lipschitz bound)
template <typename T>
int row_update_dispatch(int mode, T* W, int64_t ldw, const T* X, int64_t ldx, const T* V, int64_t ldv, const T* G,
                        int64_t m, int k, T p0, const double* p0_dev, cudaStream_t st, int splits = 1, int64_t sstride = 0);
// mode 0: MU, 1: BCD, 2: HALS
template <typename T>
int col_update_dispatch(int mode, T* H, int64_t ldh, const T* X, int64_t ldx, const T* Y, int64_t ysk, int64_t ysc,
                        const T* G, int k, int64_t n, T p0, int clamp, const double* p0_dev, cudaStream_t st, int splits = 1,
                        int64_t sstride = 0);
// (TA: element type of A; 16-bit A with fp32 factors is instantiated in inst_col_a16.cu)
template <typename T, typename TA = T>
int residual_dispatch(const TA* A, int64_t lda, const T* W, int64_t ldw, const T* H, int64_t ldh, int64_t m,
                      int64_t n, int k, int64_t chunk, unsigned gx, unsigned gy, double* P, double* col_num,
                      double* col_den, cudaStream_t st);
template <typename T>
int hals_w_col_dispatch(T* W, int64_t ldw, const T* V, int64_t ldv, const T* G, int64_t m, int k, int kk, T eps,
                        double* P, unsigned nb, cudaStream_t st);

#ifdef DNMF_INSTANTIATE_SMALL
template <typename T>
int gram_dispatch(const T* X, int64_t ldx, int64_t rows, int k, int trans, T* G, T* ws, cudaStream_t st) {
  const int kp = padded_k(k);
  const GramPlan g = gram_plan(rows);
  DNMF_DISPATCH_KP(kp, {
    if (trans) gram_partial_kernel<T, KP, true><<<(unsigned)g.blocks, kGramThreads, 0, st>>>(X, ldx, rows, k, g.rows_per_block, ws);
    else gram_partial_kernel<T, KP, false><<<(unsigned)g.blocks, kGramThreads, 0, st>>>(X, ldx, rows, k, g.rows_per_block, ws);
    DNMF_LAUNCH_CHECK("gram_partial_kernel");
    gram_reduce_kernel<T><<<(unsigned)ceil_div((int64_t)k * k * 32, 256), 256, 0, st>>>(ws, (int)g.blocks, KP, k, G);
    DNMF_LAUNCH_CHECK("gram_reduce_kernel");
  });
  return 0;
}

template <typename T>
int row_update_dispatch(int mode, T* W, int64_t ldw, const T* X, int64_t ldx, const T* V, int64_t ldv, const T* G,
                        int64_t m, int k, T p0, const double* p0_dev, cudaStream_t st, int splits, int64_t sstride) {
  const int kp = padded_k(k);
  DNMF_DISPATCH_KP(kp, {
    constexpr int RB = RowUpdCfg<T, KP>::RB;
    const unsigned grid = (unsigned)ceil_div(m, RB);
    if (mode == 0) row_update_kernel<T, KP, 0><<<grid, kRowUpdThreads, 0, st>>>(W, ldw, X, ldx, V, ldv, G, m, k, p0, p0_dev, splits, sstride);
    else row_update_kernel<T, KP, 1><<<grid, kRowUpdThreads, 0, st>>>(W, ldw, X, ldx, V, ldv, G, m, k, p0, p0_dev, splits, sstride);
  });
  DNMF_LAUNCH_CHECK("row_update_kernel");
  return 0;
}

template <typename T>
int col_update_dispatch(int mode, T* H, int64_t ldh, const T* X, int64_t ldx, const T* Y, int64_t ysk, int64_t ysc,
                        const T* G, int k, int64_t n, T p0, int clamp, const double* p0_dev, cudaStream_t st, int splits,
                        int64_t sstride) {
  const int kp = padded_k(k);
  const unsigned grid = (unsigned)ceil_div(n, kColUpdThreads);
  DNMF_DISPATCH_KP(kp, {
    if (mode == 0) col_update_kernel<T, KP, 0><<<grid, kColUpdThreads, 0, st>>>(H, ldh, X, ldx, Y, ysk, ysc, G, k, n, p0, clamp, p0_dev, splits, sstride);
    else if (mode == 1) col_update_kernel<T, KP, 1><<<grid, kColUpdThreads, 0, st>>>(H, ldh, X, ldx, Y, ysk, ysc, G, k, n, p0, clamp, p0_dev, splits, sstride);
    else col_update_kernel<T, KP, 2><<<grid, kColUpdThreads, 0, st>>>(H, ldh, X, ldx, Y, ysk, ysc, G, k, n, p0, clamp, p0_dev, splits, sstride);
  });
  DNMF_LAUNCH_CHECK("col_update_kernel");
  return 0;
}

template <typename T, typename TA>
int residual_dispatch(const TA* A, int64_t lda, const T* W, int64_t ldw, const T* H, int64_t ldh, int64_t m,
                      int64_t n, int k, int64_t chunk, unsigned gx, unsigned gy, double* P, double* col_num,
                      double* col_den, cudaStream_t st) {
  const int kp = padded_k(k);
  dim3 grid(gx, gy);
  DNMF_DISPATCH_KP(kp, (residual_kernel<T, KP, TA><<<grid, kColPassThreads, 0, st>>>(A, lda, W, ldw, H, ldh, m, n, k, chunk, P, col_num, col_den)));
  DNMF_LAUNCH_CHECK("residual_kernel");
  return 0;
}

template <typename T>
int hals_w_col_dispatch(T* W, int64_t ldw, const T* V, int64_t ldv, const T* G, int64_t m, int k, int kk, T eps,
                        double* P, unsigned nb, cudaStream_t st) {
  const int kp = padded_k(k);
  DNMF_DISPATCH_KP(kp, (hals_w_col_kernel<T, KP><<<nb, 256, 0, st>>>(W, ldw, V, ldv, G, m, k, kk, eps, P)));
  DNMF_LAUNCH_CHECK("hals_w_col_kernel");
  return 0;
}
#endif

}  // namespace dnmf
