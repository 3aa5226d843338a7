// extern "C" entry points of libdnmf (see include/dnmf.h).  Dispatch: tcgen05 path (dnmf_tc.cu) when the
// shape is eligible, generic CUDA-core kernels otherwise.  No CPU fallback anywhere.
#include "common.cuh"
#include "launch_passes.cuh"
#include "launch_small.cuh"
#include "tc_api.cuh"

using namespace dnmf;

#define DISPATCH_T DNMF_DISPATCH_T
// T: factor / output type, TA: element type of A
#define DISPATCH_A(dtype, ...)                                                           \
  if ((dtype) == DNMF_A_F16) { using T = float; using TA = __half; __VA_ARGS__; }        \
  else if ((dtype) == DNMF_A_BF16) { using T = float; using TA = __nv_bfloat16; __VA_ARGS__; } \
  else if ((dtype) == DNMF_F32) { using T = float; using TA = float; __VA_ARGS__; }      \
  else { using T = double; using TA = double; __VA_ARGS__; }

namespace {

inline int check_common(int64_t m, int64_t n, int64_t k, int dtype) {
  if (dtype != DNMF_F32 && dtype != DNMF_F64) return fail(DNMF_E_ARG, "dtype must be DNMF_F32 or DNMF_F64");
  if (m < 0 || n < 0 || k < 0) return fail(DNMF_E_ARG, "negative dimension");
  if (k > DNMF_MAX_K) return fail(DNMF_E_UNSUPPORTED, "k=%lld exceeds DNMF_MAX_K=%d", (long long)k, DNMF_MAX_K);
  return 0;
}

// entry points that read the data shard A also accept the 16-bit storage codes (fp32 factors and outputs)
inline bool is_a16(int dtype) { return dtype == DNMF_A_F16 || dtype == DNMF_A_BF16; }
inline int check_a(int64_t m, int64_t n, int64_t k, int dtype) {
  return check_common(m, n, k, is_a16(dtype) ? DNMF_F32 : dtype);
}

// element size of the factors and outputs
inline size_t esize(int dtype) { return dtype == DNMF_F64 ? 8 : 4; }

// records which kernels serve an A-streaming pass (dnmf_last_path, dnmf_pass_count)
void note_pass(bool tc) {
  tls().last_path = tc ? 1 : 0;
  (tc ? tls().tc_passes : tls().generic_passes)++;
}

// The A-streaming passes: AH (out = V = A H^T), WTA (out = Y = W^T A, or Y^T with transposed_out) and the KL forms
// KL_UHT / KL_WTU (A / (W H + eps) in place of A); W (AH) and H (WTA) are not read.  view4 == nullptr: the plain entry
// point, tcgen05 kernels when eligible, generic kernels otherwise.  view4 != nullptr: the _p form, which leaves the
// split partials in the workspace and describes them in view4, and serves only calls the tcgen05 path takes.
int run_pass(int op, const void* A, int64_t lda, const void* W, int64_t ldw, const void* H, int64_t ldh, void* out,
             int64_t ldo, int64_t m, int64_t n, int64_t k, double eps, int transposed_out, int dtype, void* ws,
             int64_t ws_bytes, int64_t* view4, cudaStream_t st) {
  const bool kl = op == DNMF_OP_KL_UHT || op == DNMF_OP_KL_WTU;
  const bool rows = op == DNMF_OP_AH || op == DNMF_OP_KL_UHT;    // one output row per row of A
  const bool deferred = view4 != nullptr;
  if (int rc = check_a(m, n, k, dtype)) return rc;
  DNMF_CHECK_ARG(A && (op == DNMF_OP_AH || W) && (op == DNMF_OP_WTA || H) && (deferred || out), "null pointer");
  DNMF_CHECK_ARG(lda >= n && (op == DNMF_OP_AH || ldw >= k) && (op == DNMF_OP_WTA || ldh >= n) &&
                 (deferred || ldo >= (rows || transposed_out ? k : n)), "leading dimension too small");
  if ((rows ? m : n) == 0 || k == 0) return deferred ? DNMF_E_UNSUPPORTED : 0;
  const bool tc = tc_eligible(op, A, lda, m, n, k, dtype);
  if (deferred && !tc) return DNMF_E_UNSUPPORTED;
  note_pass(tc);
  if (tc) {
    TcPartials d;
    if (int rc = tc_pass(op, dtype, A, lda, (const float*)W, ldw, (const float*)H, ldh, (float*)out, ldo, m, n, (int)k,
                         (float)eps, transposed_out, ws, ws_bytes, st, deferred ? &d : nullptr))
      return rc;
    if (deferred) {
      view4[0] = (int64_t)(uintptr_t)d.P; view4[1] = d.ldp; view4[2] = d.splits; view4[3] = d.split_stride;
    }
    return 0;
  }
  DISPATCH_A(dtype, {
    if (rows) return row_pass_dispatch<T, TA>(kl, (const TA*)A, lda, (const T*)H, ldh, (const T*)W, ldw, (T*)out, ldo, m, n, (int)k, (T)eps, ws, ws_bytes, st);
    return col_pass_dispatch<T, TA>(kl, (const TA*)A, lda, (const T*)W, ldw, (const T*)H, ldh, (T*)out, ldo, m, n, (int)k, (T)eps, transposed_out, ws, ws_bytes, st);
  });
  return 0;
}

}  // namespace

extern "C" {

int64_t dnmf_workspace_bytes(int op, int64_t m, int64_t n, int64_t k, int dtype) {
  if (check_a(m, n, k, dtype) != 0) return -1;
  const int kp = padded_k(k);
  int64_t bytes = 0;
  switch (op) {
    case DNMF_OP_AH:
    case DNMF_OP_KL_UHT: {
      const bool kl = (op == DNMF_OP_KL_UHT);
      Split sp;
      DISPATCH_A(dtype, sp = row_pass_plan_rt<T>(kp, kl, m, n));
      bytes = sp.splits > 1 ? sp.splits * m * k * (int64_t)esize(dtype) : 0;
      break;
    }
    case DNMF_OP_WTA:
    case DNMF_OP_KL_WTU: {
      const bool kl = (op == DNMF_OP_KL_WTU);
      Split sp;
      DISPATCH_A(dtype, sp = col_pass_plan_rt<T>(kp, kl, m, n));
      bytes = sp.splits * k * n * (int64_t)esize(dtype);   // also covers transposed_out with one split
      break;
    }
    case DNMF_OP_GRAM: {
      const GramPlan g = gram_plan(m > n ? m : n);
      bytes = g.blocks * kp * kp * (int64_t)esize(dtype);
      break;
    }
    case DNMF_OP_RESIDUAL: {
      const ResPlan r = residual_plan(m, n);
      bytes = r.col_blocks * r.chunks * 2 * (int64_t)sizeof(double);
      break;
    }
    case DNMF_OP_AH_RESIDUAL: {
      // fused tcgen05 pass, or (fallback) the A H^T pass followed by the residual pass in the same workspace
      const int64_t a = dnmf_workspace_bytes(DNMF_OP_AH, m, n, k, dtype);
      const int64_t r = dnmf_workspace_bytes(DNMF_OP_RESIDUAL, m, n, k, dtype);
      bytes = a > r ? a : r;
      break;
    }
    case DNMF_OP_SUMS: {
      // max over: colsum(m x k), rowsum(k x n), sqnorm(m x n | m x k | k x n), hals_w_col(m)
      int64_t d = 0, v;
      v = sum_plan(m, 64, 1024).chunks * (k > 0 ? k : 1); if (v > d) d = v;
      v = sum_plan(n, 2048, 256).chunks * (k > 0 ? k : 1); if (v > d) d = v;
      v = sum_plan(n, 2048, 256).chunks * (m > 0 ? m : 1); if (v > d) d = v;
      v = sum_plan(k, 2048, 256).chunks * (m > 0 ? m : 1); if (v > d) d = v;
      v = ceil_div(m > 0 ? m : 1, 256); if (v > d) d = v;
      bytes = d * (int64_t)sizeof(double);
      break;
    }
    case DNMF_OP_NNZ:
      bytes = 0;
      break;
    default:
      fail(DNMF_E_ARG, "unknown op %d", op);
      return -1;
  }
  const int64_t tcb = tc_workspace_bytes(op, m, n, k, dtype);
  if (tcb > bytes) bytes = tcb;
  return round_up(bytes, 256) + 256;
}

int dnmf_ah(const void* A, int64_t lda, const void* H, int64_t ldh, void* V, int64_t ldv, int64_t m, int64_t n,
            int64_t k, int dtype, int math_mode, void* ws, int64_t ws_bytes, void* stream) {
  return run_pass(DNMF_OP_AH, A, lda, nullptr, 0, H, ldh, V, ldv, m, n, k, 0.0, 0, dtype, ws, ws_bytes, nullptr, (cudaStream_t)stream);
}

int dnmf_wta(const void* A, int64_t lda, const void* W, int64_t ldw, void* Y, int64_t ldy, int64_t m, int64_t n,
             int64_t k, int transposed_out, int dtype, int math_mode, void* ws, int64_t ws_bytes, void* stream) {
  return run_pass(DNMF_OP_WTA, A, lda, W, ldw, nullptr, 0, Y, ldy, m, n, k, 0.0, transposed_out, dtype, ws, ws_bytes, nullptr, (cudaStream_t)stream);
}

int dnmf_kl_uht(const void* A, int64_t lda, const void* W, int64_t ldw, const void* H, int64_t ldh, void* V,
                int64_t ldv, int64_t m, int64_t n, int64_t k, double eps, int dtype, int math_mode, void* ws,
                int64_t ws_bytes, void* stream) {
  return run_pass(DNMF_OP_KL_UHT, A, lda, W, ldw, H, ldh, V, ldv, m, n, k, eps, 0, dtype, ws, ws_bytes, nullptr, (cudaStream_t)stream);
}

int dnmf_kl_wtu(const void* A, int64_t lda, const void* W, int64_t ldw, const void* H, int64_t ldh, void* Y,
                int64_t ldy, int64_t m, int64_t n, int64_t k, double eps, int transposed_out, int dtype,
                int math_mode, void* ws, int64_t ws_bytes, void* stream) {
  return run_pass(DNMF_OP_KL_WTU, A, lda, W, ldw, H, ldh, Y, ldy, m, n, k, eps, transposed_out, dtype, ws, ws_bytes, nullptr, (cudaStream_t)stream);
}

int dnmf_gram(const void* X, int64_t ldx, int64_t rows, int64_t k, int trans, void* G, int dtype, void* ws,
              int64_t ws_bytes, void* stream) {
  if (int rc = check_common(rows, 0, k, dtype)) return rc;
  DNMF_CHECK_ARG(X && G, "null pointer");
  DNMF_CHECK_ARG(ldx >= (trans ? rows : k), "leading dimension too small");
  if (k == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const int kp = padded_k(k);
  const GramPlan g = gram_plan(rows);
  const int64_t need = g.blocks * kp * kp * (int64_t)esize(dtype);
  if (ws == nullptr || ws_bytes < need) return fail(DNMF_E_WORKSPACE, "gram needs %lld workspace bytes, got %lld", (long long)need, (long long)ws_bytes);
  DISPATCH_T(dtype, return gram_dispatch<T>((const T*)X, ldx, rows, (int)k, trans, (T*)G, (T*)ws, st));
  return 0;
}

int dnmf_mu_update_w(void* W, int64_t ldw, const void* V, int64_t ldv, const void* G, int64_t m, int64_t k,
                     double eps, int dtype, void* stream) {
  if (int rc = check_common(m, 0, k, dtype)) return rc;
  DNMF_CHECK_ARG(W && V && G, "null pointer");
  if (m == 0 || k == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  DISPATCH_T(dtype, return row_update_dispatch<T>(0, (T*)W, ldw, (const T*)W, ldw, (const T*)V, ldv, (const T*)G, m, (int)k, (T)eps, nullptr, st));
  return 0;
}

static int bcd_pg_w(void* W, int64_t ldw, const void* Wm, int64_t ldwm, const void* V, int64_t ldv, const void* G,
                    int64_t m, int64_t k, double L, const double* L_dev, int dtype, void* stream) {
  if (int rc = check_common(m, 0, k, dtype)) return rc;
  DNMF_CHECK_ARG(W && Wm && V && G, "null pointer");
  if (m == 0 || k == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  DISPATCH_T(dtype, return row_update_dispatch<T>(1, (T*)W, ldw, (const T*)Wm, ldwm, (const T*)V, ldv, (const T*)G, m, (int)k, (T)L, L_dev, st));
  return 0;
}

int dnmf_bcd_pg_w(void* W, int64_t ldw, const void* Wm, int64_t ldwm, const void* V, int64_t ldv, const void* G,
                  int64_t m, int64_t k, double L, int dtype, void* stream) {
  return bcd_pg_w(W, ldw, Wm, ldwm, V, ldv, G, m, k, L, nullptr, dtype, stream);
}

int dnmf_bcd_pg_w_dev(void* W, int64_t ldw, const void* Wm, int64_t ldwm, const void* V, int64_t ldv, const void* G,
                      int64_t m, int64_t k, const double* L_dev, int dtype, void* stream) {
  DNMF_CHECK_ARG(L_dev, "null Lipschitz pointer");
  return bcd_pg_w(W, ldw, Wm, ldwm, V, ldv, G, m, k, 1.0, L_dev, dtype, stream);
}

static int col_update(int mode, void* H, int64_t ldh, const void* X, int64_t ldx, const void* Y, int64_t ysk,
                      int64_t ysc, const void* G, int64_t k, int64_t n, double p0, int clamp, int dtype,
                      void* stream, const double* p0_dev = nullptr) {
  if (int rc = check_common(0, n, k, dtype)) return rc;
  DNMF_CHECK_ARG(H && X && Y && G, "null pointer");
  if (n == 0 || k == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  DISPATCH_T(dtype, return col_update_dispatch<T>(mode, (T*)H, ldh, (const T*)X, ldx, (const T*)Y, ysk, ysc, (const T*)G, (int)k, n, (T)p0, clamp, p0_dev, st));
  return 0;
}

int dnmf_mu_update_h(void* H, int64_t ldh, const void* Y, int64_t y_stride_k, int64_t y_stride_c, const void* G,
                     int64_t k, int64_t n, double eps, int clamp, int dtype, void* stream) {
  return col_update(0, H, ldh, H, ldh, Y, y_stride_k, y_stride_c, G, k, n, eps, clamp, dtype, stream);
}

int dnmf_bcd_pg_h(void* H, int64_t ldh, const void* Hm, int64_t ldhm, const void* Y, int64_t y_stride_k,
                  int64_t y_stride_c, const void* G, int64_t k, int64_t n, double L, int dtype, void* stream) {
  return col_update(1, H, ldh, Hm, ldhm, Y, y_stride_k, y_stride_c, G, k, n, L, 0, dtype, stream);
}

int dnmf_bcd_pg_h_dev(void* H, int64_t ldh, const void* Hm, int64_t ldhm, const void* Y, int64_t y_stride_k,
                      int64_t y_stride_c, const void* G, int64_t k, int64_t n, const double* L_dev, int dtype, void* stream) {
  DNMF_CHECK_ARG(L_dev, "null Lipschitz pointer");
  return col_update(1, H, ldh, Hm, ldhm, Y, y_stride_k, y_stride_c, G, k, n, 1.0, 0, dtype, stream, L_dev);
}

int dnmf_hals_h(void* H, int64_t ldh, const void* Y, int64_t y_stride_k, int64_t y_stride_c, const void* G,
                int64_t k, int64_t n, double eps, int dtype, void* stream) {
  return col_update(2, H, ldh, H, ldh, Y, y_stride_k, y_stride_c, G, k, n, eps, 0, dtype, stream);
}

int dnmf_kl_update_w(void* W, int64_t ldw, const void* V, int64_t ldv, const void* x, int64_t m, int64_t k,
                     double eps, int dtype, void* stream) {
  if (int rc = check_common(m, 0, k, dtype)) return rc;
  DNMF_CHECK_ARG(W && V && x, "null pointer");
  if (m == 0 || k == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  DISPATCH_T(dtype, (kl_update_w_kernel<T><<<(unsigned)ceil_div(m * k, 256), 256, 0, st>>>((T*)W, ldw, (const T*)V, ldv, (const T*)x, m, (int)k, (T)eps, 1, 0)));
  DNMF_LAUNCH_CHECK("kl_update_w_kernel");
  return 0;
}

int dnmf_kl_update_h(void* H, int64_t ldh, const void* Y, int64_t y_stride_k, int64_t y_stride_c, const void* x,
                     int64_t k, int64_t n, double eps, int clamp, int dtype, void* stream) {
  if (int rc = check_common(0, n, k, dtype)) return rc;
  DNMF_CHECK_ARG(H && Y && x, "null pointer");
  if (n == 0 || k == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  DISPATCH_T(dtype, (kl_update_h_kernel<T><<<(unsigned)ceil_div(k * n, 256), 256, 0, st>>>((T*)H, ldh, (const T*)Y, y_stride_k, y_stride_c, (const T*)x, (int)k, n, (T)eps, clamp, 1, 0)));
  DNMF_LAUNCH_CHECK("kl_update_h_kernel");
  return 0;
}

// ---- deferred split reduction: pass -> partial view -> update that sums the splits itself -----------------------------
int dnmf_ah_p(const void* A, int64_t lda, const void* H, int64_t ldh, int64_t m, int64_t n, int64_t k, int dtype,
              int math_mode, void* ws, int64_t ws_bytes, int64_t* view4, void* stream) {
  return run_pass(DNMF_OP_AH, A, lda, nullptr, 0, H, ldh, nullptr, 0, m, n, k, 0.0, 0, dtype, ws, ws_bytes, view4, (cudaStream_t)stream);
}

int dnmf_wta_p(const void* A, int64_t lda, const void* W, int64_t ldw, int64_t m, int64_t n, int64_t k, int dtype,
               int math_mode, void* ws, int64_t ws_bytes, int64_t* view4, void* stream) {
  return run_pass(DNMF_OP_WTA, A, lda, W, ldw, nullptr, 0, nullptr, 0, m, n, k, 0.0, 1, dtype, ws, ws_bytes, view4, (cudaStream_t)stream);
}

int dnmf_kl_uht_p(const void* A, int64_t lda, const void* W, int64_t ldw, const void* H, int64_t ldh, int64_t m, int64_t n,
                  int64_t k, double eps, int dtype, int math_mode, void* ws, int64_t ws_bytes, int64_t* view4, void* stream) {
  return run_pass(DNMF_OP_KL_UHT, A, lda, W, ldw, H, ldh, nullptr, 0, m, n, k, eps, 0, dtype, ws, ws_bytes, view4, (cudaStream_t)stream);
}

int dnmf_kl_wtu_p(const void* A, int64_t lda, const void* W, int64_t ldw, const void* H, int64_t ldh, int64_t m, int64_t n,
                  int64_t k, double eps, int dtype, int math_mode, void* ws, int64_t ws_bytes, int64_t* view4, void* stream) {
  return run_pass(DNMF_OP_KL_WTU, A, lda, W, ldw, H, ldh, nullptr, 0, m, n, k, eps, 1, dtype, ws, ws_bytes, view4, (cudaStream_t)stream);
}

#define DNMF_VIEW(view4)                                                                                         \
  DNMF_CHECK_ARG((view4) && (view4)[0] && (view4)[2] >= 1, "bad partial view");                                   \
  const float* vp_ = reinterpret_cast<const float*>((uintptr_t)(view4)[0]);                                      \
  const int64_t vld_ = (view4)[1], vss_ = (view4)[3];                                                            \
  const int vsp_ = (int)(view4)[2]

int dnmf_mu_update_w_p(void* W, int64_t ldw, const int64_t* view4, const void* G, int64_t m, int64_t k, double eps,
                       int dtype, void* stream) {
  if (int rc = check_common(m, 0, k, dtype)) return rc;
  DNMF_CHECK_ARG(W && G && dtype == DNMF_F32, "null pointer / partial views are fp32");
  DNMF_VIEW(view4);
  if (m == 0 || k == 0) return 0;
  return row_update_dispatch<float>(0, (float*)W, ldw, (const float*)W, ldw, vp_, vld_, (const float*)G, m, (int)k, (float)eps, nullptr, (cudaStream_t)stream, vsp_, vss_);
}

int dnmf_mu_update_h_p(void* H, int64_t ldh, const int64_t* view4, const void* G, int64_t k, int64_t n, double eps,
                       int clamp, int dtype, void* stream) {
  if (int rc = check_common(0, n, k, dtype)) return rc;
  DNMF_CHECK_ARG(H && G && dtype == DNMF_F32, "null pointer / partial views are fp32");
  DNMF_VIEW(view4);
  if (n == 0 || k == 0) return 0;
  // partial layout [x = column][ldp]: stride 1 between factor rows, ldp between columns
  return col_update_dispatch<float>(0, (float*)H, ldh, (const float*)H, ldh, vp_, 1, vld_, (const float*)G, (int)k, n, (float)eps, clamp, nullptr, (cudaStream_t)stream, vsp_, vss_);
}

int dnmf_kl_update_w_p(void* W, int64_t ldw, const int64_t* view4, const void* x, int64_t m, int64_t k, double eps,
                       int dtype, void* stream) {
  if (int rc = check_common(m, 0, k, dtype)) return rc;
  DNMF_CHECK_ARG(W && x && dtype == DNMF_F32, "null pointer / partial views are fp32");
  DNMF_VIEW(view4);
  if (m == 0 || k == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  kl_update_w_kernel<float><<<(unsigned)ceil_div(m * k, 256), 256, 0, st>>>((float*)W, ldw, vp_, vld_, (const float*)x, m, (int)k, (float)eps, vsp_, vss_);
  DNMF_LAUNCH_CHECK("kl_update_w_kernel<p>");
  return 0;
}

int dnmf_kl_update_h_p(void* H, int64_t ldh, const int64_t* view4, const void* x, int64_t k, int64_t n, double eps,
                       int clamp, int dtype, void* stream) {
  if (int rc = check_common(0, n, k, dtype)) return rc;
  DNMF_CHECK_ARG(H && x && dtype == DNMF_F32, "null pointer / partial views are fp32");
  DNMF_VIEW(view4);
  if (n == 0 || k == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  kl_update_h_staged_kernel<float><<<(unsigned)ceil_div(n, 64), 256, 0, st>>>((float*)H, ldh, vp_, vld_, (const float*)x, (int)k, n, (float)eps, clamp, vsp_, vss_);
  DNMF_LAUNCH_CHECK("kl_update_h_staged_kernel");
  return 0;
}
#undef DNMF_VIEW

int dnmf_clamp_min(void* X, int64_t ldx, int64_t rows, int64_t cols, double lo, int dtype, void* stream) {
  if (int rc = check_common(rows, cols, 0, dtype)) return rc;
  DNMF_CHECK_ARG(X, "null pointer");
  if (rows * cols == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  DISPATCH_T(dtype, (clamp_min_kernel<T><<<(unsigned)ceil_div(rows * cols, 256), 256, 0, st>>>((T*)X, ldx, rows, cols, (T)lo)));
  DNMF_LAUNCH_CHECK("clamp_min_kernel");
  return 0;
}

static int sum_rows_of(const void* X, int64_t ldx, int64_t rows, int64_t cols, void* out, int out_f64, int sq,
                       int dtype, void* ws, int64_t ws_bytes, void* stream) {
  // out[c] = sum over rows
  cudaStream_t st = (cudaStream_t)stream;
  const SumPlan sp = sum_plan(rows, 64, 1024);
  const int64_t need = sp.chunks * cols * (int64_t)sizeof(double);
  if (ws == nullptr || ws_bytes < need) return fail(DNMF_E_WORKSPACE, "colsum needs %lld workspace bytes, got %lld", (long long)need, (long long)ws_bytes);
  dim3 grid((unsigned)ceil_div(cols, 32), (unsigned)sp.chunks);
  DISPATCH_T(dtype, (colsum_partial_kernel<T><<<grid, 256, 0, st>>>((const T*)X, ldx, rows, cols, sp.per_chunk, (double*)ws, sq)));
  DNMF_LAUNCH_CHECK("colsum_partial_kernel");
  const unsigned g2 = (unsigned)ceil_div(cols * 32, 256);
  if (out_f64) sum_partials_kernel<double><<<g2, 256, 0, st>>>((const double*)ws, (int)sp.chunks, cols, (double*)out);
  else if (dtype == DNMF_F32) sum_partials_kernel<float><<<g2, 256, 0, st>>>((const double*)ws, (int)sp.chunks, cols, (float*)out);
  else sum_partials_kernel<double><<<g2, 256, 0, st>>>((const double*)ws, (int)sp.chunks, cols, (double*)out);
  DNMF_LAUNCH_CHECK("sum_partials_kernel");
  return 0;
}

int dnmf_colsum(const void* X, int64_t ldx, int64_t rows, int64_t cols, void* out, int dtype, void* ws,
                int64_t ws_bytes, void* stream) {
  if (int rc = check_common(rows, cols, 0, dtype)) return rc;
  DNMF_CHECK_ARG(X && out, "null pointer");
  if (cols == 0) return 0;
  return sum_rows_of(X, ldx, rows, cols, out, 0, 0, dtype, ws, ws_bytes, stream);
}

int dnmf_colsumsq(const void* X, int64_t ldx, int64_t rows, int64_t cols, void* out, int dtype, void* ws,
                  int64_t ws_bytes, void* stream) {
  if (dtype != DNMF_F32 && dtype != DNMF_F64) return fail(DNMF_E_ARG, "dtype must be DNMF_F32 or DNMF_F64");
  DNMF_CHECK_ARG(rows >= 0 && cols >= 0 && X && out, "shape / null pointer");
  if (cols == 0) return 0;
  return sum_rows_of(X, ldx, rows, cols, out, 0, 1, dtype, ws, ws_bytes, stream);
}

int64_t dnmf_colsum_workspace_bytes(int64_t rows, int64_t cols) {
  return sum_plan(rows, 64, 1024).chunks * (cols > 0 ? cols : 1) * (int64_t)sizeof(double);
}

int dnmf_rowsum(const void* X, int64_t ldx, int64_t rows, int64_t cols, void* out, int dtype, void* ws,
                int64_t ws_bytes, void* stream) {
  if (int rc = check_common(rows, cols, 0, dtype)) return rc;
  DNMF_CHECK_ARG(X && out, "null pointer");
  if (rows == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const SumPlan sp = sum_plan(cols, 2048, 256);
  const int64_t need = sp.chunks * rows * (int64_t)sizeof(double);
  if (ws == nullptr || ws_bytes < need) return fail(DNMF_E_WORKSPACE, "rowsum needs %lld workspace bytes, got %lld", (long long)need, (long long)ws_bytes);
  dim3 grid((unsigned)rows, (unsigned)sp.chunks);
  DISPATCH_T(dtype, (rowsum_partial_kernel<T><<<grid, 256, 0, st>>>((const T*)X, ldx, rows, cols, sp.per_chunk, (double*)ws, 0)));
  DNMF_LAUNCH_CHECK("rowsum_partial_kernel");
  const unsigned g2 = (unsigned)ceil_div(rows * 32, 256);
  if (dtype == DNMF_F32) sum_partials_kernel<float><<<g2, 256, 0, st>>>((const double*)ws, (int)sp.chunks, rows, (float*)out);
  else sum_partials_kernel<double><<<g2, 256, 0, st>>>((const double*)ws, (int)sp.chunks, rows, (double*)out);
  DNMF_LAUNCH_CHECK("sum_partials_kernel");
  return 0;
}

int dnmf_sqnorm(const void* X, int64_t ldx, int64_t rows, int64_t cols, double* out, int dtype, void* ws,
                int64_t ws_bytes, void* stream) {
  if (int rc = check_a(rows, cols, 0, dtype)) return rc;
  DNMF_CHECK_ARG(X && out, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (rows == 0 || cols == 0) {
    cudaError_t e = cudaMemsetAsync(out, 0, sizeof(double), st);
    return e == cudaSuccess ? 0 : cuda_fail(e, "dnmf_sqnorm memset");
  }
  // treat as rows x cols: per-row chunk partials, then one block sums them in fixed order
  const SumPlan sp = sum_plan(cols, 2048, 256);
  const int64_t nparts = sp.chunks * rows;
  const int64_t need = nparts * (int64_t)sizeof(double);
  if (ws == nullptr || ws_bytes < need) return fail(DNMF_E_WORKSPACE, "sqnorm needs %lld workspace bytes, got %lld", (long long)need, (long long)ws_bytes);
  dim3 grid((unsigned)rows, (unsigned)sp.chunks);
  DISPATCH_A(dtype, (rowsum_partial_kernel<TA><<<grid, 256, 0, st>>>((const TA*)X, ldx, rows, cols, sp.per_chunk, (double*)ws, 1)));
  DNMF_LAUNCH_CHECK("rowsum_partial_kernel<sq>");
  sum_all_kernel<<<1, 256, 0, st>>>((const double*)ws, nparts, out);
  DNMF_LAUNCH_CHECK("sum_all_kernel");
  return 0;
}

int64_t dnmf_trace_terms_workspace_bytes(void) { return (int64_t)(2 * 1024) * (int64_t)sizeof(double); }

int dnmf_trace_terms(const void* W, int64_t ldw, const void* V, int64_t ldv, int64_t m, const void* G1, const void* G2,
                     int64_t k, double* out, int64_t* slot_counter, int64_t max_slots, int dtype, void* ws, int64_t ws_bytes,
                     void* stream) {
  if (int rc = check_common(m, 0, k, dtype)) return rc;
  DNMF_CHECK_ARG(W && V && G1 && G2 && out, "null pointer");
  DNMF_CHECK_ARG(slot_counter == nullptr || max_slots >= 1, "max_slots must be >= 1 with a slot counter");
  cudaStream_t st = (cudaStream_t)stream;
  if (ws == nullptr || ws_bytes < dnmf_trace_terms_workspace_bytes())
    return fail(DNMF_E_WORKSPACE, "trace_terms needs %lld workspace bytes, got %lld", (long long)dnmf_trace_terms_workspace_bytes(), (long long)ws_bytes);
  double* P = (double*)ws;
  // <W, V>: at most 1024 blocks of whole 2048-element spans; <G1, G2>: k*k <= 4096 elements, at most 2 blocks
  const int64_t tot0 = m * k, tot1 = k * k;
  const int64_t per0 = round_up(ceil_div(tot0 > 0 ? tot0 : 1, (int64_t)1024), (int64_t)2048);
  const int64_t n0 = tot0 > 0 ? ceil_div(tot0, per0) : 0;
  const int64_t per1 = 2048;
  const int64_t n1 = tot1 > 0 ? ceil_div(tot1, per1) : 0;
  if (n0 > 0) {
    DISPATCH_T(dtype, (dot_partial_kernel<T><<<(unsigned)n0, 256, 0, st>>>((const T*)W, ldw, (const T*)V, ldv, m, (int)k, per0, P)));
    DNMF_LAUNCH_CHECK("dot_partial_kernel<W,V>");
  }
  if (n1 > 0) {
    DISPATCH_T(dtype, (dot_partial_kernel<T><<<(unsigned)n1, 256, 0, st>>>((const T*)G1, k, (const T*)G2, k, k, (int)k, per1, P + n0)));
    DNMF_LAUNCH_CHECK("dot_partial_kernel<G,G>");
  }
  trace_store_kernel<<<1, 256, 0, st>>>(P, n0, n1, out, slot_counter, max_slots);
  DNMF_LAUNCH_CHECK("trace_store_kernel");
  return 0;
}

int dnmf_normalize(void* W, int64_t ldw, int64_t m, void* H, int64_t ldh, int64_t n, int64_t k, const void* s,
                   double eps, int dtype, void* stream) {
  if (int rc = check_common(m, n, k, dtype)) return rc;
  DNMF_CHECK_ARG(W && H && s, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (m * k > 0) {
    DISPATCH_T(dtype, (normalize_w_kernel<T><<<(unsigned)ceil_div(m * k, 256), 256, 0, st>>>((T*)W, ldw, m, (int)k, (const T*)s, (T)eps)));
    DNMF_LAUNCH_CHECK("normalize_w_kernel");
  }
  if (n * k > 0) {
    DISPATCH_T(dtype, (scale_rows_kernel<T><<<(unsigned)ceil_div(n * k, 256), 256, 0, st>>>((T*)H, ldh, (int)k, n, (const T*)s)));
    DNMF_LAUNCH_CHECK("scale_rows_kernel");
  }
  return 0;
}

int dnmf_residual_sqnorm(const void* A, int64_t lda, const void* W, int64_t ldw, const void* H, int64_t ldh,
                         int64_t m, int64_t n, int64_t k, double* out, int dtype, void* ws, int64_t ws_bytes,
                         void* stream) {
  if (int rc = check_a(m, n, k, dtype)) return rc;
  DNMF_CHECK_ARG(A && W && H && out, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (m == 0 || n == 0) {
    cudaError_t e = cudaMemsetAsync(out, 0, 2 * sizeof(double), st);
    return e == cudaSuccess ? 0 : cuda_fail(e, "dnmf_residual_sqnorm memset");
  }
  const ResPlan rp = residual_plan(m, n);
  const int64_t nb = rp.col_blocks * rp.chunks;
  const int64_t need = nb * 2 * (int64_t)sizeof(double);
  if (ws == nullptr || ws_bytes < need) return fail(DNMF_E_WORKSPACE, "residual needs %lld workspace bytes, got %lld", (long long)need, (long long)ws_bytes);
  {
    int rc = 0;
    DISPATCH_A(dtype, rc = residual_dispatch<T, TA>((const TA*)A, lda, (const T*)W, ldw, (const T*)H, ldh, m, n, (int)k, rp.chunk, (unsigned)rp.col_blocks, (unsigned)rp.chunks, (double*)ws, nullptr, nullptr, st));
    if (rc) return rc;
  }
  sum_pairs_kernel<<<1, 256, 0, st>>>((const double*)ws, nb, out);
  DNMF_LAUNCH_CHECK("sum_pairs_kernel");
  return 0;
}

int dnmf_ah_residual(const void* A, int64_t lda, const void* W, int64_t ldw, const void* H, int64_t ldh, void* V,
                     int64_t ldv, int64_t m, int64_t n, int64_t k, double* out, int dtype, void* ws, int64_t ws_bytes,
                     void* stream) {
  if (int rc = check_a(m, n, k, dtype)) return rc;
  DNMF_CHECK_ARG(A && W && H && V && out, "null pointer");
  DNMF_CHECK_ARG(lda >= n && ldh >= n && ldw >= k && ldv >= k, "leading dimension too small");
  cudaStream_t st = (cudaStream_t)stream;
  if (m > 0 && n > 0 && k >= 1 && k <= 32 && tc_eligible(DNMF_OP_KL_UHT, A, lda, m, n, k, dtype)) {
    double* pairs = nullptr;
    int64_t n_pairs = 0;
    note_pass(true);
    if (int rc = tc_ah_residual_run(A, dtype, lda, (const float*)W, ldw, (const float*)H, ldh, (float*)V, ldv, m, n,
                                    (int)k, ws, ws_bytes, &pairs, &n_pairs, st))
      return rc;
    sum_pairs_kernel<<<1, 256, 0, st>>>(pairs, n_pairs, out);
    DNMF_LAUNCH_CHECK("sum_pairs_kernel");
    return 0;
  }
  if (int rc = run_pass(DNMF_OP_AH, A, lda, nullptr, 0, H, ldh, V, ldv, m, n, k, 0.0, 0, dtype, ws, ws_bytes, nullptr, st)) return rc;
  return dnmf_residual_sqnorm(A, lda, W, ldw, H, ldh, m, n, k, out, dtype, ws, ws_bytes, stream);
}

int dnmf_column_err(const void* A, int64_t lda, const void* W, int64_t ldw, const void* H, int64_t ldh, int64_t m,
                    int64_t n, int64_t k, double* num, double* den, int dtype, void* stream) {
  if (int rc = check_a(m, n, k, dtype)) return rc;
  DNMF_CHECK_ARG(A && W && H && num && den, "null pointer");
  if (n == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t chunk = round_up(m > 0 ? m : 1, kColPassBR);
  DISPATCH_A(dtype, return residual_dispatch<T, TA>((const TA*)A, lda, (const T*)W, ldw, (const T*)H, ldh, m, n, (int)k, chunk, (unsigned)ceil_div(n, kColPassThreads), 1u, nullptr, num, den, st));
  return 0;
}

int dnmf_hals_w_col(void* W, int64_t ldw, const void* V, int64_t ldv, const void* G, int64_t m, int64_t k,
                    int64_t kk, double eps, double* sq, int dtype, void* ws, int64_t ws_bytes, void* stream) {
  if (int rc = check_common(m, 0, k, dtype)) return rc;
  DNMF_CHECK_ARG(W && V && G && sq, "null pointer");
  DNMF_CHECK_ARG(kk >= 0 && kk < k, "column index out of range");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t nb = ceil_div(m > 0 ? m : 1, 256);
  const int64_t need = nb * (int64_t)sizeof(double);
  if (ws == nullptr || ws_bytes < need) return fail(DNMF_E_WORKSPACE, "hals_w_col needs %lld workspace bytes, got %lld", (long long)need, (long long)ws_bytes);
  {
    int rc = 0;
    DISPATCH_T(dtype, rc = hals_w_col_dispatch<T>((T*)W, ldw, (const T*)V, ldv, (const T*)G, m, (int)k, (int)kk, (T)eps, (double*)ws, (unsigned)nb, st));
    if (rc) return rc;
  }
  sum_all_kernel<<<1, 256, 0, st>>>((const double*)ws, nb, sq);
  DNMF_LAUNCH_CHECK("sum_all_kernel");
  return 0;
}

int dnmf_div_col(void* W, int64_t ldw, int64_t m, int64_t kk, const double* ss_sq, int dtype, void* stream) {
  if (int rc = check_common(m, 0, 0, dtype)) return rc;
  DNMF_CHECK_ARG(W && ss_sq, "null pointer");
  if (m == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  DISPATCH_T(dtype, (div_col_kernel<T><<<(unsigned)ceil_div(m, 256), 256, 0, st>>>((T*)W, ldw, m, (int)kk, ss_sq)));
  DNMF_LAUNCH_CHECK("div_col_kernel");
  return 0;
}

int dnmf_div_cols(void* W, int64_t ldw, int64_t m, int64_t k, const void* s, int dtype, void* stream) {
  if (int rc = check_common(m, 0, k, dtype)) return rc;
  DNMF_CHECK_ARG(W && s, "null pointer");
  if (m * k == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  DISPATCH_T(dtype, (div_cols_kernel<T><<<(unsigned)ceil_div(m * k, 256), 256, 0, st>>>((T*)W, ldw, m, (int)k, (const T*)s)));
  DNMF_LAUNCH_CHECK("div_cols_kernel");
  return 0;
}

int dnmf_axpby(void* out, const void* x, const void* y, double a, double b, int64_t count, int dtype, void* stream) {
  if (int rc = check_common(count, 0, 0, dtype)) return rc;
  DNMF_CHECK_ARG(out && x && y, "null pointer");
  if (count == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  DISPATCH_T(dtype, (axpby_kernel<T><<<(unsigned)ceil_div(count, 256), 256, 0, st>>>((T*)out, (const T*)x, (const T*)y, (T)a, (T)b, count)));
  DNMF_LAUNCH_CHECK("axpby_kernel");
  return 0;
}

int dnmf_nnz_counts(const void* A, int64_t lda, int64_t m, int64_t n, int64_t* row_nnz, int64_t* col_nnz, int dtype,
                    void* stream) {
  if (int rc = check_a(m, n, 0, dtype)) return rc;
  DNMF_CHECK_ARG(A && row_nnz && col_nnz, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (n > 0) {
    cudaError_t e = cudaMemsetAsync(col_nnz, 0, n * sizeof(int64_t), st);
    if (e != cudaSuccess) return cuda_fail(e, "dnmf_nnz_counts memset");
  }
  if (m == 0 || n == 0) {
    if (m > 0) cudaMemsetAsync(row_nnz, 0, m * sizeof(int64_t), st);
    return 0;
  }
  DISPATCH_A(dtype, (row_nnz_kernel<TA><<<(unsigned)ceil_div(m, 8), 256, 0, st>>>((const TA*)A, lda, m, n, (long long*)row_nnz)));
  DNMF_LAUNCH_CHECK("row_nnz_kernel");
  const SumPlan sp = sum_plan(m, 256, 256);
  dim3 grid((unsigned)ceil_div(n, 256), (unsigned)sp.chunks);
  DISPATCH_A(dtype, (col_nnz_kernel<TA><<<grid, 256, 0, st>>>((const TA*)A, lda, m, n, sp.per_chunk, (unsigned long long*)col_nnz)));
  DNMF_LAUNCH_CHECK("col_nnz_kernel");
  return 0;
}

int dnmf_compact(const void* A, int64_t lda, const int64_t* row_idx, int64_t mr, const int64_t* col_idx, int64_t nc,
                 void* out, int64_t ldo, int dtype, void* stream) {
  if (int rc = check_a(mr, nc, 0, dtype)) return rc;
  if (mr * nc == 0) return 0;
  DNMF_CHECK_ARG(A && row_idx && col_idx && out, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  DISPATCH_A(dtype, (compact_kernel<TA><<<(unsigned)ceil_div(mr * nc, 256), 256, 0, st>>>((const TA*)A, lda, (const long long*)row_idx, mr, (const long long*)col_idx, nc, (TA*)out, ldo)));
  DNMF_LAUNCH_CHECK("compact_kernel");
  return 0;
}

int dnmf_scatter_rows(const void* X, int64_t ldx, const int64_t* row_idx, int64_t mr, int64_t cols, double* out,
                      int64_t ldo, int dtype, void* stream) {
  if (int rc = check_common(mr, cols, 0, dtype)) return rc;
  if (mr * cols == 0) return 0;
  DNMF_CHECK_ARG(X && row_idx && out, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  DISPATCH_T(dtype, (scatter_kernel<T, true><<<(unsigned)ceil_div(mr * cols, 256), 256, 0, st>>>((const T*)X, ldx, (const long long*)row_idx, mr, cols, out, ldo)));
  DNMF_LAUNCH_CHECK("scatter_kernel<rows>");
  return 0;
}

int dnmf_scatter_cols(const void* X, int64_t ldx, const int64_t* col_idx, int64_t nc, int64_t rows, double* out,
                      int64_t ldo, int dtype, void* stream) {
  if (int rc = check_common(rows, nc, 0, dtype)) return rc;
  if (rows * nc == 0) return 0;
  DNMF_CHECK_ARG(X && col_idx && out, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  DISPATCH_T(dtype, (scatter_kernel<T, false><<<(unsigned)ceil_div(rows * nc, 256), 256, 0, st>>>((const T*)X, ldx, (const long long*)col_idx, rows, nc, out, ldo)));
  DNMF_LAUNCH_CHECK("scatter_kernel<cols>");
  return 0;
}

int dnmf_perturb_uniform(const void* A, const void* U, void* X, int64_t count, double noise_var, int dtype,
                         void* stream) {
  if (int rc = check_common(count, 0, 0, dtype)) return rc;
  if (count == 0) return 0;
  DNMF_CHECK_ARG(A && U && X, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  DISPATCH_T(dtype, (perturb_uniform_kernel<T><<<(unsigned)ceil_div(count, 256), 256, 0, st>>>((const T*)A, (const T*)U, (T*)X, count, (T)(2 * noise_var), (T)noise_var)));
  DNMF_LAUNCH_CHECK("perturb_uniform_kernel");
  return 0;
}

}  // extern "C"
