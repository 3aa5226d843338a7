/*
 * libdnmf — C-ABI of the B200-native pyDNMFk update loop.
 *
 * The reference (lanl/pyDNMFk) is pure Python: it has no FFI layer, its
 * "operator API" for the hot path is the set of numpy expressions inside
 * pyDNMFk/dist_nmf.py and pyDNMFk/pyDNMF.py.  Each entry point below replaces
 * one of those expressions (cited as file:line, paths relative to the
 * reference root) and is what a maintainer would bind with ctypes from those
 * exact lines (see INTEGRATION.md).
 *
 * Conventions
 *   - every function returns int: 0 = OK, >0 = cudaError_t, <0 = argument error
 *     (DNMF_E_*); dnmf_last_error() gives the thread-local message.
 *   - all matrix pointers are DEVICE pointers to C-contiguous row-major data
 *     with an explicit leading dimension (elements, not bytes).
 *   - dtype: DNMF_F32 / DNMF_F64 (the reference's --precision float32/float64).
 *   - math_mode: DNMF_MATH_ACCURATE = fp32-accurate results (FFMA, or 3xTF32
 *     split on the tcgen05 path).  DNMF_MATH_TF32 (single-pass TF32) is
 *     reserved: this build computes DNMF_MATH_ACCURATE results for both values
 *     (single-pass TF32 cannot meet the parity tolerance of the update loop).
 *   - stream: a cudaStream_t passed as void* (0 = legacy default stream).
 *   - the library never allocates persistent device memory; scratch space is
 *     passed in (`ws`, `ws_bytes`; size from dnmf_workspace_bytes()).
 *   - all reductions are two-stage with a fixed order: results are
 *     run-to-run deterministic.
 */
#ifndef DNMF_H_
#define DNMF_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DNMF_F32 0
#define DNMF_F64 1
#define DNMF_I64 2   /* collectives only (prune counts, utils.py:122-126) */
/* 16-bit storage of the data shard A: A is fp16 / bf16, every other operand (factors, eps, partials) and every output
 * is fp32 (dnmf_compact: 16-bit in, 16-bit out).  Only the entry points that read A accept these codes:
 *   dnmf_workspace_bytes, dnmf_ah[_p], dnmf_wta[_p], dnmf_kl_uht[_p], dnmf_kl_wtu[_p], dnmf_residual_sqnorm,
 *   dnmf_ah_residual, dnmf_column_err, dnmf_sqnorm (for ||A||^2), dnmf_nnz_counts, dnmf_compact.
 * Every other entry point rejects them with DNMF_E_ARG.  dnmf_ah / dnmf_wta (and their _p forms) run on the tcgen05
 * kind::f16 kernel (dnmf_tc16.cu) for 16-byte aligned shards with lda % 8 == 0, >= 2^20 elements and k <= 64; the
 * KL contractions and everything else stream the 16-bit shard through the generic CUDA-core kernels.
 * (2 is DNMF_I64, which the collectives accept, so the 16-bit codes start at 3.) */
#define DNMF_A_F16 3
#define DNMF_A_BF16 4

#define DNMF_MATH_ACCURATE 0
#define DNMF_MATH_TF32 1

#define DNMF_E_ARG (-1)       /* bad argument (null pointer, negative size, bad dtype) */
#define DNMF_E_UNSUPPORTED (-2) /* k > DNMF_MAX_K or unsupported combination */
#define DNMF_E_WORKSPACE (-3) /* workspace too small */
#define DNMF_E_NOGPU (-4)     /* no sm_100 device */
#define DNMF_E_COMM (-5)      /* NCCL / peer-memory failure */

#define DNMF_MAX_K 64

/* op ids for dnmf_workspace_bytes */
#define DNMF_OP_AH 0
#define DNMF_OP_WTA 1
#define DNMF_OP_KL_UHT 2
#define DNMF_OP_KL_WTU 3
#define DNMF_OP_GRAM 4
#define DNMF_OP_RESIDUAL 5
#define DNMF_OP_SUMS 6
#define DNMF_OP_NNZ 7
#define DNMF_OP_AH_RESIDUAL 8

const char* dnmf_version(void);
const char* dnmf_last_error(void);
/* which code path the last dnmf_ah/dnmf_wta/dnmf_kl_* call on this thread took:
 * 0 = generic CUDA-core kernel, 1 = tcgen05 (TMA + UMMA + TMEM) kernel */
int dnmf_last_path(void);
/* A-streaming passes (dnmf_ah / dnmf_wta / dnmf_kl_*) issued on this thread since the last reset:
 * which = 1: through the tcgen05 kernels, which = 0: through the generic CUDA-core kernels (parity tests assert
 * that the large cases never touch the generic ones) */
int64_t dnmf_pass_count(int which, int reset);
/* number of kernels launched by this library on this thread since the last reset */
int64_t dnmf_launch_count(int reset);
int dnmf_device_info(int* sm_count, int* cc_major, int* cc_minor);
/* 0 = auto (tcgen05 when eligible), 1 = force generic kernels */
int dnmf_set_force_generic(int on);
/* smallest shard (m*n elements) routed to the tcgen05 path; default 2^20, tests lower it */
int dnmf_set_tc_min_elems(int64_t elems);
/* 1: dnmf_residual_sqnorm uses the tcgen05 pipeline (fp32, k <= 32) instead of the CUDA-core kernel; default 0
 * (or the DNMF_TC_RESIDUAL environment variable) */
int dnmf_set_tc_residual(int on);
/* debug: timing-ablation bits of the tcgen05 kernels (tools/prof_tc.py); non-zero values give WRONG results */
int dnmf_set_tc_debug(int flags);
/* debug/profiling: device buffer of [n_sm][16] uint64 cycle counters filled by the tcgen05 kernels (NULL = off) */
int dnmf_set_tc_profile(void* device_buf);

int64_t dnmf_workspace_bytes(int op, int64_t m, int64_t n, int64_t k, int dtype);

/* ---- A-streaming contractions ------------------------------------------------
 * dnmf_ah:  V[m x k] = A[m x n] * H[k x n]^T
 *   replaces np.matmul(A_ij, H_j.T): dist_nmf.py:198 (2-D AH_glob), :705 via :730/:887/:967/:1023 (1-D global_mm)
 * dnmf_wta: Y[k x n] = W[m x k]^T * A[m x n]      (transposed_out: writes Y^T [n x k], the
 *   Reduce_scatter layout of dist_nmf.py:167-169)
 *   replaces np.matmul(W_i.T, A_ij): dist_nmf.py:166, :705 via :749/:909/:1019
 */
int dnmf_ah(const void* A, int64_t lda, const void* H, int64_t ldh, void* V, int64_t ldv,
            int64_t m, int64_t n, int64_t k, int dtype, int math_mode,
            void* ws, int64_t ws_bytes, void* stream);
int dnmf_wta(const void* A, int64_t lda, const void* W, int64_t ldw, void* Y, int64_t ldy,
             int64_t m, int64_t n, int64_t k, int transposed_out, int dtype, int math_mode,
             void* ws, int64_t ws_bytes, void* stream);

/* ---- fused KL contractions (W H is never materialised) ----------------------
 * dnmf_kl_uht: V[m x k] = (A / (W H + eps)) * H^T     dist_nmf.py:338-339 (UHT_glob), :806,:810 (glob_UX axis=0)
 * dnmf_kl_wtu: Y[k x n] = W^T * (A / (W H + eps))     dist_nmf.py:312-313 (WTU_glob), :806,:808 (glob_UX axis=1)
 */
int dnmf_kl_uht(const void* A, int64_t lda, const void* W, int64_t ldw, const void* H, int64_t ldh,
                void* V, int64_t ldv, int64_t m, int64_t n, int64_t k, double eps,
                int dtype, int math_mode, void* ws, int64_t ws_bytes, void* stream);
int dnmf_kl_wtu(const void* A, int64_t lda, const void* W, int64_t ldw, const void* H, int64_t ldh,
                void* Y, int64_t ldy, int64_t m, int64_t n, int64_t k, double eps, int transposed_out,
                int dtype, int math_mode, void* ws, int64_t ws_bytes, void* stream);

/* ---- k x k Gram -----------------------------------------------------------------
 * trans = 0: X is [rows x k], G = X^T X    (W^T W: dist_nmf.py:113 via :222, :679 via :748)
 * trans = 1: X is [k x rows], G = X X^T    (H H^T: dist_nmf.py:113 via :242, :679 via :729)
 */
int dnmf_gram(const void* X, int64_t ldx, int64_t rows, int64_t k, int trans, void* G,
              int dtype, void* ws, int64_t ws_bytes, void* stream);

/* ---- multiplicative updates -------------------------------------------------------
 * dnmf_mu_update_w: W *= V / (W G + eps)            dist_nmf.py:244-245, :731-732
 * dnmf_mu_update_h: H *= Y / (H^T G + eps)^T        dist_nmf.py:224-225, :750-751
 *   Y element (kk, c) is read at Y[kk*y_stride_k + c*y_stride_c]  (so a Y^T shard can be used in place)
 * dnmf_kl_update_w: W *= V / (x[j] + eps)           dist_nmf.py:366,369, :828,830  (x = row sums of H)
 * dnmf_kl_update_h: H *= Y / (x[kk] + eps)          dist_nmf.py:386,389, :847,849  (x = column sums of W)
 * clamp != 0 fuses the every-10th-iteration np.maximum(., eps) of pyDNMF.py:155-157,170-172 (H side only:
 *   the reference clamps W after the H half-step has consumed the un-clamped W).
 */
int dnmf_mu_update_w(void* W, int64_t ldw, const void* V, int64_t ldv, const void* G,
                     int64_t m, int64_t k, double eps, int dtype, void* stream);
int dnmf_mu_update_h(void* H, int64_t ldh, const void* Y, int64_t y_stride_k, int64_t y_stride_c,
                     const void* G, int64_t k, int64_t n, double eps, int clamp, int dtype, void* stream);
int dnmf_kl_update_w(void* W, int64_t ldw, const void* V, int64_t ldv, const void* x,
                     int64_t m, int64_t k, double eps, int dtype, void* stream);
int dnmf_kl_update_h(void* H, int64_t ldh, const void* Y, int64_t y_stride_k, int64_t y_stride_c,
                     const void* x, int64_t k, int64_t n, double eps, int clamp, int dtype, void* stream);

/* X = max(X, lo) over a [rows x cols] matrix            pyDNMF.py:155-157,170-172 */
int dnmf_clamp_min(void* X, int64_t ldx, int64_t rows, int64_t cols, double lo, int dtype, void* stream);

/* ---- small reductions ---------------------------------------------------------------
 * dnmf_colsum: out[j] = sum_i X[i][j]   (W.sum(axis=0): dist_nmf.py:347,:793; pyDNMF.py:187; dist_nmf.py:539,:1006)
 * dnmf_rowsum: out[i] = sum_j X[i][j]   (H.sum(axis=1): dist_nmf.py:347,:793)
 * dnmf_sqnorm: out[0] = sum X^2 as float64 (np.linalg.norm(X)**2: dist_nmf.py:477-478,:942-943; utils.py:388)
 */
int dnmf_colsum(const void* X, int64_t ldx, int64_t rows, int64_t cols, void* out,
                int dtype, void* ws, int64_t ws_bytes, void* stream);
int dnmf_rowsum(const void* X, int64_t ldx, int64_t rows, int64_t cols, void* out,
                int dtype, void* ws, int64_t ws_bytes, void* stream);
int dnmf_sqnorm(const void* X, int64_t ldx, int64_t rows, int64_t cols, double* out,
                int dtype, void* ws, int64_t ws_bytes, void* stream);

/* W /= (s + eps) ; H *= s^T                          pyDNMF.py:192-193 */
int dnmf_normalize(void* W, int64_t ldw, int64_t m, void* H, int64_t ldh, int64_t n, int64_t k,
                   const void* s, double eps, int dtype, void* stream);

/* The two factor-sized inner products of the trace identity
 *     ||A - W H||_F^2 = ||A||_F^2 - 2 <W, A H^T> + <W^T W, H H^T>
 * (the per-iteration error monitor; the returned recon_err stays the direct residual, see DESIGN.md):
 *   out[2 s]     = sum_ij W[i][j] V[i][j]     W, V = A H^T: this rank's [m x k] rows (sum over ranks by the caller)
 *   out[2 s + 1] = sum_ij G1[i][j] G2[i][j]   G1 = W^T W, G2 = H H^T: the global [k x k] Grams
 * as float64, two-stage fixed-order reductions.  s = 0, or -- with `slot_counter` -- the int64 read from device memory,
 * which the call then advances (samples beyond max_slots are dropped): a CUDA-graph replay of the step appends to a
 * history.  Replaces the A-sized temporary A - W_i @ H_j of pyDNMF.py:208-209 for monitoring; the operands are what
 * dist_nmf.py:729-732 / :242-245 has at hand anyway (H H^T, A H^T) plus the W^T W of the preceding H half-step (:748). */
int64_t dnmf_trace_terms_workspace_bytes(void);
int dnmf_trace_terms(const void* W, int64_t ldw, const void* V, int64_t ldv, int64_t m,
                     const void* G1, const void* G2, int64_t k, double* out, int64_t* slot_counter,
                     int64_t max_slots, int dtype, void* ws, int64_t ws_bytes, void* stream);

/* out[0] = ||A - W H||_F^2, out[1] = ||A||_F^2 (float64), one pass over A, no m x n temporary
 *   replaces pyDNMF.py:208-209,215 and dist_nmf.py:556,:1024 */
int dnmf_residual_sqnorm(const void* A, int64_t lda, const void* W, int64_t ldw, const void* H, int64_t ldh,
                         int64_t m, int64_t n, int64_t k, double* out, int dtype,
                         void* ws, int64_t ws_bytes, void* stream);
/* per-column ||A[:,q] - (W H)[:,q]||^2 and ||A[:,q]||^2 (float64 [n] each)   pyDNMF.py:231-233 */
int dnmf_column_err(const void* A, int64_t lda, const void* W, int64_t ldw, const void* H, int64_t ldh,
                    int64_t m, int64_t n, int64_t k, double* num, double* den, int dtype, void* stream);

/* ---- HALS column sweeps ------------------------------------------------------------
 * dnmf_hals_w_col: t = W[:,kk]*G[kk,kk] + V[:,kk] - W G[:,kk]; W[:,kk] = max(t, eps); sq[0] = sum W[:,kk]^2 (float64)
 *                                                     dist_nmf.py:428-429, :889-890 ; utils.py:388
 * dnmf_scale_col:  W[:,kk] *= 1/ss  (as a division)   dist_nmf.py:431-432, :892-893
 * dnmf_hals_h:     for kk: H[kk,:] = max(H[kk,:] + Y[kk,:] - G[kk,:] H, eps)   dist_nmf.py:450-452, :911-913
 */
int dnmf_hals_w_col(void* W, int64_t ldw, const void* V, int64_t ldv, const void* G, int64_t m, int64_t k,
                    int64_t kk, double eps, double* sq, int dtype, void* ws, int64_t ws_bytes, void* stream);
int dnmf_div_col(void* W, int64_t ldw, int64_t m, int64_t kk, const double* ss_sq, int dtype, void* stream);
int dnmf_hals_h(void* H, int64_t ldh, const void* Y, int64_t y_stride_k, int64_t y_stride_c, const void* G,
                int64_t k, int64_t n, double eps, int dtype, void* stream);

/* ---- BCD building blocks -----------------------------------------------------------
 * dnmf_bcd_pg_w: W = max(0, Wm - (Wm G - V) / L)      dist_nmf.py:535-537, :1002-1004
 * dnmf_bcd_pg_h: H = max(0, Hm - (G Hm - Y) / L)      dist_nmf.py:549-552, :1018-1021
 * dnmf_div_cols: W[:,j] /= s[j]                        dist_nmf.py:542, :1011
 * dnmf_axpby:    out = a*x + b*y  (extrapolation Wm = W + ww (W - W_old), scaling)  dist_nmf.py:574-575, :1042-1043, :493-494
 */
int dnmf_bcd_pg_w(void* W, int64_t ldw, const void* Wm, int64_t ldwm, const void* V, int64_t ldv, const void* G,
                  int64_t m, int64_t k, double L, int dtype, void* stream);
int dnmf_bcd_pg_h(void* H, int64_t ldh, const void* Hm, int64_t ldhm, const void* Y, int64_t y_stride_k,
                  int64_t y_stride_c, const void* G, int64_t k, int64_t n, double L, int dtype, void* stream);
int dnmf_div_cols(void* W, int64_t ldw, int64_t m, int64_t k, const void* s, int dtype, void* stream);
int dnmf_axpby(void* out, const void* x, const void* y, double a, double b, int64_t count, int dtype, void* stream);

/* ---- shard ops: zero row/column pruning and perturbation ---------------------------
 * dnmf_nnz_counts: row_nnz[i] = #(A[i,:] != 0), col_nnz[j] = #(A[:,j] != 0)  (int64)   utils.py:119-120
 * dnmf_compact:    out = A[np.ix_(rowmask, colmask)] given the kept indices             utils.py:155
 * dnmf_scatter_rows / dnmf_scatter_cols: float64 zero-filled un-prune                   utils.py:194-199
 * dnmf_perturb_uniform: X = A * (1 + nv + 2 nv u)  with u supplied (host RNG order kept) pyDNMFk.py:42-44
 */
int dnmf_nnz_counts(const void* A, int64_t lda, int64_t m, int64_t n, int64_t* row_nnz, int64_t* col_nnz,
                    int dtype, void* stream);
int dnmf_compact(const void* A, int64_t lda, const int64_t* row_idx, int64_t mr, const int64_t* col_idx, int64_t nc,
                 void* out, int64_t ldo, int dtype, void* stream);
int dnmf_scatter_rows(const void* X, int64_t ldx, const int64_t* row_idx, int64_t mr, int64_t cols,
                      double* out, int64_t ldo, int dtype, void* stream);
int dnmf_scatter_cols(const void* X, int64_t ldx, const int64_t* col_idx, int64_t nc, int64_t rows,
                      double* out, int64_t ldo, int dtype, void* stream);
int dnmf_perturb_uniform(const void* A, const void* U, void* X, int64_t count, double noise_var,
                         int dtype, void* stream);

/* ==== NMFk-level rows (SURVEY.md section 8f) =======================================================
 * Ensemble tensors are C-contiguous: W_all [m_loc, k, P], H_all [k, n_loc, P] (P = perturbations).
 *
 * dnmf_colsumsq: out[j] = sum_i X[i][j]^2 (wide matrices, e.g. the m x (k P) view of W_all)
 *                                             dist_clustering.py:33 (W_all*W_all).sum(axis=0), :120 (centroids**2).sum(0)
 * dnmf_colsum_workspace_bytes: scratch of dnmf_colsum / dnmf_colsumsq for a rows x cols input
 * dnmf_scale_groups: X[i0,i1,i2] op= f(s[i0*s0 + i1*s1 + i2*s2]) on a contiguous [d0,d1,d2] tensor;
 *   mode 0: *= s   1: /= s   2: /= sqrt(s+eps)   3: *= sqrt(s+eps)   4: /= (s+eps)   5: *= (s+eps)
 *                                             dist_clustering.py:36-39, :123-125 ; dist_svd.py:72-77
 * dnmf_greedy_lsa: the greedy assignment + change_order of dist_clustering.py:49-69 for all P perturbations at
 *   once; D [k, k*P] holds centroid-feature similarities at D[r*ldd + c*P + p]; order[p*k + r] = c (int32)
 * dnmf_permute_groups: out[.., r, .., p] = in[.., src(p, r), .., p] along axis 0 or 1 of [d0, d1, P];
 *   sequential = 0: src = order[p][r], the gather W_sub[:, j] of dist_clustering.py:81;
 *   sequential = 1: the outcome of `for r: X[r] = X[order[p][r]]` done in place, which is what the list-of-views
 *   assignment to H_all[:, :, p] (dist_clustering.py:116) amounts to under numpy >= 1.20 (rows already overwritten
 *   are read back: src(r) = j[r] if j[r] >= r else src(j[r]))
 * dnmf_median_last: med[row] = np.median(X[row, :P]); mad[row] = median(|X[row,:] - med[row]|) (either may be NULL)
 *                                             dist_clustering.py:118 ; :41-47 (mad, flag=1) ; pyDNMFk.py:241
 * dnmf_silhouettes: out[kk*P + n] (float64) from the (k P) x (k P) cosine Gram   dist_clustering.py:146-159
 */
int dnmf_colsumsq(const void* X, int64_t ldx, int64_t rows, int64_t cols, void* out,
                  int dtype, void* ws, int64_t ws_bytes, void* stream);
int64_t dnmf_colsum_workspace_bytes(int64_t rows, int64_t cols);
int dnmf_scale_groups(void* X, int64_t d0, int64_t d1, int64_t d2, const void* s, int64_t s0, int64_t s1, int64_t s2,
                      int mode, double eps, int dtype, void* stream);
int dnmf_greedy_lsa(const void* D, int64_t ldd, int64_t k, int64_t P, int32_t* order, int dtype, void* stream);
int dnmf_permute_groups(const void* in, void* out, int64_t d0, int64_t d1, int64_t P, int axis, const int32_t* order,
                        int sequential, int dtype, void* stream);
int dnmf_median_last(const void* X, int64_t rows, int64_t P, void* med, void* mad, int dtype, void* stream);
int dnmf_silhouettes(const void* G, int64_t ldg, int64_t k, int64_t P, double* out, int dtype, void* stream);

/* ---- nnsvd initialisation (dist_svd.py) ---------------------------------------------------------
 * dnmf_rank1_sub:  M = (T)(M - sigma (u v^T)) with float64 u, v, sigma[0] (deflation)         dist_svd.py:160-162
 * dnmf_matvec_f64: y = A x (trans = 0) or y = A^T x (trans = 1); A of `dtype`, x / y / accumulation float64
 *                  (B @ currV: dist_svd.py:121 ; A @ v, A.T @ u: :166,:172)
 * dnmf_power_normalize: v_out = y / ||y||, r[0] = <v_out, v_last>                              dist_svd.py:123-124
 * dnmf_div_store:  dst[i*stride] = src[i] / sqrt(sq[0])    (u = u_unnorm / sig)                dist_svd.py:168,:174
 * dnmf_posneg_colsumsq: out[j] = sum max(X[:,j],0)^2, out[k+j] = sum max(-X[:,j],0)^2          dist_svd.py:222-235
 * dnmf_nnsvd_pick: out = pos[j] ? cp[j] max(X,0) / dp[j] : cn[j] max(-X,0) / dn[j], coef = [cp|dp|cn|dn]   :241-242
 */
int dnmf_rank1_sub(void* M, int64_t ldm, int64_t rows, int64_t cols, const double* u, const double* v, const double* sigma,
                   int dtype, void* stream);
int64_t dnmf_matvec_workspace_bytes(int64_t rows, int64_t cols, int trans);
int dnmf_matvec_f64(const void* A, int64_t lda, int64_t rows, int64_t cols, const double* x, double* y, int trans,
                    int dtype, void* ws, int64_t ws_bytes, void* stream);
int dnmf_power_normalize(const double* y, const double* v_last, double* v_out, double* r, int64_t d, void* stream);
/* the whole loop `while True: v = normalize(B @ v); if |<v, v_prev>| > thr: break` (dist_svd.py:117-134) in ONE launch
 * for a small Gram matrix B [d x d], d <= 512 (same arithmetic as dnmf_matvec_f64 + dnmf_power_normalize per step);
 * thr = 1 - eps as the reference computes it; cmp_f32 = 1 when that value is a float32 scalar (fp32 data): numpy then
 * compares in float32, which stops later than the float64 comparison would;
 * v: start vector in, result out; scratch: 2 d doubles; iters_out (device int, may be NULL): steps taken */
int dnmf_power_iterate(const void* B, int64_t ldb, int64_t d, double* v, double thr, int cmp_f32, int max_iter,
                       double* scratch, int* iters_out, int dtype, void* stream);
int dnmf_div_store(const double* src, const double* sq, double* dst, int64_t n, int64_t stride, void* stream);
int dnmf_posneg_colsumsq(const double* X, int64_t ldx, int64_t rows, int64_t k, double* out, void* stream);
int dnmf_nnsvd_pick(const double* X, int64_t ldx, int64_t rows, int64_t k, const double* coef, const int32_t* pos,
                    double* out, int64_t ldo, int transpose_out, void* stream);

/* ---- whole-fit on-chip multiplicative updates for shards that fit in shared memory ------------------------------
 * dnmf_mu_fit_resident: `batch` independent fits in ONE launch, each on one CTA (shards up to ~200 KB) or on a
 *   thread-block cluster of 2..16 CTAs (shards of a few MB: row blocks of A and W per CTA, H replicated, the
 *   W^T A / W^T W partials summed through distributed shared memory).  A_b, W_b, H_b (device arrays of `batch`
 *   device pointers; A_b [m x n] with leading dimension lda, W_b [m x k], H_b [k x n] contiguous) are loaded into
 *   shared memory and iterations i = it_begin .. it_end-1 of PyNMF.fit's loop body run on chip:
 *   update() (kl = 0: dist_nmf.py:715-771 FRO-MU, kl = 1: :803-869 KL-MU; W half-step only if w_update) followed by
 *   the clamp max(., eps) when i % 10 == 0 (pyDNMF.py:151-157,168-172).  The batch is the NMFk perturbation
 *   ensemble (pyDNMFk.py:226-233).  Single-process grids only (no collectives inside).
 * dnmf_mu_fit_resident_smem_bytes: shared memory per CTA one fit needs, or -1 if it does not fit / is not supported.
 * dnmf_mu_fit_resident_cluster_size: CTAs per fit for this shape (1, or the cluster size 2..16; 0 = unsupported).
 */
int64_t dnmf_mu_fit_resident_smem_bytes(int64_t m, int64_t n, int64_t k, int kl, int dtype);
int dnmf_mu_fit_resident_cluster_size(int64_t m, int64_t n, int64_t k, int kl, int dtype);
int dnmf_mu_fit_resident(const void* const* A_ptrs, int64_t lda, void* const* W_ptrs, void* const* H_ptrs, int64_t batch,
                         int64_t m, int64_t n, int64_t k, int kl, int w_update, int64_t it_begin, int64_t it_end,
                         double eps, int dtype, void* stream);

/* V = A H^T and out[0] = ||A - W H||_F^2, out[1] = ||A||_F^2 in ONE pass over A (fp32, k <= 32: tcgen05 kernel that
 * recomputes each W H tile on the tensor cores like the KL path; otherwise the two separate passes): the BCD iteration's
 * dist_nmf.py:1023 (A H^T) and :1024 (objective), which the reference runs as two passes plus an m x n temporary. */
int dnmf_ah_residual(const void* A, int64_t lda, const void* W, int64_t ldw, const void* H, int64_t ldh, void* V,
                     int64_t ldv, int64_t m, int64_t n, int64_t k, double* out, int dtype, void* ws, int64_t ws_bytes,
                     void* stream);

/* ---- update fused with the pass's split reduction ("fused epilogue") ------------------------------------------------
 * An A-streaming pass is split over the reduced dimension (deterministic split-K); dnmf_ah / dnmf_wta / dnmf_kl_* end with
 * a launch that sums the per-split partials into V / Y, which the update kernel then reads back.  The _p variants leave
 * the partials in the workspace and describe them in view4 = {device pointer of P[split][x][ldp], ldp, splits,
 * split stride (elements)}; the _p updates (and the row grid's exchange) take that view and add the splits themselves in
 * the same order: bit-identical results, one launch and one factor-sized HBM round trip less per half-step
 * (dist_nmf.py:730-732, :749-751, :806-830, :808-849 as pass + update = 2 launches).
 * The pass variants return DNMF_E_UNSUPPORTED, without side effects, when the call is not served by the tcgen05 path
 * (fp64, small or unaligned shards): the caller then uses the plain entry points.  fp32 A or a 16-bit A (DNMF_A_*) for
 * the passes; the partials and the _p updates are fp32 (dtype DNMF_F32).
 * The view is valid until the next call that uses the same workspace. */
int dnmf_ah_p(const void* A, int64_t lda, const void* H, int64_t ldh, int64_t m, int64_t n, int64_t k, int dtype,
              int math_mode, void* ws, int64_t ws_bytes, int64_t* view4, void* stream);
int dnmf_wta_p(const void* A, int64_t lda, const void* W, int64_t ldw, int64_t m, int64_t n, int64_t k, int dtype,
               int math_mode, void* ws, int64_t ws_bytes, int64_t* view4, void* stream);
int dnmf_kl_uht_p(const void* A, int64_t lda, const void* W, int64_t ldw, const void* H, int64_t ldh, int64_t m, int64_t n,
                  int64_t k, double eps, int dtype, int math_mode, void* ws, int64_t ws_bytes, int64_t* view4, void* stream);
int dnmf_kl_wtu_p(const void* A, int64_t lda, const void* W, int64_t ldw, const void* H, int64_t ldh, int64_t m, int64_t n,
                  int64_t k, double eps, int dtype, int math_mode, void* ws, int64_t ws_bytes, int64_t* view4, void* stream);
int dnmf_mu_update_w_p(void* W, int64_t ldw, const int64_t* view4, const void* G, int64_t m, int64_t k, double eps,
                       int dtype, void* stream);
int dnmf_mu_update_h_p(void* H, int64_t ldh, const int64_t* view4, const void* G, int64_t k, int64_t n, double eps,
                       int clamp, int dtype, void* stream);
int dnmf_kl_update_w_p(void* W, int64_t ldw, const int64_t* view4, const void* x, int64_t m, int64_t k, double eps,
                       int dtype, void* stream);
int dnmf_kl_update_h_p(void* H, int64_t ldh, const int64_t* view4, const void* x, int64_t k, int64_t n, double eps,
                       int clamp, int dtype, void* stream);

/* ---- FRO-BCD with its scalars on the device (dist_nmf.py:996-1047): the same arithmetic as dnmf_bcd_pg_w / _h with the
 * Lipschitz bound read from device memory, and the iteration's control state (Lipschitz bounds, objective, momentum
 * weights, accept / restore decision) kept in a 16-double device vector:
 *   state[0] L_W  [1] L_W old  [2] L_H  [3] L_H old  [4] obj_old  [5] t_old  [6] accept  [7] ww  [8] wh  [9] obj
 *   [10] rw  [11] restores so far
 * dnmf_bcd_state phase 0: in[0] = ||A||^2 (init, :951-969); 1: in[0] = ||H H^T||_F^2 (:1000-1001); 2: in[0] =
 * ||W^T W||_F^2 (:1016-1017); 3: in[0] = ||A - W H||_F^2 -> obj, t, ww, wh, accept (:1024-1047).
 * dnmf_bcd_advance (which 0 = W with ww, 1 = H with wh): accept -> Xm = X + w (X - X_old), X_old = X; restore -> Xm = X_old.
 * dnmf_bcd_keep: accept -> kept = cur; restore -> cur = kept  (H H^T and A H^T of the last accepted H, instead of the
 * reference's recomputation :1034-1035, which costs another pass over A). */
int dnmf_bcd_pg_w_dev(void* W, int64_t ldw, const void* Wm, int64_t ldwm, const void* V, int64_t ldv, const void* G,
                      int64_t m, int64_t k, const double* L_dev, int dtype, void* stream);
int dnmf_bcd_pg_h_dev(void* H, int64_t ldh, const void* Hm, int64_t ldhm, const void* Y, int64_t y_stride_k,
                      int64_t y_stride_c, const void* G, int64_t k, int64_t n, const double* L_dev, int dtype, void* stream);
int dnmf_bcd_state(int phase, double* state, const double* in, void* stream);
int dnmf_bcd_advance(const void* X, void* Xm, void* X_old, int64_t count, const double* state, int which, int dtype,
                     void* stream);
int dnmf_bcd_keep(void* cur, void* kept, int64_t count, const double* state, int dtype, void* stream);

/* ---- communicators: dist_comm.py:16-56 (MPI_comm: world + row / column sub-communicators) as NCCL communicators
 * owned by this library, one process per GPU.  The 128-byte id is created on one rank (dnmf_comm_unique_id) and
 * handed to the others by the launcher's own plumbing (torch.distributed object broadcast, a file, MPI ...).
 * Collectives are SUM reductions / plain copies on DEVICE buffers, in place where MPI's allreduce is
 * (dist_nmf.py:114, :681, :707, utils.py:122-126), enqueued on `stream` (capturable into a CUDA graph).
 * dtype: DNMF_F32 / DNMF_F64 / DNMF_I64.  Counts are elements.
 *   dnmf_allreduce       comm.allreduce(x)                              dist_nmf.py:114,681,707,799; pyDNMF.py:217
 *   dnmf_allgather       comm.allgather(x) of equal shards, rank order  dist_nmf.py:163,195,284,288
 *   dnmf_reduce_scatter  comm.Reduce_scatter(send, recv, op=SUM)        dist_nmf.py:169,202,315,341
 *   dnmf_bcast           comm.bcast(x, root)                            pyDNMF.py:121,129
 *   dnmf_comm_split      Cart_sub / Split (color, key)                  dist_comm.py:34,48
 */
int dnmf_comm_load(const char* libnccl_path);      /* optional: where libnccl.so.2 lives (default: already-loaded copy) */
int dnmf_comm_nccl_version(int* version);
int dnmf_comm_unique_id(void* id_out_128);
int dnmf_comm_init_rank(const void* id_128, int nranks, int rank, void** comm_out);   /* uses the current device */
int dnmf_comm_split(void* comm, int color, int key, void** comm_out);                /* color < 0: not a member */
int dnmf_comm_rank(void* comm, int* rank, int* size);
int dnmf_comm_destroy(void* comm);
int dnmf_allreduce(void* comm, void* buf, int64_t count, int dtype, void* stream);
int dnmf_allgather(void* comm, const void* send, void* recv, int64_t count_per_rank, int dtype, void* stream);
int dnmf_reduce_scatter(void* comm, const void* send, void* recv, int64_t recv_count, int dtype, void* stream);
int dnmf_bcast(void* comm, void* buf, int64_t count, int dtype, int root, void* stream);
int dnmf_group_start(void);
int dnmf_group_end(void);

/* ---- peer-mapped device memory (NVLink / NVSwitch): the one place the library allocates device memory, because the
 * allocation has to be exportable.  dnmf_symm_alloc returns a zero-filled buffer and its 64-byte CUDA IPC handle;
 * every other rank of the node maps it with dnmf_symm_open and may then load / store through the returned pointer. */
int dnmf_symm_alloc(int64_t bytes, void** ptr, void* handle_out_64);
int dnmf_symm_open(const void* handle_64, void** ptr);
int dnmf_symm_close(void* ptr);
int dnmf_symm_free(void* ptr);

/* ---- fused H half-step of the P x 1 row grid over peer memory.
 * Replaces, per iteration: allreduce(W^T W) dist_nmf.py:679-681, allreduce(W^T A) :705-708, and the update :750-751
 * (FRO-MU), :832-849 (KL-MU: allreduce of colsum(W) :797-799 and of W^T U :808), :895-913 (FRO-HALS) by
 * push (reduce-scatter of the partial into the column-chunk owners) -> update of the owned columns from the sum over
 * ranks in rank order -> write of the new columns into every replica (all-gather); three launches, no NCCL call.
 *   bases[q]: rank q's exchange region (dnmf_xchg_bytes bytes from dnmf_symm_alloc) as mapped on this rank
 *   Yt:  this rank's partial (W_i^T A_i)^T, n x k;  aux: its k x k Gram W_i^T W_i (mode 0, 2) or colsum(W_i) (mode 3)
 *   mode 0 FRO-MU, 2 FRO-HALS, 3 KL-MU;  p0 = eps;  H (k x n) is the replica of this rank, updated in place.
 * dnmf_xchg_error reads the region's error word (set when a wait for a peer timed out). */
int64_t dnmf_xchg_bytes(int nranks, int64_t n, int64_t k, int dtype);
int dnmf_xchg_update_h(void* const* bases, int nranks, int me, int mode, void* H, int64_t ldh, const void* Yt, int64_t ldy,
                       const void* aux, int64_t n, int64_t k, double p0, int clamp, int dtype, void* stream);
/* the same with this rank's partial given as the split-K partials of dnmf_wta_p / dnmf_kl_wtu_p (view4, see above) */
int dnmf_xchg_update_h_p(void* const* bases, int nranks, int me, int mode, void* H, int64_t ldh, const int64_t* view4,
                         const void* aux, int64_t n, int64_t k, double p0, int clamp, int dtype, void* stream);
int dnmf_xchg_error(const void* local_region, int* error_out, void* stream);

/* HALS W sweep (dist_nmf.py:888-893, 2-D :427-432) as ONE cooperative launch: the k Gauss-Seidel column updates with
 * their k dependent global norms (utils.py:388-391) run inside a persistent grid; block partials are summed in a fixed
 * order behind a grid barrier and, for nranks > 1, the per-rank sums travel through the peers' exchange regions
 * (bases, as in dnmf_xchg_update_h; xchg_n = the n the regions were sized for) instead of k all-reduces.
 * scratch: k * 1024 doubles + 256 bytes of device memory, zeroed once by the caller (the kernel leaves it zeroed). */
int dnmf_hals_w_sweep(void* W, int64_t ldw, const void* V, int64_t ldv, const void* G, int64_t m, int64_t k, double eps,
                      void* const* bases, int nranks, int me, int64_t xchg_n, void* scratch, int64_t scratch_bytes, int dtype,
                      void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DNMF_H_ */
