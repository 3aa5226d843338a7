// Interface between the C-ABI dispatch (dnmf_api.cu) and the tcgen05 / TMA / TMEM path (dnmf_tc.cu).
#pragma once
#include "common.cuh"

namespace dnmf {

// true when the tcgen05 path handles this call: fp32, k in {16, 32, 64}, 16-byte aligned shard with
// lda % 4 == 0, shard large enough to fill the machine, sm_100 device, and not forced off; for a 16-bit A (DNMF_A_*):
// AH / WTA only, lda % 8 == 0 (the kind::f16 kernels of dnmf_tc16.cu).
bool tc_eligible(int op, const void* A, int64_t lda, int64_t m, int64_t n, int64_t k, int dtype);
void tc_set_min_elems(int64_t elems);
void tc_set_debug(int flags);      // timing-ablation bits (tests/tools only; results become wrong when non-zero)
void tc_set_profile(void* buf);   // debug: device buffer [grid][16] of cycle counts per warp role, or nullptr
int64_t tc_workspace_bytes(int op, int64_t m, int64_t n, int64_t k, int dtype);

// Split-K partials an A-streaming pass leaves in its workspace when the final reduction is deferred to the consumer:
// P[split][x][ldp] (x = row of A for AH / UHT, column of A for WTA / WTU), `splits` buffers `split_stride` elements apart.
struct TcPartials {
  const float* P = nullptr;
  int64_t ldp = 0, split_stride = 0;
  int splits = 0;
};

// (`defer` != nullptr: skip the final reduce_partials launch and describe the partials instead; `out` is then unused)
int tc_ah(const float* A, int64_t lda, const float* H, int64_t ldh, float* V, int64_t ldv, int64_t m, int64_t n,
          int k, int math_mode, void* ws, int64_t ws_bytes, cudaStream_t st, TcPartials* defer = nullptr);
int tc_wta(const float* A, int64_t lda, const float* W, int64_t ldw, float* Y, int64_t ldy, int64_t m, int64_t n,
           int k, int transposed_out, int math_mode, void* ws, int64_t ws_bytes, cudaStream_t st, TcPartials* defer = nullptr);
int tc_kl_uht(const float* A, int64_t lda, const float* W, int64_t ldw, const float* H, int64_t ldh, float* V,
              int64_t ldv, int64_t m, int64_t n, int k, float eps, int math_mode, void* ws, int64_t ws_bytes,
              cudaStream_t st, TcPartials* defer = nullptr);
int tc_kl_wtu(const float* A, int64_t lda, const float* W, int64_t ldw, const float* H, int64_t ldh, float* Y,
              int64_t ldy, int64_t m, int64_t n, int k, float eps, int transposed_out, int math_mode, void* ws,
              int64_t ws_bytes, cudaStream_t st, TcPartials* defer = nullptr);

// 16-bit A (dtype DNMF_A_F16 / DNMF_A_BF16), fp32 factors and outputs: the tcgen05 kind::f16 kernels of dnmf_tc16.cu
int64_t tc16_workspace_bytes(int op, int64_t m, int64_t n, int64_t k, int dtype);
int tc16_ah(const void* A, int64_t lda, const float* H, int64_t ldh, float* V, int64_t ldv, int64_t m, int64_t n, int k,
            int dtype, void* ws, int64_t ws_bytes, cudaStream_t st, TcPartials* defer = nullptr);
int tc16_wta(const void* A, int64_t lda, const float* W, int64_t ldw, float* Y, int64_t ldy, int64_t m, int64_t n, int k,
             int transposed_out, int dtype, void* ws, int64_t ws_bytes, cudaStream_t st, TcPartials* defer = nullptr);

// V = A H^T plus ||A - W H||^2, ||A||^2 in one pass (fp32, k <= 32): per-thread float64 pairs like tc_residual_run
int64_t tc_ah_residual_workspace_bytes(int64_t m, int64_t n);
int tc_ah_residual_run(const float* A, int64_t lda, const float* W, int64_t ldw, const float* H, int64_t ldh, float* V,
                       int64_t ldv, int64_t m, int64_t n, int k, void* ws, int64_t ws_bytes, double** out_pairs,
                       int64_t* n_pairs, cudaStream_t st);

// ||A - W H||^2, ||A||^2 on the tcgen05 pipeline (opt-in, DNMF_TC_RESIDUAL=1; fp32, k <= 32): per-thread float64 pairs in
// the workspace, to be summed by the caller in a fixed order.
bool tc_residual_enabled();
void tc_set_residual(int on);
int64_t tc_residual_workspace_bytes(int64_t m, int64_t n);
int tc_residual_run(const float* A, int64_t lda, const float* W, int64_t ldw, const float* H, int64_t ldh, int64_t m,
                    int64_t n, int k, void* ws, int64_t ws_bytes, double** out_pairs, int64_t* n_pairs, cudaStream_t st);

}  // namespace dnmf
