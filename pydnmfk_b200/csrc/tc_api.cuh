// Interface between the C-ABI dispatch (dnmf_api.cu) and the tcgen05 / TMA / TMEM path (dnmf_tc.cu).
#pragma once
#include "common.cuh"

namespace dnmf {

// true when the tcgen05 path handles this call: fp32, k in {16, 32, 64}, 16-byte aligned shard with
// lda % 4 == 0, shard large enough to fill the machine, sm_100 device, and not forced off; for a 16-bit A (DNMF_A_*):
// lda % 8 == 0 (AH / WTA: the kind::f16 kernels of dnmf_tc16.cu; KL: the 16-bit build of the fused KL kernel).
bool tc_eligible(int op, const void* A, int64_t lda, int64_t m, int64_t n, int64_t k, int dtype);
void tc_set_min_elems(int64_t elems);
// workspace bytes of the tcgen05 pass for (op, dtype), 0 when there is none; DNMF_OP_AH_RESIDUAL: the fused pass of
// tc_ah_residual_run
int64_t tc_workspace_bytes(int op, int64_t m, int64_t n, int64_t k, int dtype);

// Split-K partials an A-streaming pass leaves in its workspace when the final reduction is deferred to the consumer:
// P[split][x][ldp] (x = row of A for AH / UHT, column of A for WTA / WTU), `splits` buffers `split_stride` elements apart.
struct TcPartials {
  const float* P = nullptr;
  int64_t ldp = 0, split_stride = 0;
  int splits = 0;
};

// One A-streaming pass on the tcgen05 kernels, for a call tc_eligible accepted: op DNMF_OP_AH (out = V = A H^T),
// DNMF_OP_WTA (out = Y = W^T A, or Y^T with transposed_out), DNMF_OP_KL_UHT / DNMF_OP_KL_WTU (the same with A / (W H + eps)
// in place of A).  A is fp32 or 16-bit (dtype).  `defer` != nullptr: skip the final reduction and
// describe the partials instead; `out` is then unused.
int tc_pass(int op, int dtype, const void* A, int64_t lda, const float* W, int64_t ldw, const float* H, int64_t ldh,
            float* out, int64_t ldo, int64_t m, int64_t n, int k, float eps, int transposed_out, void* ws,
            int64_t ws_bytes, cudaStream_t st, TcPartials* defer);

// V = A H^T plus ||A - W H||^2, ||A||^2 in one pass (A fp32 or 16-bit per dtype, k <= 32): per-thread float64 pairs in
// the workspace, to be summed by the caller in a fixed order
int tc_ah_residual_run(const void* A, int dtype, int64_t lda, const float* W, int64_t ldw, const float* H, int64_t ldh,
                       float* V, int64_t ldv, int64_t m, int64_t n, int k, void* ws, int64_t ws_bytes, double** out_pairs,
                       int64_t* n_pairs, cudaStream_t st);

}  // namespace dnmf
