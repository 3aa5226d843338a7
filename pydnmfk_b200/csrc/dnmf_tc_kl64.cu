// Fused KL contractions on the tcgen05 path for 32 < k <= 64: the kernels of dnmf_tc_kl.cu built for a 64-wide factor
// (KL_KK = 64: Fx hi | lo takes 128 tensor-memory columns, the accumulator 128, which leaves two 64-column rings of two
// slots each -- hence two splitter groups; GEMM1 runs 24 N = 64 MMAs per tile pair over two swizzle atoms along k).
// Exports tc_kl_layout_k64 / tc_kl_run_k64; dnmf_tc.cu dispatches on k.
#define KL_KK 64
#include "dnmf_tc_kl.cu"
