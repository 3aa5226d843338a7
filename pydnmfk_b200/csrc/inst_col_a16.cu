// explicit instantiation of the generic col-owner pass and of the residual kernel for a 16-bit A (fp16 / bf16) with
// fp32 factors
#define DNMF_INSTANTIATE_COL
#define DNMF_INSTANTIATE_SMALL
#include "launch_small.cuh"
namespace dnmf {
template int col_pass_dispatch<float, __half>(bool, const __half*, int64_t, const float*, int64_t, const float*, int64_t, float*, int64_t, int64_t, int64_t, int, float, int, void*, int64_t, cudaStream_t);
template int col_pass_dispatch<float, __nv_bfloat16>(bool, const __nv_bfloat16*, int64_t, const float*, int64_t, const float*, int64_t, float*, int64_t, int64_t, int64_t, int, float, int, void*, int64_t, cudaStream_t);
template int residual_dispatch<float, __half>(const __half*, int64_t, const float*, int64_t, const float*, int64_t, int64_t, int64_t, int, int64_t, unsigned, unsigned, double*, double*, double*, cudaStream_t);
template int residual_dispatch<float, __nv_bfloat16>(const __nv_bfloat16*, int64_t, const float*, int64_t, const float*, int64_t, int64_t, int64_t, int, int64_t, unsigned, unsigned, double*, double*, double*, cudaStream_t);
}
