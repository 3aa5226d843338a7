// explicit instantiation of the generic row-owner pass for a 16-bit A (fp16 / bf16) with fp32 factors
#define DNMF_INSTANTIATE_ROW
#include "launch_passes.cuh"
namespace dnmf {
template int row_pass_dispatch<float, __half>(bool, const __half*, int64_t, const float*, int64_t, const float*, int64_t, float*, int64_t, int64_t, int64_t, int, float, void*, int64_t, cudaStream_t);
template int row_pass_dispatch<float, __nv_bfloat16>(bool, const __nv_bfloat16*, int64_t, const float*, int64_t, const float*, int64_t, float*, int64_t, int64_t, int64_t, int, float, void*, int64_t, cudaStream_t);
}
