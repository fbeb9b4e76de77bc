// Host launchers of the wide-level channel-mix kernels (wide_mix.cu): levels of 192 < C <= 1024 channels, whose C x C
// matrix does not fit the shared memory of the single-pass kernels.  The C ABI entry points (nfdpm_channel_mix,
// nfdpm_mix_bwd, nfdpm_mix_inv_param_grad) dispatch here for C > kWideMixMin only, after their argument checks.
#pragma once
#include "common.cuh"

namespace nfdpm {

constexpr int kWideMixMin = 192;    // widest level of the single-pass kernels
constexpr int kWideMixMax = 1024;   // widest level of any kernel (nfdpm_mix_prepare's bound)

// y[b,o,p] = sum_i mt[i*C+o] x[b,i,p] + beta[o], i ascending (the order of chanmix_generic_kernel)
int chanmix_wide(const float* x, float* y, const float* mt, const float* beta, int B, int C, int P, int64_t xbs,
                 int64_t ybs, cudaStream_t st);

// nfdpm_mix_bwd for wide levels: one partial row per image (nfdpm_mix_bwd_tiles returns 1)
int mix_bwd_wide(const float* du, int64_t du_bs, const float* da1, int64_t lda1, const float* x, int64_t x_bs,
                 const float* mt, float* dx, int64_t dx_bs, float* part, int B, int C, int H, int W, cudaStream_t st);

// nfdpm_mix_inv_param_grad of one wide item (the fields of nfdpm_mix_grad_item; scratch: C*C + C floats)
int mix_inv_param_grad_wide(const float* part, int B, int C, const float* s, const float* winv, const float* dld_sum,
                            float P, float* d_weight, float* d_scale, float* d_bias, float* scratch, cudaStream_t st);

}  // namespace nfdpm
