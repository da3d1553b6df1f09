// gd_adam_step: the optimizer step of the training loop (quantum/decoder_v2_4.py:323, 338) on the flat fp32 master
// weight vector the decode kernels read -- one launch instead of torch.optim's per-tensor / foreach kernels over the
// 12 parameter tensors.  The data-parallel variant fuses the same update into the peer-memory all-reduce (gd_p2p.cu).
#include "gd_adam.cuh"
#include "gd_common.cuh"
#include <algorithm>

namespace gd {

__global__ void __launch_bounds__(256) adam_kernel(const AdamCoef c, float* __restrict__ w, const float* __restrict__ g,
                                                   float* __restrict__ m, float* __restrict__ v, const float gscale, const long long n) {
    gd::pdl_enter();
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        float wi = w[i], mi = m[i], vi = v[i];
        adam_update(c, g[i] * gscale, wi, mi, vi);
        w[i] = wi; m[i] = mi; v[i] = vi;
    }
}

}  // namespace gd

extern "C" int gd_adam_step(const gd_adam* opt, float* weights_dev, const float* grad_dev, float* exp_avg_dev,
                            float* exp_avg_sq_dev, int64_t n, float grad_scale, void* stream) {
    GD_CHECK_ARG(opt && weights_dev && grad_dev && exp_avg_dev && exp_avg_sq_dev, "gd_adam_step: NULL argument");
    GD_CHECK_ARG(n > 0 && opt->step >= 1, "gd_adam_step: n and step must be positive");
    GD_CHECK_ARG(opt->beta1 >= 0. && opt->beta1 < 1. && opt->beta2 >= 0. && opt->beta2 < 1. && opt->eps >= 0. && opt->lr >= 0.
                 && opt->weight_decay >= 0., "gd_adam_step: invalid hyper-parameters");
    const gd::AdamCoef c = gd::adam_coef(opt->lr, opt->beta1, opt->beta2, opt->eps, opt->weight_decay, opt->step);
    const int grid = (int)std::min<int64_t>((n + 255) / 256, 1184);
    GD_CUDA(gd::pdl_launch(gd::adam_kernel, dim3(grid), dim3(256), 0, (cudaStream_t)stream, c, weights_dev, grad_dev, exp_avg_dev,
                           exp_avg_sq_dev, grad_scale, (long long)n));
    GD_CUDA(cudaGetLastError());
    return GD_OK;
}
