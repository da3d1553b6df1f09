// Elementwise probe of the sum-product device primitives (gd_math.cuh, gd_nodemath.cuh) for
// tests/test_sum_product_math_gpu.py: each kernel evaluates one primitive exactly as the decode and
// training kernels inline it, so the test sees the same arithmetic without a change to the library's ABI.
#include "gd_nodemath.cuh"

namespace {

enum Fn {
    LOG_ABS_TANH_HALF_CLAMPED = 0,   // bp_log_abs_tanh_half<true>(a, param)
    LOG_ABS_TANH_HALF = 1,           // bp_log_abs_tanh_half<false>(a, param)
    NBP_T = 2,                       // NodeMath<GD_PROG_NEURAL_BP>::nbp_t(a)
    ONE_MINUS_EXP = 3,               // bp_one_minus_exp(u, ex2(-u log2 e)), as bp_check_out and bp_dcheck_out call it
    CHECK_OUT = 4,                   // bp_check_out(ext, odd, param)
    DCHECK_OUT = 5,                  // bp_dcheck_out(ext, odd, param)
    DLOG_ABS_TANH_HALF = 6,          // bp_dlog_abs_tanh_half(a, bp_log_abs_tanh_half<false>(a, param), param), as gd_backward_nbp.cu
};

__global__ void probe_kernel(int fn, const float* in, float* out, int n, float param, bool odd) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float a = in[i];
    float r = 0.f;
    switch (fn) {
        case LOG_ABS_TANH_HALF_CLAMPED: r = gd::bp_log_abs_tanh_half<true>(a, param); break;
        case LOG_ABS_TANH_HALF: r = gd::bp_log_abs_tanh_half<false>(a, param); break;
        case NBP_T: r = gd::NodeMath<GD_PROG_NEURAL_BP, 0>::nbp_t(a); break;
        case ONE_MINUS_EXP: r = gd::bp_one_minus_exp(a, gd::ex2_approx(-a * gd::kLog2e)); break;
        case CHECK_OUT: r = gd::bp_check_out(a, odd, param); break;
        case DCHECK_OUT: r = gd::bp_dcheck_out(a, odd, param); break;
        case DLOG_ABS_TANH_HALF: r = gd::bp_dlog_abs_tanh_half(a, gd::bp_log_abs_tanh_half<false>(a, param), param); break;
        default: r = __int_as_float(0x7fffffff); break;
    }
    out[i] = r;
}

}  // namespace

// out[i] = primitive fn at in[i] (device pointers, n elements), on the legacy default stream.  Returns the launch's cudaError_t.
extern "C" int sp_math_probe(int fn, const float* in, float* out, int n, float param, int odd) {
    if (n <= 0) return 0;
    probe_kernel<<<(n + 255) / 256, 256>>>(fn, in, out, n, param, odd != 0);
    return (int)cudaGetLastError();
}
