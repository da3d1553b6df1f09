// The training loss of quantum/decoder_v2_4.py:304-317 (LossFunc.forward, train branch) and its gradient,
// fused and SPARSE:   z = y + pred   (per syndrome, V entries)
//   loss = sum_c |sin(pi/2 * sum_{v in check c} z_v)|  +  sum_k |sin(pi/2 * logical_k . z)|
// The reference transposes pred / y with an O(B) Python cat loop and multiplies by the DENSE H^T
// ([C, V]) and `logical`; here a warp owns one syndrome, walks the CSC check lists, and writes
// dL/dpred and dL/dlogit (pred = sigmoid(-logit)  =>  dL/dlogit = -dL/dpred * pred * (1 - pred))
// directly in the layout the backward kernel reads.  Per-syndrome losses are written out and summed
// by the caller in a fixed order (deterministic).
#include "gd_common.cuh"

namespace gd {

__global__ void __launch_bounds__(128) loss_kernel(const float* __restrict__ prob, const uint8_t* __restrict__ y,
                                                   const uint8_t* __restrict__ logical, int K, GraphTables tb,
                                                   long long B, int V, int C, float* __restrict__ loss_per,
                                                   float* __restrict__ grad_prob, float* __restrict__ grad_logit) {
    extern __shared__ float lsm[];   // [4 warps][V + C + K]
    pdl_enter();
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    float* z = lsm + (size_t)wib * (V + C + K);
    float* gc = z + V;               // d loss / d s_c  per check
    float* gl = gc + C;              // d loss / d (logical_k . z)
    constexpr float kHalfPi = 1.57079632679489662f;
    for (long long b = blockIdx.x * 4ll + wib; b < B; b += gridDim.x * 4ll) {
        const float* pb = prob + b * V;
        for (int v = lane; v < V; v += 32) z[v] = pb[v] + (float)y[b * V + v];
        __syncwarp();
        float loss = 0.f;
        for (int c = lane; c < C; c += 32) {
            float s = 0.f;
            for (int i = tb.chk_ptr[c]; i < tb.chk_ptr[c + 1]; ++i) s += z[tb.edge_var[tb.chk_edges[i]]];
            float sn, cs;
            sincospif(0.5f * s, &sn, &cs);
            loss += fabsf(sn);
            gc[c] = (sn < 0.f ? -cs : cs) * kHalfPi;
        }
        for (int k = 0; k < K; ++k) {
            float s = 0.f;
            for (int v = lane; v < V; v += 32) s += logical[k * V + v] ? z[v] : 0.f;
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            float sn, cs;
            sincospif(0.5f * s, &sn, &cs);
            if (lane == 0) {
                loss += fabsf(sn);
                gl[k] = (sn < 0.f ? -cs : cs) * kHalfPi;
            }
        }
        for (int o = 16; o > 0; o >>= 1) loss += __shfl_xor_sync(0xffffffffu, loss, o);
        if (lane == 0) loss_per[b] = loss;
        __syncwarp();
        for (int v = lane; v < V; v += 32) {
            float gp = 0.f;
            for (int i = tb.var_ptr[v]; i < tb.var_ptr[v + 1]; ++i) gp += gc[tb.edge_chk[tb.var_edges[i]]];
            for (int k = 0; k < K; ++k) gp += logical[k * V + v] ? gl[k] : 0.f;
            const float p = pb[v];
            if (grad_prob) grad_prob[b * V + v] = gp;
            if (grad_logit) grad_logit[b * V + v] = -gp * p * (1.0f - p);
        }
        __syncwarp();
    }
}

}  // namespace gd

extern "C" int gd_loss_v2_4(const gd_graph* g, const uint8_t* logical_dev, int32_t K, const float* prob_dev,
                            const uint8_t* y_dev, float* loss_per_syndrome_dev, float* grad_prob_dev,
                            float* grad_logit_dev, int64_t B, void* stream) {
    GD_CHECK_ARG(g != nullptr, "gd_loss_v2_4: graph is NULL");
    GD_CHECK_ARG(K >= 0 && (K == 0 || logical_dev), "gd_loss_v2_4: logical is NULL with K=%d", K);
    GD_CHECK_ARG(B >= 0, "gd_loss_v2_4: negative B");
    if (B == 0) return GD_OK;
    GD_CHECK_ARG(prob_dev && y_dev && loss_per_syndrome_dev, "gd_loss_v2_4: NULL buffer");
    int64_t blocks = (B + 3) / 4;
    if (blocks > (int64_t)g->sm_count * 16) blocks = (int64_t)g->sm_count * 16;
    const int smem = 4 * (g->V + g->C + K) * (int)sizeof(float);
    gd::DeviceGuard dg(g->device);
    GD_CUDA(dg.status());
    cudaError_t e = cudaSuccess;
    if (smem > 48 * 1024) e = cudaFuncSetAttribute(gd::loss_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e == cudaSuccess) {
        e = gd::pdl_launch(gd::loss_kernel, dim3((unsigned)blocks), dim3(128), (size_t)smem, (cudaStream_t)stream,
                           prob_dev, y_dev, logical_dev, K, g->t, B, g->V, g->C, loss_per_syndrome_dev, grad_prob_dev, grad_logit_dev);
    }
    GD_CUDA(e);
    return GD_OK;
}
