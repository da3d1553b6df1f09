// Hard-decision evaluation on the device with the SPARSE parity-check tables instead of the
// reference's dense matmul: residual-syndrome and logical-failure counters with the semantics of
// LossFunc.forward(train=0) in quantum/neural_BP.py:338-348 (loss_a = decodes whose residual
// error e xor ehat violates a check; loss_b = decodes that satisfy every check but flip a logical).
#include "gd_common.cuh"

namespace gd {

// one warp per sample
__global__ void __launch_bounds__(128) eval_kernel(const uint8_t* __restrict__ err, const uint8_t* __restrict__ hard,
                                                   const uint8_t* __restrict__ logical, int K, GraphTables tb,
                                                   long long B, int V, int C, unsigned long long* counts) {
    const int lane = threadIdx.x & 31;
    unsigned long long n_syn = 0, n_log = 0;
    for (long long b = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5; b < B;
         b += ((long long)gridDim.x * blockDim.x) >> 5) {
        const uint8_t* eb = err + b * V;
        const uint8_t* hb = hard + b * V;
        int bad = 0;
        for (int c = lane; c < C; c += 32) {
            int par = 0;
            for (int i = tb.chk_ptr[c]; i < tb.chk_ptr[c + 1]; ++i) {
                const int v = tb.edge_var[tb.chk_edges[i]];
                par ^= (eb[v] ^ hb[v]) & 1;
            }
            bad |= par;
        }
        bad = __any_sync(0xffffffffu, bad);
        int lbad = 0;
        for (int k = 0; k < K; ++k) {
            int par = 0;
            for (int v = lane; v < V; v += 32) par ^= logical[k * V + v] & (eb[v] ^ hb[v]) & 1;
            par = __popc(__ballot_sync(0xffffffffu, par)) & 1;
            lbad |= par;
        }
        if (lane == 0) {
            n_syn += bad ? 1 : 0;
            n_log += (!bad && lbad) ? 1 : 0;
        }
    }
    if (lane == 0 && (n_syn | n_log)) {
        if (n_syn) atomicAdd(counts + 0, n_syn);
        if (n_log) atomicAdd(counts + 1, n_log);
        atomicAdd(counts + 2, n_syn + n_log);
    }
}

}  // namespace gd

extern "C" int gd_eval_failures(const gd_graph* g, const uint8_t* logical_dev, int32_t K, const uint8_t* err_dev,
                                const uint8_t* hard_dev, int64_t B, unsigned long long* counts_dev, void* stream) {
    GD_CHECK_ARG(g != nullptr, "gd_eval_failures: graph is NULL");
    GD_CHECK_ARG(K >= 0 && (K == 0 || logical_dev), "gd_eval_failures: logical is NULL with K=%d", K);
    GD_CHECK_ARG(B >= 0, "gd_eval_failures: negative B");
    if (B == 0) return GD_OK;
    GD_CHECK_ARG(err_dev && hard_dev && counts_dev, "gd_eval_failures: NULL buffer");
    int64_t blocks = (B + 3) / 4;
    if (blocks > (int64_t)g->sm_count * 16) blocks = (int64_t)g->sm_count * 16;
    gd::DeviceGuard dg(g->device);
    GD_CUDA(dg.status());
    gd::eval_kernel<<<(int)blocks, 128, 0, (cudaStream_t)stream>>>(err_dev, hard_dev, logical_dev, K, g->t, B, g->V,
                                                                  g->C, counts_dev);
    cudaError_t e = cudaGetLastError();
    GD_CUDA(e);
    return GD_OK;
}
