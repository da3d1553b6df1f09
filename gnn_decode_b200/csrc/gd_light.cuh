// Internal interface of the node-owner kernels for the light programs: the forward (gd_decode_light.cu) and the CGNNI
// backward (gd_backward_light.cu) share the parameter block, the planner and the [E][tile] shared-memory layout.
#pragma once
#include "gd_common.cuh"
#include "gd_nodemath.cuh"

namespace gd {

struct LightParams {
    const float* x;
    float* prob;
    float* logit;
    uint8_t* hard;
    const float* weights;
    GraphTables tb;
    long long B;
    int T, V, C, E, N;
    int tile, lanes, R, hid, hp, n_tiles, trows;
    int off_w, off_tab, off_x, off_m, off_t;
    // training: m after every iteration, stash[it][E][B] (CGNNI forward with stash), or the stash the backward reads
    float* stash;
};

struct LightPlan {
    LightParams p;
    int threads, grid, smem, npad, cps;
    bool ok;
    const char* why;   // train mode: why the graph cannot take the node-owner kernel (ok == false)
};

// Plans the node-owner kernel for (graph, model, B).  train: the forward with stash / the backward, which have no other
// kernel -- the "is this kernel worth it" gates are skipped and the ReLU MLPs are always the piecewise-linear tables;
// extra_rows [tile] float rows per syndrome and extra_bytes of fixed shared memory are reserved after the forward's
// layout (the backward's dm rows and weight-gradient bins).
void plan_light(const gd_graph* g, const gd_model* m, int64_t B, LightPlan* out, bool train = false, int extra_rows = 0,
                int extra_bytes = 0);

// CGNNI backward (gd_backward_light.cu): workspace floats (-1 and gd_last_error() if the graph cannot take the kernel), and the
// gradient of gd_decode_bwd (a gd_status).
int64_t light_bwd_workspace_floats(const gd_graph* g, const gd_model* model, int64_t B);
int light_backward(const gd_graph* g, const gd_model* model, const float* weights_dev, const float* x_dev, const float* stash_dev,
                   const float* grad_logit_dev, float* grad_weights_dev, float* workspace_dev, int accumulate, int64_t B,
                   cudaStream_t st);

#ifdef __CUDACC__
// Variable phase of the light programs: the owner of variable v turns the messages of its edges (rows var_ptr[v] .. of
// m_st) and its prior into the values the check phase sums (rows of t_st).  Summation order is ascending edge id.
// The backward recomputes t with it; it is the same arithmetic, in the same order, as the loop inlined in
// decode_light_kernel, so every recomputed value is bit-identical to the forward's.  (The forward keeps its inlined copy:
// calling this function there changes the register allocation of the inference kernels.)
template <int PROG, int NPAD>
__device__ __forceinline__ void light_var_phase(const NodeMath<PROG, NPAD>& nm, const uint16_t* var_ptr, const float* xT,
                                                const float* m_st, float* t_st, int V, int R, int r, int tile, int l4) {
    for (int v = r; v < V; v += R) {
        const int b = var_ptr[v], d = var_ptr[v + 1] - b;
        const float4 pr = lds4(xT + v * tile + l4);
        const float* rows = m_st + b * tile + l4;
        float* tout = t_st + b * tile + l4;
        switch (d) {
            case 1: nm.template var_node<1>(rows, tile, pr, tout); break;
            case 2: nm.template var_node<2>(rows, tile, pr, tout); break;
            case 3: nm.template var_node<3>(rows, tile, pr, tout); break;
            case 4: nm.template var_node<4>(rows, tile, pr, tout); break;
            default: {
                float acc[4] = {0.f, 0.f, 0.f, 0.f};
                for (int k = 0; k < d; ++k) {      // ascending edge id
                    const float4 mv = lds4(rows + k * tile);
                    acc[0] += mv.x; acc[1] += mv.y; acc[2] += mv.z; acc[3] += mv.w;
                }
                const float prv[4] = {pr.x, pr.y, pr.z, pr.w};
                for (int k = 0; k < d; ++k) {
                    const float4 mv = lds4(rows + k * tile);
                    const float ext[4] = {acc[0] - mv.x, acc[1] - mv.y, acc[2] - mv.z, acc[3] - mv.w};
                    float out[4];
                    nm.var_update(ext, prv, out);
                    stg4(tout + k * tile, out);
                }
            } break;
        }
    }
}
#endif

}  // namespace gd
