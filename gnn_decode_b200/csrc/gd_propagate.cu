// One MessagePassing.propagate() (+ optionally the fused GraphConv.update) on batch-major
// [B, E] messages -- the compatibility path behind GraphConv.forward / propagate().
// Reference: quantum/decoder_v2_4.py:85-148,253-257; classical/CGNNI.py:52-112,238-242;
// quantum/QGNNI.py:54-116,207-214; quantum/BP.py:101-124; classical/BP.py:99-123.
//
// One warp per (syndrome, 32 nodes) would starve on degree-1 nodes, so the mapping is one thread
// per (syndrome b, node n): it sums its segment in ascending edge id (deterministic; same order
// as the CPU index_add_), then writes sum-minus-self -> post -> update for each of its edges.
#include "gd_common.cuh"
#include "gd_math.cuh"

namespace gd {

struct PropParams {
    const float* m;
    const float* x;
    const float* w;
    float* out;
    GraphTables tb;
    long long B;
    int V, C, E, N, hid, hp, fuse;
};

template <int PROG, int PHASE>
__global__ void __launch_bounds__(128) propagate_kernel(const PropParams p) {
    extern __shared__ __align__(16) float wsm[];
    constexpr bool kIsBP = (PROG == GD_PROG_BP_QUANTUM || PROG == GD_PROG_BP_CLASSICAL);
    constexpr bool kNBP = (PROG == GD_PROG_NEURAL_BP);
    constexpr bool kGRU = (PROG == GD_PROG_GRU_CA);
    constexpr bool kV3 = (PROG == GD_PROG_V3_0);         // decoder_v3_0.py:103-112: plain sums, cat the node input in both phases
    constexpr bool kV122 = (PROG == GD_PROG_V1_2_2);     // decoder_v1_2_2.py:105-124: cat prior / sum-product check rule
    // (V3_0 / V1_2_2: the un-fused form only -- their update()s run in the caller, or everything in the fused decoder)
    constexpr bool kHasMlp = (PROG == GD_PROG_V2_4) || kGRU || (!kIsBP && !kNBP && !kV3 && !kV122 && PHASE == GD_PHASE_CHK);
    const int hp = p.hp, h = p.hid;
    MlpSmem W{};
    if (kHasMlp && p.fuse) {
        const float* w = p.w;
        const bool sp = PROG == GD_PROG_V2_4;
        const float s1 = sp ? kLog2e : 1.f, s2 = sp ? kLn2 : 1.f;
        const bool two = PROG == GD_PROG_V2_4 && PHASE == GD_PHASE_VAR;
        for (int k = threadIdx.x; k < hp; k += blockDim.x) {
            const bool in = k < h;
            wsm[k] = in ? w[two ? 2 * k : k] * s1 : 0.f;
            wsm[hp + k] = (in && two) ? w[2 * k + 1] * s1 : 0.f;
            wsm[2 * hp + k] = in ? w[(two ? 2 : 1) * h + k] * s1 : 0.f;
            wsm[3 * hp + k] = in ? w[(two ? 3 : 2) * h + k] * s2 : 0.f;
        }
        W = MlpSmem{wsm, wsm + hp, wsm + 2 * hp, wsm + 3 * hp, w[(two ? 4 : 3) * h]};
        __syncthreads();
    }
    const int n_nodes = PHASE == GD_PHASE_VAR ? p.V : p.C;
    const int32_t* ptr = PHASE == GD_PHASE_VAR ? p.tb.var_ptr : p.tb.chk_ptr;
    const int32_t* ids = PHASE == GD_PHASE_VAR ? p.tb.var_edges : p.tb.chk_edges;
    const long long total = p.B * n_nodes;
    for (long long gi = blockIdx.x * (long long)blockDim.x + threadIdx.x; gi < total;
         gi += (long long)gridDim.x * blockDim.x) {
        const long long b = gi / n_nodes;
        const int n = (int)(gi - b * n_nodes);
        const float* mb = p.m + b * p.E;
        const float extra = p.x ? p.x[b * p.N + (PHASE == GD_PHASE_VAR ? n : p.V + n)] : 0.f;
        const int e0 = ptr[n], e1 = ptr[n + 1];
        float acc = 0.f, cnt = 0.f;
        for (int i = e0; i < e1; ++i) {
            const float v = mb[ids[i]];
            if constexpr (PHASE == GD_PHASE_VAR || kGRU || kV3) {
                acc += v;                                      // QGNNNI_ca.py:101: no tanh in either phase
            } else if constexpr (kNBP || kV122) {
                acc += bp_log_abs_tanh_half<false>(v, -46.0517019f);
                cnt += v < 0.f ? 1.f : 0.f;
            } else if constexpr (kIsBP) {
                acc += bp_log_abs_tanh_half(v, PROG == GD_PROG_BP_QUANTUM ? -46.0517019f : -16.1180957f);
                cnt += v < 0.f ? 1.f : 0.f;
            } else {
                acc += tanh_half(v);
            }
        }
        for (int i = e0; i < e1; ++i) {
            const int e = ids[i];
            const float v = mb[e];
            float self, res0, res1 = extra;
            bool two_out = false;
            if constexpr (PHASE == GD_PHASE_VAR) {
                self = v;
                const float ext = acc - self;
                if constexpr (PROG == GD_PROG_V2_4) {          // cat[ext, prior] -> mlp
                    if (p.fuse) {
                        float a0[1] = {ext}, a1[1] = {extra}, o[1];
                        mlp_softplus<1, true>(W, hp, a0, a1, o);
                        res0 = o[0];
                    } else { res0 = ext; two_out = true; }
                } else if constexpr (kV3 || kV122) {          // cat[ext, prior]; update() is the caller's
                    res0 = ext; two_out = true;
                } else if constexpr (kNBP) {                  // neural_BP.py:122-124,253-255: cat[ext, prior]; update = ext + prior * W_p
                    if (p.fuse) res0 = ext + extra * p.w[e];
                    else { res0 = ext; two_out = true; }
                } else if constexpr (kGRU) {                  // QGNNNI_ca.py:103-106,208-209: mlp1(ext + prior)
                    res0 = ext + extra;
                    if (p.fuse) {
                        float a0[1] = {res0}, o[1];
                        mlp_relu<1>(W, hp, a0, o);
                        res0 = o[0];
                    }
                } else {
                    res0 = ext + extra;                        // + post / extra; update = identity
                }
            } else if constexpr (kV3) {                       // decoder_v3_0.py:103,111: cat[sum - self, syndrome]
                res0 = acc - v; two_out = true;
            } else if constexpr (kV122) {                     // decoder_v1_2_2.py:105-119: eps 1e-20 / 1e-12, no input clamp; identity update
                const float lg = bp_log_abs_tanh_half<false>(v, -46.0517019f);
                int k = (int)(cnt - (v < 0.f ? 1.f : 0.f));
                k += extra < 0.f ? 1 : 0;
                res0 = bp_check_out(acc - lg, k & 1, 1e-12f);
            } else if constexpr (kGRU) {                      // QGNNNI_ca.py:109,206-207: mlp2((sum - self) * s)
                res0 = (acc - v) * extra;
                if (p.fuse) {
                    float a0[1] = {res0}, o[1];
                    mlp_relu<1>(W, hp, a0, o);
                    res0 = o[0];
                }
            } else if constexpr (kNBP) {                      // neural_BP.py:108-122
                const float lg = bp_log_abs_tanh_half<false>(v, -46.0517019f);
                int k = (int)(cnt - (v < 0.f ? 1.f : 0.f));
                k += extra < 0.f ? 1 : 0;
                res0 = bp_check_out(acc - lg, k & 1, 1e-15f);
            } else if constexpr (kIsBP) {
                const float lg = bp_log_abs_tanh_half(v, PROG == GD_PROG_BP_QUANTUM ? -46.0517019f : -16.1180957f);
                int k = (int)(cnt - (v < 0.f ? 1.f : 0.f));
                if constexpr (PROG == GD_PROG_BP_QUANTUM) k += extra < 0.f ? 1 : 0;
                res0 = bp_check_out(acc - lg, k & 1, PROG == GD_PROG_BP_QUANTUM ? 1e-12f : 1e-7f);
            } else {
                self = tanh_half(v);
                const float ext = acc - self;
                if (p.fuse) {
                    float a0[1] = {ext}, o[1];
                    if constexpr (PROG == GD_PROG_V2_4) mlp_softplus<1, false>(W, hp, a0, a0, o);
                    else mlp_relu<1>(W, hp, a0, o);
                    res0 = PROG == GD_PROG_CGNNI ? o[0] : o[0] * extra;
                } else {
                    res0 = ext;
                    two_out = PROG != GD_PROG_CGNNI;           // QGNNI / v2_4 cat the syndrome sign
                }
            }
            if (two_out) {
                p.out[(b * p.E + e) * 2] = res0;
                p.out[(b * p.E + e) * 2 + 1] = res1;
            } else {
                p.out[b * p.E + e] = res0;
            }
        }
    }
}

template <int PROG>
static int launch_prop(const PropParams& p, int phase, int grid, int smem, cudaStream_t st) {
    if (phase == GD_PHASE_VAR) propagate_kernel<PROG, GD_PHASE_VAR><<<grid, 128, smem, st>>>(p);
    else propagate_kernel<PROG, GD_PHASE_CHK><<<grid, 128, smem, st>>>(p);
    GD_CUDA(cudaGetLastError());
    return GD_OK;
}

}  // namespace gd

extern "C" int gd_propagate_features(int32_t program, int32_t phase) {
    if (phase == GD_PHASE_VAR)
        return (program == GD_PROG_V2_4 || program == GD_PROG_NEURAL_BP || program == GD_PROG_V3_0 || program == GD_PROG_V1_2_2) ? 2 : 1;
    if (phase == GD_PHASE_CHK) return (program == GD_PROG_V2_4 || program == GD_PROG_QGNNI || program == GD_PROG_V3_0) ? 2 : 1;
    return -1;
}

extern "C" int gd_propagate_fwd(const gd_graph* g, const gd_model* model, int32_t phase, int32_t fuse_update,
                                const float* m_dev, const float* x_dev, const float* weights_dev, float* out_dev,
                                int64_t B, void* stream) {
    GD_CHECK_ARG(g != nullptr, "gd_propagate_fwd: graph is NULL");
    GD_CHECK_ARG(gd_model_valid(model), "gd_propagate_fwd: invalid model");
    GD_CHECK_ARG(phase == GD_PHASE_VAR || phase == GD_PHASE_CHK, "gd_propagate_fwd: phase must be 0 (var) or 1 (chk)");
    GD_CHECK_ARG(B >= 0, "gd_propagate_fwd: negative B");
    if (B == 0) return GD_OK;
    GD_CHECK_ARG(m_dev && out_dev, "gd_propagate_fwd: m / out is NULL");
    const int prog = model->program;
    const bool x_optional = (prog == GD_PROG_CGNNI || prog == GD_PROG_BP_CLASSICAL) && phase == GD_PHASE_CHK;
    GD_CHECK_ARG(x_dev || x_optional, "gd_propagate_fwd: x (extra/post) is NULL");
    const bool ext_only = prog == GD_PROG_V3_0 || prog == GD_PROG_V1_2_2;     // update() of these scripts is not part of this kernel
    if (ext_only && fuse_update && !(prog == GD_PROG_V1_2_2 && phase == GD_PHASE_CHK)) {
        gd::set_error("gd_propagate_fwd: program %d has no fused update in the propagate kernel (use fuse_update = 0 or gd_decode_fwd)", prog);
        return GD_ERR_UNSUPPORTED;
    }
    const bool bp = prog == GD_PROG_BP_QUANTUM || prog == GD_PROG_BP_CLASSICAL || prog == GD_PROG_NEURAL_BP || ext_only;
    const bool has_mlp = fuse_update && ((!bp && (prog == GD_PROG_V2_4 || prog == GD_PROG_GRU_CA || phase == GD_PHASE_CHK)) ||
                                         (prog == GD_PROG_NEURAL_BP && phase == GD_PHASE_VAR));   // W_p[E] there
    GD_CHECK_ARG(!has_mlp || weights_dev, "gd_propagate_fwd: weights is NULL");
    gd::PropParams p;
    p.m = m_dev; p.x = x_optional && (prog == GD_PROG_CGNNI || prog == GD_PROG_BP_CLASSICAL) ? nullptr : x_dev;
    p.w = weights_dev; p.out = out_dev; p.tb = g->t; p.B = B;
    p.V = g->V; p.C = g->C; p.E = (int)g->E; p.N = g->N;
    p.hid = bp ? 0 : model->hidden; p.hp = (p.hid + 3) / 4 * 4; p.fuse = fuse_update ? 1 : 0;
    const int64_t total = B * (phase == GD_PHASE_VAR ? g->V : g->C);
    int64_t blocks = (total + 127) / 128;
    if (blocks > (int64_t)g->sm_count * 16) blocks = (int64_t)g->sm_count * 16;
    const int smem = 4 * p.hp * (int)sizeof(float) + 16;
    cudaStream_t st = (cudaStream_t)stream;
    gd::DeviceGuard dg(g->device);
    GD_CUDA(dg.status());
    int rc;
    switch (prog) {
        case GD_PROG_CGNNI: rc = gd::launch_prop<GD_PROG_CGNNI>(p, phase, (int)blocks, smem, st); break;
        case GD_PROG_QGNNI: rc = gd::launch_prop<GD_PROG_QGNNI>(p, phase, (int)blocks, smem, st); break;
        case GD_PROG_V2_4: rc = gd::launch_prop<GD_PROG_V2_4>(p, phase, (int)blocks, smem, st); break;
        case GD_PROG_BP_QUANTUM: rc = gd::launch_prop<GD_PROG_BP_QUANTUM>(p, phase, (int)blocks, smem, st); break;
        case GD_PROG_NEURAL_BP: rc = gd::launch_prop<GD_PROG_NEURAL_BP>(p, phase, (int)blocks, smem, st); break;
        case GD_PROG_GRU_CA: rc = gd::launch_prop<GD_PROG_GRU_CA>(p, phase, (int)blocks, smem, st); break;
        case GD_PROG_V3_0: rc = gd::launch_prop<GD_PROG_V3_0>(p, phase, (int)blocks, smem, st); break;
        case GD_PROG_V1_2_2: rc = gd::launch_prop<GD_PROG_V1_2_2>(p, phase, (int)blocks, smem, st); break;
        default: rc = gd::launch_prop<GD_PROG_BP_CLASSICAL>(p, phase, (int)blocks, smem, st); break;
    }
    return rc;
}
