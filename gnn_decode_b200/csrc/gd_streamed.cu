// Streamed global-memory decoder for codes whose edge state does not fit shared memory
// (BASELINE config 5: hypergraph-product [[1600,64]], V = 3200, C = 1536, E = 10752).
// Same arithmetic as gd_decode.cu (reference GNNI.forward), different data movement:
//   * each persistent CTA owns a slab in global memory  xT[N][tile] | m[E][tile] | t[E][tile]
//     (batch-minor: lanes = syndromes, so every state access is one coalesced 128-byte line);
//   * NODE-OWNER phases: thread (s, r) owns variable nodes v == r (mod R) in the variable phase
//     and check nodes c == r (mod R) in the check phase.  It reads its node's deg messages,
//     sums them in ascending edge id, and writes the deg outgoing messages -- m and t are each
//     read and written exactly as often as the algorithm requires (m: R,R,W  t: W,R per
//     iteration = 20 bytes/edge/iteration in fp32, the algorithmic figure of SURVEY.md 8d),
//     there are no node-sum arrays and only two barriers per iteration;
//   * graph tables are read from global memory through the read-only path (warp-uniform ->
//     one broadcast transaction per warp), MLP weights sit in shared memory.
#include "gd_common.cuh"
#include "gd_math.cuh"
#include "gd_options.cuh"
#include "gd_decode.cuh"
#include <stdlib.h>
#include <string.h>

namespace gd {

__device__ __forceinline__ void stage_mlp_s(float* dst, int hp, int hid, const float* w1, int w1_stride, bool two_in,
                                            const float* b1, const float* w2, float s1, float s2, int tid, int nthr) {
    for (int k = tid; k < hp; k += nthr) {
        const bool in = k < hid;
        dst[k] = in ? w1[k * w1_stride] * s1 : 0.f;
        dst[hp + k] = (in && two_in) ? w1[k * w1_stride + 1] * s1 : 0.f;
        dst[2 * hp + k] = in ? b1[k] * s1 : 0.f;
        dst[3 * hp + k] = in ? w2[k] * s2 : 0.f;
    }
}


// Softplus MLP on up to D edges of one node, 4 at a time (second block only when d > 4).
template <bool TWO_IN, int D>
__device__ __forceinline__ void mlp_softplus_blocks(const MlpSmem& W, int hp, int d, const float (&x0)[D],
                                                    const float (&x1)[D], float (&out)[D]) {
    float a[4], b[4], o[4];
#pragma unroll
    for (int blk = 0; blk < D; blk += 4) {
        if (blk == 0 || d > blk) {
#pragma unroll
            for (int j = 0; j < 4; ++j) { a[j] = x0[blk + j]; b[j] = x1[blk + j]; }
            mlp_softplus_x2<4, TWO_IN, 2>(W, hp, a, b, o);   // packed f32x2 + FMA-pipe polynomial lg2 (see gd_math.cuh)
#pragma unroll
            for (int j = 0; j < 4; ++j) out[blk + j] = o[j];
        }
    }
}

// VD / CD: register batch sizes (4 or 8) for variable / check nodes = the graph's max degrees rounded
// up; larger degrees take the generic loops.  VSORT: edges are sorted by variable (the canonical
// H.to_sparse() order), so a variable's edges are the contiguous rows var_ptr[v] .. var_ptr[v+1]-1.
template <int PROG, int VD, int CD, bool VSORT>
__global__ void __launch_bounds__(1024, 1) decode_streamed_kernel(const StreamParams p) {
    extern __shared__ __align__(16) float wsm[];
    constexpr bool kIsBP = (PROG == GD_PROG_BP_QUANTUM || PROG == GD_PROG_BP_CLASSICAL);
    constexpr bool kSoftplus = (PROG == GD_PROG_V2_4);
    const int tile = p.tile, R = p.R, E = p.E, V = p.V, C = p.C, N = p.N, hp = p.hp;
    const int tid = threadIdx.x, nthr = blockDim.x;
    const int s = tid % tile, r = tid / tile;
    float* xT = p.slab + (size_t)blockIdx.x * p.slab_floats;
    float* m_st = xT + (size_t)N * tile;
    float* t_st = m_st + (size_t)E * tile;
    const GraphTables tb = p.tb;

    MlpSmem W1{}, W2{}, W3{};
    if constexpr (!kIsBP) {
        const float* w = p.weights;
        const int h = p.hid;
        const float s1 = kSoftplus ? kLog2e : 1.f, s2 = kSoftplus ? kLn2 : 1.f;
        float* slot = wsm;
        if constexpr (PROG == GD_PROG_V2_4) {
            stage_mlp_s(slot, hp, h, w, 2, true, w + 2 * h, w + 3 * h, s1, s2, tid, nthr);
            W1 = MlpSmem{slot, slot + hp, slot + 2 * hp, slot + 3 * hp, w[4 * h]};
            w += 4 * h + 1;
            slot += 4 * hp;
        }
        stage_mlp_s(slot, hp, h, w, 1, false, w + h, w + 2 * h, s1, s2, tid, nthr);
        W2 = MlpSmem{slot, slot + hp, slot + 2 * hp, slot + 3 * hp, w[3 * h]};
        w += 3 * h + 1;
        slot += 4 * hp;
        stage_mlp_s(slot, hp, h, w, 1, false, w + h, w + 2 * h, s1, s2, tid, nthr);
        W3 = MlpSmem{slot, slot + hp, slot + 2 * hp, slot + 3 * hp, w[3 * h]};
    }
    __syncthreads();
    // V2_4: the two 1 -> h -> 1 MLPs as cubic tables on their compact domains (gd_math.cuh CubicTab; same scheme
    // as the resident kernel, DESIGN.md 4.1)
    CubicTab ctab{}, rtab{};
    bool use_ctab = false, use_rtab = false;
    float rtab_R = 0.f;
    if constexpr (PROG == GD_PROG_V2_4) {
        if (p.ctab_n > 0) {
            float* tabs = wsm + 3 * 4 * hp;
            float4* cdst = reinterpret_cast<float4*>(tabs);
            float4* rdst = cdst + p.ctab_n;
            float* F = reinterpret_cast<float*>(rdst + p.rtab_n);
            unsigned int* fmax_bits = reinterpret_cast<unsigned int*>(F + (p.ctab_n > p.rtab_n ? p.ctab_n : p.rtab_n) + 8);
            const float step = 2.0f * p.ctab_R / (float)p.ctab_n;
            use_ctab = cubic_tab_bound(p.weights + 4 * p.hid + 1, p.hid, step) <= 1e-7f;
            if (use_ctab) {
                const float fm = cubic_tab_build(W2, hp, p.ctab_R, p.ctab_n, cdst, F, tid, nthr);
                ctab = CubicTab{cdst, 1.0f / step, p.ctab_R / step, (float)p.ctab_n - 0.001f};
                if (p.rtab_n > 0 && p.T > 0) {
                    if (tid == 0) *fmax_bits = 0u;
                    __syncthreads();
                    atomicMax(fmax_bits, __float_as_uint(fm));
                    __syncthreads();
                    rtab_R = (float)p.T * (__uint_as_float(*fmax_bits) * 1.02f + 1e-6f);
                    const float rstep = 2.0f * rtab_R / (float)p.rtab_n;
                    use_rtab = cubic_tab_bound(p.weights + 7 * p.hid + 2, p.hid, rstep) <= 4e-6f;
                    if (use_rtab) {
                        cubic_tab_build(W3, hp, rtab_R, p.rtab_n, rdst, F, tid, nthr);
                        rtab = CubicTab{rdst, 1.0f / rstep, rtab_R / rstep, (float)p.rtab_n - 0.001f};
                    }
                }
            }
        }
    }

    for (int tix = blockIdx.x; tix < p.n_tiles; tix += gridDim.x) {
        const long long s0 = (long long)tix * tile;
        const int nvalid = (int)min((long long)tile, p.B - s0);
        // ---- transpose the input slab x[tile][N] -> xT[N][tile] (coalesced reads), zero m ----
        for (int i = tid; i < tile * N; i += nthr) {
            const int si = i / N, n = i - si * N;
            xT[(size_t)n * tile + si] = si < nvalid ? __ldg(p.x + s0 * N + i) : 0.f;
        }
        for (int e = r; e < E; e += R) m_st[(size_t)e * tile + s] = 0.f;
        __syncthreads();

        for (int it = 0; it < p.T; ++it) {
            // ---- variable phase: owner of variable v ----
            for (int v = r; v < V; v += R) {
                const int b = __ldg(tb.var_ptr + v), d = __ldg(tb.var_ptr + v + 1) - b;
                const float prior = xT[(size_t)v * tile + s];
                if (d <= VD) {
                    // batched: issue all loads of the node first (memory-level parallelism), then compute
                    uint32_t at[VD];
                    float val[VD], res[VD], pr[VD];
#pragma unroll
                    for (int k = 0; k < VD; ++k) {
                        const int kk = k < d ? k : 0;
                        at[k] = (uint32_t)(VSORT ? b + kk : __ldg(tb.var_edges + b + kk)) * tile + s;
                    }
#pragma unroll
                    for (int k = 0; k < VD; ++k) val[k] = k < d ? m_st[at[k]] : 0.f;
                    float acc = 0.f;
#pragma unroll
                    for (int k = 0; k < VD; ++k) acc += val[k];        // ascending edge id; padded slots add 0
#pragma unroll
                    for (int k = 0; k < VD; ++k) { val[k] = acc - val[k]; pr[k] = prior; }
                    if constexpr (PROG == GD_PROG_V2_4) {
                        mlp_softplus_blocks<true, VD>(W1, hp, d, val, pr, res);
#pragma unroll
                        for (int k = 0; k < VD; ++k) if (k < d) t_st[at[k]] = tanh_half_fast(res[k]);
                    } else {
#pragma unroll
                        for (int k = 0; k < VD; ++k) if (k < d) {
                            const float a = val[k] + prior;
                            if constexpr (kIsBP) {
                                t_st[at[k]] = bp_log_abs_tanh_half(a, PROG == GD_PROG_BP_QUANTUM ? -46.0517019f : -16.1180957f);
                                m_st[at[k]] = a < 0.f ? 1.f : 0.f;
                            } else {
                                t_st[at[k]] = tanh_half_fast(a);
                            }
                        }
                    }
                } else {
                    const int e_end = b + d;
                    float acc = 0.f;
                    for (int i = b; i < e_end; ++i) acc += m_st[(size_t)__ldg(tb.var_edges + i) * tile + s];
                    for (int i = b; i < e_end; ++i) {
                        const size_t at1 = (size_t)__ldg(tb.var_edges + i) * tile + s;
                        const float ext = acc - m_st[at1];
                        if constexpr (PROG == GD_PROG_V2_4) {
                            float a0[1] = {ext}, a1[1] = {prior}, o[1];
                            mlp_softplus<1, true>(W1, hp, a0, a1, o);
                            t_st[at1] = tanh_half_fast(o[0]);
                        } else if constexpr (kIsBP) {
                            const float a = ext + prior;
                            t_st[at1] = bp_log_abs_tanh_half(a, PROG == GD_PROG_BP_QUANTUM ? -46.0517019f : -16.1180957f);
                            m_st[at1] = a < 0.f ? 1.f : 0.f;   // sign flag; this variable's sum is already taken
                        } else {
                            t_st[at1] = tanh_half_fast(ext + prior);
                        }
                    }
                }
            }
            __syncthreads();
            // ---- check phase: owner of check c ----
            for (int c = r; c < C; c += R) {
                const int b = __ldg(tb.chk_ptr + c), d = __ldg(tb.chk_ptr + c + 1) - b;
                const float sg = PROG == GD_PROG_CGNNI || PROG == GD_PROG_BP_CLASSICAL ? 1.f : xT[(size_t)(V + c) * tile + s];
                if (d <= CD) {
                    uint32_t at[CD];
                    float val[CD], old[CD], res[CD];
#pragma unroll
                    for (int k = 0; k < CD; ++k) at[k] = (uint32_t)__ldg(tb.chk_edges + b + (k < d ? k : 0)) * tile + s;
#pragma unroll
                    for (int k = 0; k < CD; ++k) { val[k] = k < d ? t_st[at[k]] : 0.f; old[k] = k < d ? m_st[at[k]] : 0.f; }
                    float acc = 0.f, cnt = 0.f;
#pragma unroll
                    for (int k = 0; k < CD; ++k) { acc += val[k]; if constexpr (kIsBP) cnt += old[k]; }
#pragma unroll
                    for (int k = 0; k < CD; ++k) val[k] = acc - val[k];
                    if constexpr (kIsBP) {
#pragma unroll
                        for (int k = 0; k < CD; ++k) if (k < d) {
                            int q = (int)(cnt - old[k]);
                            if constexpr (PROG == GD_PROG_BP_QUANTUM) q += sg < 0.f ? 1 : 0;
                            m_st[at[k]] = bp_check_out(val[k], q & 1, PROG == GD_PROG_BP_QUANTUM ? 1e-12f : 1e-7f);
                        }
                    } else {
                        if (kSoftplus && use_ctab) {
#pragma unroll
                            for (int k = 0; k < CD; ++k) res[k] = cubic_tab_eval(ctab, val[k]);
                        } else if constexpr (kSoftplus) mlp_softplus_blocks<false, CD>(W2, hp, d, val, val, res);
                        else mlp_relu<CD>(W2, hp, val, res);
#pragma unroll
                        for (int k = 0; k < CD; ++k) if (k < d) m_st[at[k]] = res[k] * sg + old[k];
                    }
                } else {
                    const int e_end = b + d;
                    float acc = 0.f, cnt = 0.f;
                    for (int i = b; i < e_end; ++i) {
                        const size_t at1 = (size_t)__ldg(tb.chk_edges + i) * tile + s;
                        acc += t_st[at1];
                        if constexpr (kIsBP) cnt += m_st[at1];
                    }
                    for (int i = b; i < e_end; ++i) {
                        const size_t at1 = (size_t)__ldg(tb.chk_edges + i) * tile + s;
                        const float ext = acc - t_st[at1];
                        if constexpr (kIsBP) {
                            int q = (int)(cnt - m_st[at1]);
                            if constexpr (PROG == GD_PROG_BP_QUANTUM) q += sg < 0.f ? 1 : 0;
                            m_st[at1] = bp_check_out(ext, q & 1, PROG == GD_PROG_BP_QUANTUM ? 1e-12f : 1e-7f);
                        } else {
                            float a0[1] = {ext}, o[1];
                            if (kSoftplus && use_ctab) o[0] = cubic_tab_eval(ctab, ext);
                            else if constexpr (kSoftplus) mlp_softplus<1, false>(W2, hp, a0, a0, o);
                            else mlp_relu<1>(W2, hp, a0, o);
                            m_st[at1] = o[0] * sg + m_st[at1];
                        }
                    }
                }
            }
            __syncthreads();
        }
        // ---- read-out (variable owner) ----
        constexpr bool kClamp = (PROG == GD_PROG_CGNNI || PROG == GD_PROG_BP_CLASSICAL);
        for (int v = r; v < V; v += R) {
            const int b = __ldg(tb.var_ptr + v), e_end = __ldg(tb.var_ptr + v + 1);
            float acc = 0.f;
            for (int i = b; i < e_end; ++i) {
                const float mv = m_st[(size_t)__ldg(tb.var_edges + i) * tile + s];
                if constexpr (PROG == GD_PROG_V2_4) {
                    float a0[1] = {mv}, o[1];
                    if (use_rtab && fabsf(mv) <= rtab_R) o[0] = cubic_tab_eval(rtab, mv);
                    else mlp_softplus<1, false>(W3, hp, a0, a0, o);
                    acc += o[0];
                } else {
                    acc += mv;
                }
            }
            float lg = acc + xT[(size_t)v * tile + s];
            if constexpr (PROG == GD_PROG_CGNNI || PROG == GD_PROG_QGNNI) {
                float xi[1] = {lg}, oo[1];
                mlp_relu<1>(W3, hp, xi, oo);
                lg = oo[0];
            }
            if (s < nvalid) {
                float pr = sigmoid_neg(lg);
                if (kClamp) pr = fminf(fmaxf(pr, 1e-7f), 1.0f - 1e-7f);
                const long long o = (s0 + s) * V + v;
                if (p.prob) p.prob[o] = pr;
                if (p.logit) p.logit[o] = lg;
                if (p.hard) p.hard[o] = pr > 0.5f;
            }
        }
        __syncthreads();
    }
}

int plan_streamed(const gd_graph* g, const gd_model* m, int64_t B, StreamPlan* out) {
    const bool bp = m->program == GD_PROG_BP_QUANTUM || m->program == GD_PROG_BP_CLASSICAL;
    StreamParams& p = out->p;
    memset(&p, 0, sizeof(p));
    p.B = B; p.T = m->iters; p.V = g->V; p.C = g->C; p.E = (int)g->E; p.N = g->N;
    p.hid = bp ? 0 : m->hidden; p.hp = (p.hid + 7) / 8 * 8; p.tb = g->t;
    const int n_slots = bp ? 0 : (m->program == GD_PROG_V2_4 ? 3 : 2);
    out->smem = n_slots * 4 * p.hp * 4 + 16;
    if (m->program == GD_PROG_V2_4 && !opt_on(OPT_NO_CTAB)) {
        p.ctab_n = 512;
        p.rtab_n = 2048;
        p.ctab_R = (float)(g->max_chk_deg > 1 ? g->max_chk_deg - 1 : 1);
        const int big = p.ctab_n > p.rtab_n ? p.ctab_n : p.rtab_n;
        out->smem += (p.ctab_n + p.rtab_n) * 16 + (big + 8) * 4 + 16;
    }
    // tile: multiple of 8 (32-byte sectors stay whole) that wastes the fewest tile slots over the rounds
    int tile = 32;
    {
        double best = -1.0;
        for (int t = 24; t <= 128; t += 8) {
            const int64_t n_t = (B + t - 1) / t;
            const int64_t rounds = (n_t + g->sm_count - 1) / g->sm_count;
            const double eff = (double)B / ((double)rounds * g->sm_count * t) * (t % 32 == 0 ? 1.0 : 0.97);
            if (eff > best + 1e-9) { best = eff; tile = t; }
        }
    }
    p.tile = tile;
    const int maxthr = 1024;
    int R = maxthr / tile;
    const int maxn = g->V > g->C ? g->V : g->C;
    if (R > maxn) R = maxn;
    if (R < 1) R = 1;
    while (R > 1 && (R * tile) % 32) --R;
    if ((R * tile) % 32) { tile = 32; p.tile = 32; R = maxthr / 32; }
    p.R = R;
    out->threads = R * tile;
    p.n_tiles = (int)((B + tile - 1) / tile);
    out->grid = p.n_tiles < g->sm_count ? p.n_tiles : g->sm_count;
    p.slab_floats = ((long long)g->N + 2 * g->E) * tile;
    return GD_OK;
}

int streamed_decode(gd_graph* g, const StreamPlan& plan, const gd_model* model, const DecodeIO& io, cudaStream_t st) {
    StreamPlan pl = plan;
    pl.p.x = io.x; pl.p.prob = io.prob; pl.p.logit = io.logit; pl.p.hard = io.hard; pl.p.weights = io.weights;
    pl.p.slab = streamed_slab(g, (size_t)pl.grid * (size_t)pl.p.slab_floats * sizeof(float));
    if (!pl.p.slab) return GD_ERR_CUDA;
    void (*k)(const StreamParams);
    const bool v8 = g->max_var_deg > 4, c8 = g->max_chk_deg > 4;
    bool vsort = true;
    for (size_t i = 0; i < g->h_var_edges.size() && vsort; ++i) vsort = g->h_var_edges[i] == (int32_t)i;
#define GD_SK(P)                                                                                         \
    (vsort ? (v8 ? (c8 ? decode_streamed_kernel<P, 8, 8, true> : decode_streamed_kernel<P, 8, 4, true>)  \
                 : (c8 ? decode_streamed_kernel<P, 4, 8, true> : decode_streamed_kernel<P, 4, 4, true>)) \
           : (c8 ? decode_streamed_kernel<P, 8, 8, false> : decode_streamed_kernel<P, 8, 4, false>))
    switch (model->program) {
        case GD_PROG_CGNNI: k = GD_SK(GD_PROG_CGNNI); break;
        case GD_PROG_QGNNI: k = GD_SK(GD_PROG_QGNNI); break;
        case GD_PROG_V2_4: k = GD_SK(GD_PROG_V2_4); break;
        case GD_PROG_BP_QUANTUM: k = GD_SK(GD_PROG_BP_QUANTUM); break;
        default: k = GD_SK(GD_PROG_BP_CLASSICAL); break;
    }
#undef GD_SK
    if (pl.smem > 48 * 1024) GD_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, pl.smem));
    k<<<pl.grid, pl.threads, pl.smem, st>>>(pl.p);
    GD_CUDA(cudaGetLastError());
    return GD_OK;
}

}  // namespace gd
