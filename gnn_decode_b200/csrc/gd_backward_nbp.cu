// Backward of neural BP (quantum/neural_BP.py, training; decoder_v1_1 runs the same program with per-edge weights gathered
// from its type tables): gradient of a loss w.r.t. the (2T+2)E + 1 weights, given dL/dlogit [B, V].
//
// Forward, per syndrome, layer l = 0 .. T-1, edge e = (v, c), s_c the check input ±1, pi_v the prior:
//   q_e = W_l[e] m^l_e,  u_e = sum_{e' in v, e' != e} q_e' + W_p,l[e] pi_v,
//   L_e = log clamp(|tanh(u_e/2)|, 1e-20),  S_e = sum_{e' in c, e' != e} L_e',  sigma_e = ± (parity of the siblings and s_c),
//   m^{l+1}_e = log(1+o_e) - log(1-o_e) + alpha m^l_e,  o_e = clamp(sigma_e e^{S_e}, -1+1e-15, 1-1e-15);
//   logit_v = sum_{e in v} (W[e] m^T_e + W_p[e] pi_v).
// Backward, g = dL/dm^{l+1}, from g_e = dlogit_v W[e] (dW[e] = sum_b dlogit_v m^T_e, dW_p[e] = sum_b dlogit_v pi_v):
//   dalpha += g_e m^l_e,  dS_e = g_e sigma_e / sinh(-S_e),  dL_e = sum_{e' in c, e' != e} dS_e',  du_e = dL_e / sinh(u_e),
//   dW_p,l[e] += du_e pi_v,  dq_e = sum_{e' in v, e' != e} du_e',  dW_l[e] += dq_e m^l_e,  g_e <- alpha g_e + W_l[e] dq_e.
// (the clamps pass nothing where they bind; the parity carries no gradient).  oracle/nbp_grad.py states the same in fp64.
//
// The forward (decode_streamed_tma_kernel<GD_PROG_NEURAL_BP, 0, true>) stashes m^1 .. m^T, [T][E][B].  Everything else is
// recomputed here with the forward's device code in the forward's order (NodeMath::nbp_u / nbp_t, the exclusive sums), so
// every clamp decision and sign parity is the forward's.
//
// Mapping: the streamed kernel's.  A lane owns four syndromes of the CTA's tile, a warp owns whole nodes, and the state of a
// tile lives in batch-minor rows [.][tile] of a per-CTA slab of the caller's workspace:
//   xT[N] | dlogit[V] | m^l[E] | L, then dL[E] | dS (checks past the unrolled degrees), then du[E] | g[E].
// Per layer: load m^l; variable owners recompute L; check owners form dS and dL; variable owners form du, dq, the weight
// gradients and the next g.  Rows are read with plain 128-bit loads (through L2): the slab is written and read by the same CTA.
//
// Weight gradients: for each (layer, edge) the owner warp sums over its tile's syndromes in registers in a fixed order (four per
// lane, then a fixed shuffle tree) and lane 0 adds the sum to the CTA's record in the workspace -- the record's only writer,
// visiting its tiles in a fixed order.  dalpha is accumulated per lane in double.  nbp_reduce_kernel sums the records in a fixed
// order in double.  No floating-point atomics: bit-reproducible run to run.
#include "gd_common.cuh"
#include "gd_math.cuh"
#include "gd_decode.cuh"
#include "gd_nodemath.cuh"
#include <string.h>

namespace gd {

using NbpMath = NodeMath<GD_PROG_NEURAL_BP, 0>;
constexpr int kNbpBwdThreads = 512;
constexpr int kNbpBwdWarps = kNbpBwdThreads / 32;

struct NbpBwdParams {
    const float* x;
    const float* stash;          // [T][E][B]: m^1 .. m^T
    const float* grad_logit;     // [B][V]
    const float* weights;        // packed order of gd_model (include/gnn_decode.h)
    GraphTables tb;
    float* slab;                 // per CTA: slab_floats
    float* records;              // per CTA: rec_floats = (2T+2)E weight gradients, rounded up to 4
    double* alpha_parts;         // per warp of every CTA: its share of dL/dalpha
    long long B;
    long long slab_floats;
    int rec_floats;
    int T, V, C, E, N, tile, lanes, n_tiles;
};

static __device__ __forceinline__ float4 ldcg4(const float* p) { return __ldcg(reinterpret_cast<const float4*>(p)); }

// this lane's four values summed, then over the warp in a fixed butterfly order (lane 0's result is used); lanes past the tile
// give 0.  Every lane of the warp calls it.
static __device__ __forceinline__ float warp_sum4(const float (&v)[4], bool active) {
    float s = active ? (v[0] + v[1]) + (v[2] + v[3]) : 0.f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    return s;
}

// the sign row's share of the parity (neural_BP.py:116: (1 - s_c) / 2), as NodeMath::nbp_sign_count
static __device__ __forceinline__ void nbp_sign_row(const float* srow, int (&cnt)[4]) {
    const float4 s4 = ldcg4(srow);
    cnt[0] = s4.x < 0.f ? 1 : 0; cnt[1] = s4.y < 0.f ? 1 : 0; cnt[2] = s4.z < 0.f ? 1 : 0; cnt[3] = s4.w < 0.f ? 1 : 0;
}

// dS of one edge: g sigma / sinh(-S), the parity without the edge's own flag (as nbp_chk_out takes it)
static __device__ __forceinline__ void nbp_edge_ds(const float (&ext)[4], const float4 tv, const int (&cnt)[4], const float4 g4, float (&ds)[4]) {
    const float t4[4] = {tv.x, tv.y, tv.z, tv.w}, g[4] = {g4.x, g4.y, g4.z, g4.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int q = cnt[j] - (t4[j] > 0.f ? 1 : 0);
        ds[j] = g[j] * bp_dcheck_out(ext[j], q & 1, NbpMath::kEps2);
    }
}

// check owner, degree D, in registers: L rows (t_r) -> dL rows (in place)
template <int D>
static __device__ __forceinline__ void nbp_bwd_chk_node(float* t_r, const float* g_r, const int32_t* edges, const float* srow, int tile,
                                             int l4, bool active) {
    size_t e[D];
    float4 tv[D];
#pragma unroll
    for (int k = 0; k < D; ++k) {
        e[k] = (size_t)__ldg(edges + k) * tile + l4;
        tv[k] = ldcg4(t_r + e[k]);
    }
    int cnt[4];
    nbp_sign_row(srow, cnt);
    float ext[D][4];
    NbpMath::nbp_exclusive<D>(tv, ext, cnt);
    float ds[D][4];
#pragma unroll
    for (int k = 0; k < D; ++k) nbp_edge_ds(ext[k], tv[k], cnt, ldcg4(g_r + e[k]), ds[k]);
    // dL = exclusive sums of dS, prefix + suffix (dS spans many orders of magnitude: no "all minus own")
    float run[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int k = 0; k < D; ++k)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float v = ds[k][j];
            ds[k][j] = run[j];
            run[j] += v;
            ext[k][j] = v;                 // (ext is dead: it keeps dS for the suffix pass)
        }
    run[0] = run[1] = run[2] = run[3] = 0.f;
#pragma unroll
    for (int k = D - 1; k >= 0; --k) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            ds[k][j] += run[j];
            run[j] += ext[k][j];
        }
        if (active) stg4(t_r + e[k], ds[k]);
    }
}

// check owner, any degree (past the unrolled ones): dS of every edge to d_r, then each dL directly, O(d^2)
static __device__ void nbp_bwd_chk_any(float* t_r, float* d_r, const float* g_r, const int32_t* edges, const float* srow, int tile, int l4,
                            bool active, int d) {
    int cnt[4];
    nbp_sign_row(srow, cnt);
    for (int k = 0; k < d; ++k) {
        const float4 tv = ldcg4(t_r + (size_t)__ldg(edges + k) * tile + l4);
        cnt[0] += tv.x > 0.f ? 1 : 0; cnt[1] += tv.y > 0.f ? 1 : 0; cnt[2] += tv.z > 0.f ? 1 : 0; cnt[3] += tv.w > 0.f ? 1 : 0;
    }
    const auto row = [&](int i) { return ldcg4(t_r + (size_t)__ldg(edges + i) * tile + l4); };
    for (int k = 0; k < d; ++k) {
        const size_t ek = (size_t)__ldg(edges + k) * tile + l4;
        float ext[4], ds[4];
        NbpMath::nbp_exclusive_any(row, d, k, ext);
        nbp_edge_ds(ext, ldcg4(t_r + ek), cnt, ldcg4(g_r + ek), ds);
        if (active) stg4(d_r + ek, ds);
    }
    for (int k = 0; k < d; ++k) {
        float dl[4] = {0.f, 0.f, 0.f, 0.f};
        for (int i = 0; i < d; ++i) {
            if (i == k) continue;
            const float4 v = ldcg4(d_r + (size_t)__ldg(edges + i) * tile + l4);
            dl[0] += v.x; dl[1] += v.y; dl[2] += v.z; dl[3] += v.w;
        }
        if (active) stg4(t_r + (size_t)__ldg(edges + k) * tile + l4, dl);
    }
}

__global__ void __launch_bounds__(kNbpBwdThreads, 1) nbp_bwd_kernel(const NbpBwdParams p) {
    const int tile = p.tile, E = p.E, V = p.V, C = p.C, N = p.N, T = p.T;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const bool active = lane < p.lanes;
    const int l4 = active ? lane * 4 : 0;
    const GraphTables tb = p.tb;
    float* const xT = p.slab + (size_t)blockIdx.x * p.slab_floats;
    float* const dlg = xT + (size_t)N * tile;
    float* const m_r = dlg + (size_t)V * tile;
    float* const t_r = m_r + (size_t)E * tile;
    float* const d_r = t_r + (size_t)E * tile;
    float* const g_r = d_r + (size_t)E * tile;
    float* const rec = p.records + (size_t)blockIdx.x * p.rec_floats;
    const float alpha = __ldg(p.weights + (size_t)(2 * T + 2) * E);
    for (int i = tid; i < p.rec_floats; i += kNbpBwdThreads) rec[i] = 0.f;
    double dalpha = 0.0;

    // m^l of the tile's syndromes -> m_r (m^0 = 0; rows past the batch are 0)
    auto load_m = [&](int l, long long s0, int nvalid) {
        const float* src = p.stash + (size_t)(l > 0 ? l - 1 : 0) * E * p.B + s0;
        for (int i = tid; i < E * tile; i += kNbpBwdThreads) {
            const int e = i / tile, si = i - e * tile;
            m_r[i] = (l > 0 && si < nvalid) ? __ldcg(src + (size_t)e * p.B + si) : 0.f;
        }
    };
    // u of this variable's edges needs the sum over all of them of W_l m^l, ascending edge id (the forward's order)
    auto var_acc = [&](const float* wl, int b, int d, bool with_m, float (&acc)[4]) {
        acc[0] = acc[1] = acc[2] = acc[3] = 0.f;
        if (with_m)
            for (int k = 0; k < d; ++k) {
                const float4 mv = ldcg4(m_r + (size_t)(b + k) * tile + l4);
                const float wk = __ldg(wl + b + k);
                acc[0] = fmaf(mv.x, wk, acc[0]); acc[1] = fmaf(mv.y, wk, acc[1]);
                acc[2] = fmaf(mv.z, wk, acc[2]); acc[3] = fmaf(mv.w, wk, acc[3]);
            }
    };

    for (int tix = blockIdx.x; tix < p.n_tiles; tix += gridDim.x) {
        const long long s0 = (long long)tix * tile;
        const int nvalid = (int)min((long long)tile, p.B - s0);
        for (int i = tid; i < tile * N; i += kNbpBwdThreads) {
            const int si = i / N, n = i - si * N;
            xT[(size_t)n * tile + si] = si < nvalid ? __ldg(p.x + (size_t)(s0 + si) * N + n) : 0.f;
        }
        for (int i = tid; i < tile * V; i += kNbpBwdThreads) {
            const int si = i / V, v = i - si * V;
            dlg[(size_t)v * tile + si] = si < nvalid ? __ldg(p.grad_logit + (size_t)(s0 + si) * V + v) : 0.f;
        }
        load_m(T, s0, nvalid);
        __syncthreads();

        // ---- read-out (neural_BP.py:308-312): g = dlogit W, dW += dlogit m^T, dW_p += dlogit prior ----
        {
            const float* wr = p.weights + (size_t)2 * T * E;
            for (int v = w; v < V; v += kNbpBwdWarps) {
                const int b = __ldg(tb.var_ptr + v), d = __ldg(tb.var_ptr + v + 1) - b;
                const float4 dl4 = ldcg4(dlg + (size_t)v * tile + l4), pr4 = ldcg4(xT + (size_t)v * tile + l4);
                const float dl[4] = {dl4.x, dl4.y, dl4.z, dl4.w};
                const float dp[4] = {dl4.x * pr4.x, dl4.y * pr4.y, dl4.z * pr4.z, dl4.w * pr4.w};
                const float sdp = d > 0 ? warp_sum4(dp, active) : 0.f;
                for (int k = 0; k < d; ++k) {
                    const size_t e = (size_t)(b + k);
                    const float4 m4 = ldcg4(m_r + e * tile + l4);
                    const float wk = __ldg(wr + e);
                    const float gm[4] = {dl[0] * m4.x, dl[1] * m4.y, dl[2] * m4.z, dl[3] * m4.w};
                    const float gg[4] = {dl[0] * wk, dl[1] * wk, dl[2] * wk, dl[3] * wk};
                    const float sgm = warp_sum4(gm, active);
                    if (active) stg4(g_r + e * tile + l4, gg);
                    if (lane == 0) {
                        rec[(size_t)2 * T * E + e] += sgm;
                        rec[(size_t)(2 * T + 1) * E + e] += sdp;
                    }
                }
            }
        }
        __syncthreads();

        for (int l = T - 1; l >= 0; --l) {
            load_m(l, s0, nvalid);
            __syncthreads();
            const float* wl = p.weights + (size_t)l * 2 * E;
            const bool with_m = l > 0;
            // ---- variable owner: L of every edge, the forward's variable phase ----
            for (int v = w; v < V; v += kNbpBwdWarps) {
                const int b = __ldg(tb.var_ptr + v), d = __ldg(tb.var_ptr + v + 1) - b;
                const float4 pr4 = ldcg4(xT + (size_t)v * tile + l4);
                const float prv[4] = {pr4.x, pr4.y, pr4.z, pr4.w};
                float acc[4];
                var_acc(wl, b, d, with_m, acc);
                for (int k = 0; k < d; ++k) {
                    const size_t e = (size_t)(b + k);
                    const float wk = __ldg(wl + e), wpk = __ldg(wl + E + e);
                    float4 mv = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (with_m) mv = ldcg4(m_r + e * tile + l4);
                    const float m4[4] = {mv.x, mv.y, mv.z, mv.w};
                    float out[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) out[j] = NbpMath::nbp_t(NbpMath::nbp_u(acc[j], m4[j], wk, prv[j], wpk));
                    if (active) stg4(t_r + e * tile + l4, out);
                }
            }
            __syncthreads();
            // ---- check owner: dS, then dL = the exclusive sums of dS over the check ----
            for (int c = w; c < C; c += kNbpBwdWarps) {
                const int b = __ldg(tb.chk_ptr + c), d = __ldg(tb.chk_ptr + c + 1) - b;
                const int32_t* edges = tb.chk_edges + b;
                const float* srow = xT + (size_t)(V + c) * tile + l4;
#define GD_NBP_BWD_CHK(D) nbp_bwd_chk_node<D>(t_r, g_r, edges, srow, tile, l4, active)
                GD_DEGREE_SWITCH(d, GD_NBP_BWD_CHK, nbp_bwd_chk_any(t_r, d_r, g_r, edges, srow, tile, l4, active, d))
#undef GD_NBP_BWD_CHK
            }
            __syncthreads();
            // ---- variable owner: du, dq, the weight gradients of layer l and alpha, g <- alpha g + W_l dq ----
            for (int v = w; v < V; v += kNbpBwdWarps) {
                const int b = __ldg(tb.var_ptr + v), d = __ldg(tb.var_ptr + v + 1) - b;
                const float4 pr4 = ldcg4(xT + (size_t)v * tile + l4);
                const float prv[4] = {pr4.x, pr4.y, pr4.z, pr4.w};
                float acc[4];
                var_acc(wl, b, d, with_m, acc);
                for (int k = 0; k < d; ++k) {
                    const size_t e = (size_t)(b + k);
                    const float wk = __ldg(wl + e), wpk = __ldg(wl + E + e);
                    float4 mv = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (with_m) mv = ldcg4(m_r + e * tile + l4);
                    const float m4[4] = {mv.x, mv.y, mv.z, mv.w};
                    const float4 dl4 = ldcg4(t_r + e * tile + l4);
                    const float dl[4] = {dl4.x, dl4.y, dl4.z, dl4.w};
                    float du[4], dup[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float u = NbpMath::nbp_u(acc[j], m4[j], wk, prv[j], wpk);
                        du[j] = dl[j] * bp_dlog_abs_tanh_half(u, bp_log_abs_tanh_half<false>(u, NbpMath::kLogEps1), NbpMath::kLogEps1);
                        dup[j] = du[j] * prv[j];
                    }
                    if (active) stg4(d_r + e * tile + l4, du);
                    const float s = warp_sum4(dup, active);
                    if (lane == 0) rec[(size_t)(2 * l + 1) * E + e] += s;
                }
                for (int k = 0; k < d; ++k) {
                    const size_t e = (size_t)(b + k);
                    float dq[4] = {0.f, 0.f, 0.f, 0.f};
                    for (int i = 0; i < d; ++i) {                // ascending, the edge's own du left out
                        if (i == k) continue;
                        const float4 v4 = ldcg4(d_r + (size_t)(b + i) * tile + l4);
                        dq[0] += v4.x; dq[1] += v4.y; dq[2] += v4.z; dq[3] += v4.w;
                    }
                    float4 mv = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (with_m) mv = ldcg4(m_r + e * tile + l4);
                    const float m4[4] = {mv.x, mv.y, mv.z, mv.w};
                    const float4 g4 = ldcg4(g_r + e * tile + l4);
                    const float g[4] = {g4.x, g4.y, g4.z, g4.w};
                    const float wk = __ldg(wl + e);
                    float dqm[4], gn[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        dqm[j] = dq[j] * m4[j];
                        gn[j] = fmaf(alpha, g[j], wk * dq[j]);
                    }
                    if (active) {
                        dalpha += (double)((g[0] * m4[0] + g[1] * m4[1]) + (g[2] * m4[2] + g[3] * m4[3]));
                        stg4(g_r + e * tile + l4, gn);
                    }
                    const float s = warp_sum4(dqm, active);
                    if (lane == 0) rec[(size_t)2 * l * E + e] += s;
                }
            }
            __syncthreads();
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) dalpha += __shfl_xor_sync(0xffffffffu, dalpha, o);
    if (lane == 0) p.alpha_parts[(size_t)blockIdx.x * kNbpBwdWarps + w] = dalpha;
}

// the CTA records (and the per-warp alpha shares) summed in a fixed order in double -> the (2T+2)E + 1 gradients
__global__ void nbp_reduce_kernel(const float* __restrict__ records, int n_rec, int rec_floats, int n_w, const double* alpha_parts,
                                  float* __restrict__ grad, int accumulate) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n_w) return;
    double a = 0.0;
    if (i < n_w) {
        for (int r = 0; r < n_rec; ++r) a += (double)records[(size_t)r * rec_floats + i];
    } else {
        for (int q = 0; q < n_rec * kNbpBwdWarps; ++q) a += alpha_parts[q];
    }
    grad[i] = accumulate ? grad[i] + (float)a : (float)a;
}

struct NbpBwdPlan {
    NbpBwdParams p;
    int grid;
    int64_t off_records, off_slab;    // workspace offsets in floats (the alpha shares come first)
};

// The forward's tile and grid (plan_streamed_tma, which also refuses graphs outside the canonical edge order).
static int plan_nbp_bwd(const gd_graph* g, const gd_model* m, int64_t B, NbpBwdPlan* out) {
    StreamTmaPlan fp;
    plan_streamed_tma(g, m, B, &fp, true);
    if (!fp.ok) {
        set_error("gd_decode_bwd: the neural BP backward cannot take this graph: %s", fp.why);
        return GD_ERR_UNSUPPORTED;
    }
    NbpBwdParams& p = out->p;
    memset(&p, 0, sizeof(p));
    p.B = B; p.T = m->iters; p.V = g->V; p.C = g->C; p.E = (int)g->E; p.N = g->N;
    p.tb = g->t;
    p.tile = fp.p.tile; p.lanes = fp.p.lanes; p.n_tiles = fp.p.n_tiles;
    p.rec_floats = (int)(((2LL * p.T + 2) * p.E + 3) & ~3LL);
    p.slab_floats = ((long long)p.N + p.V + 4LL * p.E) * p.tile;
    out->grid = fp.grid;
    out->off_records = (int64_t)out->grid * kNbpBwdWarps * 2;
    out->off_slab = out->off_records + (int64_t)out->grid * p.rec_floats;
    return GD_OK;
}

int64_t nbp_bwd_workspace_floats(const gd_graph* g, const gd_model* model, int64_t B) {
    NbpBwdPlan pl;
    if (plan_nbp_bwd(g, model, B, &pl) != GD_OK) return -1;
    return pl.off_slab + (int64_t)pl.grid * pl.p.slab_floats;
}

int nbp_backward(const gd_graph* g, const gd_model* model, const float* weights_dev, const float* x_dev, const float* stash_dev,
                 const float* grad_logit_dev, float* grad_weights_dev, float* workspace_dev, int accumulate, int64_t B,
                 cudaStream_t st) {
    NbpBwdPlan pl;
    const int rc = plan_nbp_bwd(g, model, B, &pl);
    if (rc != GD_OK) return rc;
    GD_CHECK_ARG(((uintptr_t)workspace_dev & 15) == 0, "gd_decode_bwd: workspace must be 16-byte aligned");
    NbpBwdParams& p = pl.p;
    p.x = x_dev; p.stash = stash_dev; p.grad_logit = grad_logit_dev; p.weights = weights_dev;
    p.alpha_parts = reinterpret_cast<double*>(workspace_dev);
    p.records = workspace_dev + pl.off_records;
    p.slab = workspace_dev + pl.off_slab;
    nbp_bwd_kernel<<<pl.grid, kNbpBwdThreads, 0, st>>>(p);
    GD_CUDA(cudaGetLastError());
    const int n_w = (int)((2LL * p.T + 2) * p.E);
    nbp_reduce_kernel<<<(n_w + 1 + 255) / 256, 256, 0, st>>>(p.records, pl.grid, p.rec_floats, n_w, p.alpha_parts,
                                                            grad_weights_dev, accumulate);
    GD_CUDA(cudaGetLastError());
    return GD_OK;
}

}  // namespace gd
