// Backward of the CGNNI decoder (classical/CGNNI.py, training): gradient of a loss w.r.t. the 6h+2 MLP weights
// (ggc2.mlp2 | mlp), given dL/dlogit [B, V].  Replaces autograd through the reference's T x ~25 eager ops.
//
// Forward, per iteration it (m^0 = 0, edges in the canonical variable-sorted order):
//   a_e = sum_{e' in var(e), e' != e} m^it_e' + prior_v,   t_e = tanh(a_e / 2),
//   u_e = sum_{e' in chk(e), e' != e} t_e',                  m^{it+1}_e = f2(u_e) + m^it_e;
//   logit_v = f3(res_v),  res_v = sum_{e in v} m^T_e + prior_v.
// f2 / f3 are 1 -> h -> 1 ReLU MLPs, evaluated (forward and here) as the piecewise-linear tables of gd_math.cuh.
//
// Mapping: the node-owner mapping, tile geometry and [E][tile] shared layout of decode_light_kernel (gd_light.cuh).  The
// forward stashes m^{it+1} only (stash[it][E][B]); t is recomputed here with the forward's device code in the forward's
// order, so every u_e lands in the same table segment as in the forward.  Per tile:
//   read-out (variable owner): dres_v = dlogit_v S3(res_v), dm_e = dres_v(e);
//   it = T-1 .. 0: load m^it, recompute t;
//     check owner:    du_e = dm_e S2(u_e),  dt_e = sum of the other du of the check,  da_e = dt_e (1 - t_e^2) / 2;
//     variable owner: dm_e += sum of the other da of the variable (the residual carries the old dm_e).
// Weight gradients: between two breakpoints a ReLU MLP is one line with a fixed set of active units, so its weight gradient
// is determined by sum g and sum g x per segment.  Those bins are summed over the lane group in registers (a fixed shuffle
// tree), then added as 64-bit fixed-point integers into shared memory -- integer adds commute, so the result does not depend
// on the order the groups arrive in.  The fixed-point scale is 2^32 / 2^e, e the exponent of the CTA's largest |dlogit|:
// a power of two, so the loss scale does not change the relative resolution.  Every CTA writes its bins to the workspace;
// cgnni_contract_kernel sums them in a fixed order in double and contracts them with the weights (the active sets of
// pwl_build) into the 6h+2 gradients.  Bit-reproducible run to run.
#include "gd_common.cuh"
#include "gd_math.cuh"
#include "gd_light.cuh"
#include <string.h>

namespace gd {

// per-CTA record of the workspace, in 64-bit words: bins [f2: sum g | sum g x][f3: sum g | sum g x] x NPAD, then the scale
// exponent
static int light_bwd_record_words(int npad) { return 4 * npad + 1; }

// One lane group (the `lanes` threads that own one node, converged) adds its four syndromes' (seg, g, g x) to the bins.
template <int NPAD>
__device__ __forceinline__ void bins_add4(long long* bins, const int (&seg)[4], const float (&g)[4], const float (&x)[4],
                                          unsigned gmask, int lanes, bool leader, float scale) {
    unsigned present = 0u;
#pragma unroll
    for (int j = 0; j < 4; ++j) present |= g[j] != 0.f ? 1u << seg[j] : 0u;
    present = __reduce_or_sync(gmask, present);
    while (present) {
        const int s = __ffs(present) - 1;
        present &= present - 1u;
        float sg = 0.f, sgx = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (seg[j] == s) { sg += g[j]; sgx = fmaf(g[j], x[j], sgx); }
        for (int o = lanes >> 1; o > 0; o >>= 1) {
            sg += __shfl_xor_sync(gmask, sg, o);
            sgx += __shfl_xor_sync(gmask, sgx, o);
        }
        if (leader) {
            fx_add(bins + s, __float2ll_rn(sg * scale));
            fx_add(bins + NPAD + s, __float2ll_rn(sgx * scale));
        }
    }
}

struct BwdGroup {
    long long* bins;   // f2 bins of this CTA (shared)
    unsigned gmask;
    int lanes;
    bool leader;
    float scale;
};

// check owner, degree D, values in registers: t rows -> da rows (in place), bins of f2
template <int NPAD, int D>
__device__ __forceinline__ void bwd_chk_node(const PwlSmem& P2, float* t_l4, const float* dm_l4, int tile, const uint16_t* edges,
                                             const BwdGroup& bg) {
    int e[D];
#pragma unroll
    for (int k = 0; k < D; ++k) e[k] = edges[k] * tile;
    float4 tv[D];
#pragma unroll
    for (int k = 0; k < D; ++k) tv[k] = lds4(t_l4 + e[k]);
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int k = 0; k < D; ++k) {      // ascending edge id, as the forward
        acc[0] += tv[k].x; acc[1] += tv[k].y; acc[2] += tv[k].z; acc[3] += tv[k].w;
    }
    float du[D][4], dacc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int k = 0; k < D; ++k) {
        const float t4[4] = {tv[k].x, tv[k].y, tv[k].z, tv[k].w};
        const float4 d4 = lds4(dm_l4 + e[k]);
        const float dm[4] = {d4.x, d4.y, d4.z, d4.w};
        float u[4];
        int sg[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            u[j] = acc[j] - t4[j];
            sg[j] = pwl_segment<NPAD>(P2, u[j]);
            du[k][j] = dm[j] * P2.seg[sg[j]].x;
            dacc[j] += du[k][j];
        }
        bins_add4<NPAD>(bg.bins, sg, dm, u, bg.gmask, bg.lanes, bg.leader, bg.scale);
    }
#pragma unroll
    for (int k = 0; k < D; ++k) {
        const float t4[4] = {tv[k].x, tv[k].y, tv[k].z, tv[k].w};
        float da[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) da[j] = 0.5f * (dacc[j] - du[k][j]) * fmaf(-t4[j], t4[j], 1.0f);
        stg4(t_l4 + e[k], da);
    }
}

// variable owner, degree D: dm_e += sum of the other da of the variable
template <int D>
__device__ __forceinline__ void bwd_var_node(const float* da_rows, float* dm_rows, int tile) {
    float4 dv[D];
#pragma unroll
    for (int k = 0; k < D; ++k) dv[k] = lds4(da_rows + k * tile);
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int k = 0; k < D; ++k) {
        acc[0] += dv[k].x; acc[1] += dv[k].y; acc[2] += dv[k].z; acc[3] += dv[k].w;
    }
#pragma unroll
    for (int k = 0; k < D; ++k) {
        const float4 m4 = lds4(dm_rows + k * tile);
        const float out[4] = {m4.x + (acc[0] - dv[k].x), m4.y + (acc[1] - dv[k].y), m4.z + (acc[2] - dv[k].z),
                              m4.w + (acc[3] - dv[k].w)};
        stg4(dm_rows + k * tile, out);
    }
}

template <int NPAD>
__global__ void __launch_bounds__(512, 2) cgnni_bwd_light_kernel(const LightParams p, const float* __restrict__ grad_logit,
                                                                 long long* __restrict__ records, int off_dm, int off_bins) {
    extern __shared__ __align__(128) unsigned char smem[];
    using NM = NodeMath<GD_PROG_CGNNI, NPAD>;
    const int tile = p.tile, E = p.E, V = p.V, C = p.C, N = p.N, R = p.R;
    const int tid = threadIdx.x, nthr = blockDim.x;
    const int lg = tid % p.lanes, l4 = lg * 4, r = tid / p.lanes;
    const bool worker = r < R;
    float* const xT = reinterpret_cast<float*>(smem + p.off_x);
    float* const m_st = reinterpret_cast<float*>(smem + p.off_m);
    float* const t_st = reinterpret_cast<float*>(smem + p.off_t);
    float* const dm_st = reinterpret_cast<float*>(smem + off_dm);
    long long* const bins = reinterpret_cast<long long*>(smem + off_bins);   // [f2 | f3][sum g | sum g x][NPAD]
    unsigned int* const gmax = reinterpret_cast<unsigned int*>(bins + 4 * NPAD);
    uint16_t* const var_ptr = reinterpret_cast<uint16_t*>(smem + p.off_tab);
    uint16_t* const chk_ptr = var_ptr + (V + 1);
    uint16_t* const chk_edges = chk_ptr + (C + 1);
    for (int i = tid; i <= V; i += nthr) var_ptr[i] = (uint16_t)p.tb.var_ptr[i];
    for (int i = tid; i <= C; i += nthr) chk_ptr[i] = (uint16_t)p.tb.chk_ptr[i];
    for (int i = tid; i < E; i += nthr) chk_edges[i] = (uint16_t)p.tb.chk_edges[i];
    for (int i = tid; i < 4 * NPAD; i += nthr) bins[i] = 0;
    if (tid == 0) *gmax = 0u;

    NM nm{};
    nm.hp = p.hp;
    {
        float* wsm = reinterpret_cast<float*>(smem + p.off_w);
        const float* wt = p.weights;
        const int h = p.hid;
        float* t2 = wsm;
        float* t3 = wsm + pwl_smem_floats(NPAD);
        const int warp = tid >> 5, nwarp = (nthr + 31) >> 5;
        if (warp == 0) pwl_build(t2, reinterpret_cast<float2*>(t2 + NPAD), NPAD, wt, wt + h, wt + 2 * h, wt[3 * h], h, tid & 31);
        if (warp == (nwarp > 1 ? 1 : 0)) {
            const float* w3 = wt + 3 * h + 1;
            pwl_build(t3, reinterpret_cast<float2*>(t3 + NPAD), NPAD, w3, w3 + h, w3 + 2 * h, w3[3 * h], h, tid & 31);
        }
        nm.P2 = PwlSmem{t2, reinterpret_cast<const float2*>(t2 + NPAD)};
        nm.P3 = PwlSmem{t3, reinterpret_cast<const float2*>(t3 + NPAD)};
    }
    __syncthreads();
    // fixed-point scale of this CTA's bins: 2^32 over the power of two just above its largest |dlogit|
    {
        float mx = 0.f;
        for (int tix = blockIdx.x; tix < p.n_tiles; tix += gridDim.x) {
            const long long s0 = (long long)tix * tile;
            const int n = (int)min((long long)tile, p.B - s0) * V;
            for (int i = tid; i < n; i += nthr) mx = fmaxf(mx, fabsf(__ldg(grad_logit + s0 * V + i)));
        }
        for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        if ((tid & 31) == 0) atomicMax(gmax, __float_as_uint(mx));
    }
    __syncthreads();
    int ex = 0;
    {
        const float mx = __uint_as_float(*gmax);
        if (mx > 0.f && mx <= 3.0e38f) frexpf(mx, &ex);
        ex = max(-60, min(60, ex));
    }
    const int sexp = 32 - ex;
    const unsigned gmask = p.lanes == 32 ? 0xffffffffu : ((1u << p.lanes) - 1u) << ((tid & 31) & ~(p.lanes - 1));
    const BwdGroup bg2{bins, gmask, p.lanes, lg == 0, ldexpf(1.0f, sexp)};
    const size_t EB = (size_t)E * (size_t)p.B;

    for (int tix = blockIdx.x; tix < p.n_tiles; tix += gridDim.x) {
        const long long s0 = (long long)tix * tile;
        const int nvalid = (int)min((long long)tile, p.B - s0);
        // m^slot+1 (stash slot `slot`, zeros for slot < 0) -> m_st; columns past the batch are zero
        auto load_m = [&](int slot) {
            const int q4 = tile / 4;
            for (int i = tid; i < E * q4; i += nthr) {
                const int e = i / q4, c = (i - e * q4) * 4;
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (slot >= 0 && c < nvalid) {
                    const float* src = p.stash + (size_t)slot * EB + (size_t)e * p.B + s0 + c;
                    if ((p.B & 3) == 0) {
                        v = __ldcs(reinterpret_cast<const float4*>(src));
                    } else {
                        float vv[4] = {0.f, 0.f, 0.f, 0.f};
                        for (int j = 0; j < 4 && c + j < nvalid; ++j) vv[j] = __ldcs(src + j);
                        v = make_float4(vv[0], vv[1], vv[2], vv[3]);
                    }
                }
                *reinterpret_cast<float4*>(m_st + e * tile + c) = v;
            }
        };
        // ---- x[tile][N] -> xT[N][tile] (as the forward) ----
        {
            const float* xg = p.x + s0 * N;
            const int pitch = N | 1;
            if (p.trows >= pitch) {
                for (int i = tid; i < tile * N; i += nthr) {
                    const int si = i / N, n = i - si * N;
                    t_st[si * pitch + n] = si < nvalid ? __ldcg(xg + i) : 0.f;
                }
                __syncthreads();
                for (int i = tid; i < tile * N; i += nthr) {
                    const int n = i / tile, si = i - n * tile;
                    xT[i] = t_st[si * pitch + n];
                }
            } else {
                for (int i = tid; i < tile * N; i += nthr) {
                    const int si = i / N, n = i - si * N;
                    xT[n * tile + si] = si < nvalid ? __ldcg(xg + i) : 0.f;
                }
            }
        }
        __syncthreads();
        // ---- dlogit [tile][V] -> t_st as [V][tile]; m^T -> m_st ----
        {
            const float* gl = grad_logit + s0 * V;
            for (int i = tid; i < tile * V; i += nthr) {
                const int si = i / V, v = i - si * V;
                t_st[v * tile + si] = si < nvalid ? __ldg(gl + i) : 0.f;
            }
            load_m(p.T - 1);
        }
        __syncthreads();
        // ---- read-out (variable owner): bins of f3, dm = dres on the variable's edges ----
        if (worker)
            for (int v = r; v < V; v += R) {
                const int b = var_ptr[v], d = var_ptr[v + 1] - b;
                const float4 pr = lds4(xT + v * tile + l4);
                float acc[4] = {0.f, 0.f, 0.f, 0.f};
                for (int k = 0; k < d; ++k) {
                    const float4 mv = lds4(m_st + (b + k) * tile + l4);
                    acc[0] += mv.x; acc[1] += mv.y; acc[2] += mv.z; acc[3] += mv.w;
                }
                const float res[4] = {acc[0] + pr.x, acc[1] + pr.y, acc[2] + pr.z, acc[3] + pr.w};
                const float4 g4 = lds4(t_st + v * tile + l4);
                const float g[4] = {g4.x, g4.y, g4.z, g4.w};
                int sg[4];
                float dres[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    sg[j] = pwl_segment<NPAD>(nm.P3, res[j]);
                    dres[j] = g[j] * nm.P3.seg[sg[j]].x;
                }
                bins_add4<NPAD>(bins + 2 * NPAD, sg, g, res, gmask, p.lanes, lg == 0, bg2.scale);
                for (int k = 0; k < d; ++k) stg4(dm_st + (b + k) * tile + l4, dres);
            }
        __syncthreads();

        for (int it = p.T - 1; it >= 0; --it) {
            load_m(it - 1);
            __syncthreads();
            if (worker) light_var_phase(nm, var_ptr, xT, m_st, t_st, V, R, r, tile, l4);     // t^it, as the forward
            __syncthreads();
            // ---- check owner: du = dm S2(u), bins of f2, da = (sum of the other du) (1 - t^2) / 2 into the t rows ----
            if (worker)
                for (int c = r; c < C; c += R) {
                    const int b = chk_ptr[c], d = chk_ptr[c + 1] - b;
                    const uint16_t* edges = chk_edges + b;
#define GD_BC(D) bwd_chk_node<NPAD, D>(nm.P2, t_st + l4, dm_st + l4, tile, edges, bg2)
                    switch (d) {
                        case 1: GD_BC(1); break;
                        case 2: GD_BC(2); break;
                        case 3: GD_BC(3); break;
                        case 4: GD_BC(4); break;
                        default: {   // du staged in the m rows (m^it is dead once t is recomputed)
                            float acc[4] = {0.f, 0.f, 0.f, 0.f}, dacc[4] = {0.f, 0.f, 0.f, 0.f};
                            for (int k = 0; k < d; ++k) {
                                const float4 tv = lds4(t_st + edges[k] * tile + l4);
                                acc[0] += tv.x; acc[1] += tv.y; acc[2] += tv.z; acc[3] += tv.w;
                            }
                            for (int k = 0; k < d; ++k) {
                                const int eo = edges[k] * tile + l4;
                                const float4 tv = lds4(t_st + eo), d4 = lds4(dm_st + eo);
                                const float t4[4] = {tv.x, tv.y, tv.z, tv.w}, dm[4] = {d4.x, d4.y, d4.z, d4.w};
                                float u[4], du[4];
                                int sg[4];
#pragma unroll
                                for (int j = 0; j < 4; ++j) {
                                    u[j] = acc[j] - t4[j];
                                    sg[j] = pwl_segment<NPAD>(nm.P2, u[j]);
                                    du[j] = dm[j] * nm.P2.seg[sg[j]].x;
                                    dacc[j] += du[j];
                                }
                                bins_add4<NPAD>(bins, sg, dm, u, gmask, p.lanes, lg == 0, bg2.scale);
                                stg4(m_st + eo, du);
                            }
                            for (int k = 0; k < d; ++k) {
                                const int eo = edges[k] * tile + l4;
                                const float4 tv = lds4(t_st + eo), u4 = lds4(m_st + eo);
                                const float t4[4] = {tv.x, tv.y, tv.z, tv.w}, du[4] = {u4.x, u4.y, u4.z, u4.w};
                                float da[4];
#pragma unroll
                                for (int j = 0; j < 4; ++j) da[j] = 0.5f * (dacc[j] - du[j]) * fmaf(-t4[j], t4[j], 1.0f);
                                stg4(t_st + eo, da);
                            }
                        } break;
                    }
#undef GD_BC
                }
            __syncthreads();
            // ---- variable owner: dm += sum of the other da of the variable ----
            if (worker)
                for (int v = r; v < V; v += R) {
                    const int b = var_ptr[v], d = var_ptr[v + 1] - b;
                    const float* da_rows = t_st + b * tile + l4;
                    float* dm_rows = dm_st + b * tile + l4;
                    switch (d) {
                        case 0: case 1: break;      // no siblings: dm is unchanged
                        case 2: bwd_var_node<2>(da_rows, dm_rows, tile); break;
                        case 3: bwd_var_node<3>(da_rows, dm_rows, tile); break;
                        case 4: bwd_var_node<4>(da_rows, dm_rows, tile); break;
                        default: {
                            float acc[4] = {0.f, 0.f, 0.f, 0.f};
                            for (int k = 0; k < d; ++k) {
                                const float4 dv = lds4(da_rows + k * tile);
                                acc[0] += dv.x; acc[1] += dv.y; acc[2] += dv.z; acc[3] += dv.w;
                            }
                            for (int k = 0; k < d; ++k) {
                                const float4 dv = lds4(da_rows + k * tile), m4 = lds4(dm_rows + k * tile);
                                const float out[4] = {m4.x + (acc[0] - dv.x), m4.y + (acc[1] - dv.y), m4.z + (acc[2] - dv.z),
                                                      m4.w + (acc[3] - dv.w)};
                                stg4(dm_rows + k * tile, out);
                            }
                        } break;
                    }
                }
            __syncthreads();
        }
    }
    // ---- this CTA's bins -> its workspace record ----
    long long* rec = records + (size_t)blockIdx.x * (4 * NPAD + 1);
    for (int i = tid; i < 4 * NPAD; i += nthr) rec[i] = bins[i];
    if (tid == 0) rec[4 * NPAD] = sexp;
}

// Sum the CTA records in a fixed order (double), then contract with the weights: for unit u of an MLP with weights
// (a_u, b_u, c_u), b2, active on the segments j it is active on in pwl_build (a_u = 0: everywhere iff b_u > 0),
//   dW1_u = c_u sum_{j active} Sgx_j,  db1_u = c_u sum_{j active} Sg_j,  dW2_u = sum_{j active} (a_u Sgx_j + b_u Sg_j),  db2 = sum_j Sg_j.
template <int NPAD>
__global__ void cgnni_contract_kernel(const long long* __restrict__ records, int n_rec, const float* __restrict__ weights, int h,
                                      float* __restrict__ grad, int accumulate) {
    __shared__ double S[4 * NPAD];
    const int rw = 4 * NPAD + 1;
    for (int i = threadIdx.x; i < 4 * NPAD; i += blockDim.x) {
        double a = 0.0;
        for (int b = 0; b < n_rec; ++b) {
            const long long* rec = records + (size_t)b * rw;
            a += ldexp((double)rec[i], -(int)rec[4 * NPAD]);
        }
        S[i] = a;
    }
    __syncthreads();
    const int t = threadIdx.x;
    if (t >= 2 * (h + 1)) return;
    const int mlp = t / (h + 1), u = t - mlp * (h + 1);
    const float* w = weights + mlp * (3 * h + 1);
    const double* Sg = S + mlp * 2 * NPAD;
    const double* Sgx = Sg + NPAD;
    float* out = grad + mlp * (3 * h + 1);
    if (u == h) {
        double a = 0.0;
        for (int j = 0; j < NPAD; ++j) a += Sg[j];
        out[3 * h] = accumulate ? out[3 * h] + (float)a : (float)a;
        return;
    }
    const double a = (double)w[u], b = (double)w[h + u], c = (double)w[2 * h + u];
    const float inf = __int_as_float(0x7f800000);
    const float tu = a != 0.0 ? (float)(-b / a) : inf;
    int rank = 0;                    // the breakpoint's position in pwl_build's sorted list
    for (int v = 0; v < h; ++v) {
        const double av = (double)w[v];
        const float tv = av != 0.0 ? (float)(-(double)w[h + v] / av) : inf;
        rank += (tv < tu || (tv == tu && v < u)) ? 1 : 0;
    }
    double G = 0.0, GX = 0.0;
    for (int j = 0; j < NPAD; ++j) {
        const bool active = a == 0.0 ? b > 0.0 : (a > 0.0 ? rank < j : rank >= j);
        if (active) { G += Sg[j]; GX += Sgx[j]; }
    }
    const float g1 = (float)(c * GX), gb = (float)(c * G), g2 = (float)(a * GX + b * G);
    out[u] = accumulate ? out[u] + g1 : g1;
    out[h + u] = accumulate ? out[h + u] + gb : gb;
    out[2 * h + u] = accumulate ? out[2 * h + u] + g2 : g2;
}

struct LightBwdPlan {
    LightPlan pl;
    int off_dm, off_bins;
};

static int plan_light_bwd(const gd_graph* g, const gd_model* m, int64_t B, LightBwdPlan* out) {
    const int npad = m->hidden < 16 ? 16 : 32;
    const int bins_bytes = (4 * npad + 2) * 8;
    plan_light(g, m, B, &out->pl, true, (int)g->E, bins_bytes);
    if (!out->pl.ok) {
        set_error("gd_decode_bwd: CGNNI training needs the node-owner kernel: %s", out->pl.why);
        return GD_ERR_UNSUPPORTED;
    }
    LightPlan& pl = out->pl;
    out->off_dm = pl.smem;
    out->off_bins = (out->off_dm + (int)g->E * pl.p.tile * 4 + 15) / 16 * 16;
    pl.smem = out->off_bins + bins_bytes;
    return GD_OK;
}

int64_t light_bwd_workspace_floats(const gd_graph* g, const gd_model* model, int64_t B) {
    LightBwdPlan bp;
    if (plan_light_bwd(g, model, B, &bp) != GD_OK) return -1;
    return (int64_t)bp.pl.grid * light_bwd_record_words(bp.pl.npad) * 2;
}

int light_backward(const gd_graph* g, const gd_model* model, const float* weights_dev, const float* x_dev, const float* stash_dev,
                   const float* grad_logit_dev, float* grad_weights_dev, float* workspace_dev, int accumulate, int64_t B,
                   cudaStream_t st) {
    LightBwdPlan bp;
    int rc = plan_light_bwd(g, model, B, &bp);
    if (rc != GD_OK) return rc;
    GD_CHECK_ARG(((uintptr_t)workspace_dev & 7) == 0, "gd_decode_bwd: workspace must be 8-byte aligned");
    LightPlan& pl = bp.pl;
    pl.p.x = x_dev; pl.p.weights = weights_dev; pl.p.stash = const_cast<float*>(stash_dev);
    long long* records = reinterpret_cast<long long*>(workspace_dev);
    void (*k)(const LightParams, const float*, long long*, int, int) =
        pl.npad == 16 ? cgnni_bwd_light_kernel<16> : cgnni_bwd_light_kernel<32>;
    GD_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, pl.smem));
    k<<<pl.grid, pl.threads, pl.smem, st>>>(pl.p, grad_logit_dev, records, bp.off_dm, bp.off_bins);
    GD_CUDA(cudaGetLastError());
    if (pl.npad == 16) cgnni_contract_kernel<16><<<1, 128, 0, st>>>(records, pl.grid, weights_dev, model->hidden, grad_weights_dev, accumulate);
    else cgnni_contract_kernel<32><<<1, 128, 0, st>>>(records, pl.grid, weights_dev, model->hidden, grad_weights_dev, accumulate);
    GD_CUDA(cudaGetLastError());
    return GD_OK;
}

}  // namespace gd
