// Resident fused decoder for the LIGHT phase programs -- classical/CGNNI.py, quantum/QGNNI.py and the
// two sum-product decoders (quantum/BP.py, classical/BP.py): a few dozen FP32 instructions per edge and
// iteration, so the edge-owner kernel of gd_decode.cu (built around decoder_v2_4's 256 Softplus units per
// edge-iteration: four barriers, node-sum arrays, one syndrome per lane) spends most of its issue slots on
// loop / index / barrier overhead there (ncu, QGNNI toric L=5: 129 lane-instructions per edge-iteration
// against ~30 of arithmetic).  This kernel keeps the same state in shared memory but maps it like the
// TMA-staged streamed kernel:
//   * a lane owns FOUR syndromes (one float4 of every batch-minor row m[E][tile], t[E][tile], xT[N][tile]):
//     every index / table load and loop step is amortised over four syndromes and gives 4-way ILP;
//   * NODE-OWNER phases: thread group r owns variables v == r (mod R), then checks c == r (mod R); it reads
//     the node's messages once, sums them in ascending edge id (same order as the CPU index_add_ of the
//     reference), and writes the outgoing messages -- no node-sum arrays, TWO barriers per iteration;
//   * node degrees 1..4 run fully unrolled with the values in registers (gd_nodemath.cuh), larger degrees
//     (BCH(63,45): check degree 24) take the generic loops;
//   * the 1 -> h -> 1 ReLU MLPs are evaluated as the piecewise-linear functions they are (gd_math.cuh).
// Requires the canonical variable-sorted edge order (H.to_sparse()); other graphs keep the edge-owner kernel.
#include "gd_common.cuh"
#include "gd_math.cuh"
#include "gd_options.cuh"
#include "gd_decode.cuh"
#include "gd_nodemath.cuh"
#include "gd_light.cuh"
#include <stdlib.h>
#include <math.h>
#include <string.h>
#include <vector>

namespace gd {

#define GD_DEGREE_SWITCH4(d, CALL, ...)     \
    switch (d) {                            \
        case 1: { CALL(1); } break;         \
        case 2: { CALL(2); } break;         \
        case 3: { CALL(3); } break;         \
        case 4: { CALL(4); } break;         \
        default: { __VA_ARGS__; } break;    \
    }

// One check of degree D, state in shared memory: t_l4 / m_l4 point at this lane's float4 column.
template <int PROG, int NPAD, int D>
__device__ __forceinline__ void light_chk_node(const NodeMath<PROG, NPAD>& nm, const float* t_l4, float* m_l4, int tile,
                                               const uint16_t* edges, const float4 s4) {
    using NM = NodeMath<PROG, NPAD>;
    int e[D];
#pragma unroll
    for (int k = 0; k < D; ++k) e[k] = edges[k] * tile;
    float4 tv[D];
#pragma unroll
    for (int k = 0; k < D; ++k) tv[k] = lds4(t_l4 + e[k]);
    const float sg[4] = {s4.x, s4.y, s4.z, s4.w};
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    int cnt[4] = {0, 0, 0, 0};
#pragma unroll
    for (int k = 0; k < D; ++k) {
        const float t4[4] = {tv[k].x, tv[k].y, tv[k].z, tv[k].w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if constexpr (NM::kIsBP) {
                acc[j] -= fabsf(t4[j]);
                cnt[j] += t4[j] > 0.f ? 1 : 0;
            } else {
                acc[j] += t4[j];
            }
        }
    }
    if constexpr (PROG == GD_PROG_BP_QUANTUM) {
#pragma unroll
        for (int j = 0; j < 4; ++j) cnt[j] += sg[j] < 0.f ? 1 : 0;
    }
#pragma unroll
    for (int k = 0; k < D; ++k) {
        const float t4[4] = {tv[k].x, tv[k].y, tv[k].z, tv[k].w};
        float out[4];
        if constexpr (NM::kIsBP) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int q = cnt[j] - (t4[j] > 0.f ? 1 : 0);
                out[j] = bp_check_out(acc[j] + fabsf(t4[j]), q & 1, NM::kEps2);
            }
        } else {
            float ext[4], oo[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) ext[j] = acc[j] - t4[j];
            nm.chk_mlp(ext, oo);
            const float4 mo = lds4(m_l4 + e[k]);
            out[0] = fmaf(oo[0], sg[0], mo.x);
            out[1] = fmaf(oo[1], sg[1], mo.y);
            out[2] = fmaf(oo[2], sg[2], mo.z);
            out[3] = fmaf(oo[3], sg[3], mo.w);
        }
        stg4(m_l4 + e[k], out);
    }
}

// STASH (CGNNI training): m after every iteration also goes to p.stash[it][E][B] for the backward (gd_backward_light.cu)
template <int PROG, int NPAD, bool STASH = false>
__global__ void __launch_bounds__(512, 2) decode_light_kernel(const LightParams p) {
    extern __shared__ __align__(128) unsigned char smem[];
    using NM = NodeMath<PROG, NPAD>;
    constexpr bool kIsBP = NM::kIsBP;
    constexpr bool kSign = NM::kSign;
    constexpr bool kClamp = (PROG == GD_PROG_CGNNI || PROG == GD_PROG_BP_CLASSICAL);
    const int tile = p.tile, E = p.E, V = p.V, C = p.C, N = p.N, R = p.R;
    const int tid = threadIdx.x, nthr = blockDim.x;
    const int l4 = (tid % p.lanes) * 4, r = tid / p.lanes;
    const bool worker = r < R;                        // threads beyond R * lanes only help with the copies
    float* const xT = reinterpret_cast<float*>(smem + p.off_x);
    float* const m_st = reinterpret_cast<float*>(smem + p.off_m);
    float* const t_st = reinterpret_cast<float*>(smem + p.off_t);
    uint16_t* const var_ptr = reinterpret_cast<uint16_t*>(smem + p.off_tab);
    uint16_t* const chk_ptr = var_ptr + (V + 1);
    uint16_t* const chk_edges = chk_ptr + (C + 1);
    for (int i = tid; i <= V; i += nthr) var_ptr[i] = (uint16_t)p.tb.var_ptr[i];
    for (int i = tid; i <= C; i += nthr) chk_ptr[i] = (uint16_t)p.tb.chk_ptr[i];
    for (int i = tid; i < E; i += nthr) chk_edges[i] = (uint16_t)p.tb.chk_edges[i];

    NM nm{};
    nm.hp = p.hp;
    if constexpr (!kIsBP) {
        float* wsm = reinterpret_cast<float*>(smem + p.off_w);
        const float* wt = p.weights;
        const int h = p.hid, hp = p.hp;
        if constexpr (NPAD > 0) {
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
        } else {
            float* slot = wsm;
            stage_mlp_t(slot, hp, h, wt, 1, false, wt + h, wt + 2 * h, 1.f, 1.f, tid, nthr);
            nm.W2 = MlpSmem{slot, slot + hp, slot + 2 * hp, slot + 3 * hp, wt[3 * h]};
            wt += 3 * h + 1;
            slot += 4 * hp;
            stage_mlp_t(slot, hp, h, wt, 1, false, wt + h, wt + 2 * h, 1.f, 1.f, tid, nthr);
            nm.W3 = MlpSmem{slot, slot + hp, slot + 2 * hp, slot + 3 * hp, wt[3 * h]};
        }
    }
    __syncthreads();

    for (int tix = blockIdx.x; tix < p.n_tiles; tix += gridDim.x) {
        const long long s0 = (long long)tix * tile;
        const int nvalid = (int)min((long long)tile, p.B - s0);
        if (p.gate_in) {   // gated launch: this tile's chunk may still be on its way from the host
            if (tid == 0) gate_wait(p.gate_in + tix / p.gate_chunk_tiles, p.gate_epoch, p.gate_err);
            __syncthreads();
        }
        // ---- x[tile][N] (coalesced reads) -> xT[N][tile]; m = 0 ----
        {
            const float* xg = p.x + s0 * N;
            const int pitch = N | 1;
            if (p.trows >= pitch) {
                // conflict-free transpose through the (idle) t region: rows of odd pitch
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
            for (int i = tid; i < E * tile; i += nthr) m_st[i] = 0.f;
        }
        __syncthreads();

        for (int it = 0; it < p.T; ++it) {
            // ---- variable phase: owner of variable v (edges of v are the contiguous rows var_ptr[v] ..) ----
            if (worker)
                for (int v = r; v < V; v += R) {
                    const int b = var_ptr[v], d = var_ptr[v + 1] - b;
                    const float4 pr = lds4(xT + v * tile + l4);
                    const float* rows = m_st + b * tile + l4;
                    float* tout = t_st + b * tile + l4;
#define GD_LV(D) nm.template var_node<D>(rows, tile, pr, tout)
                    GD_DEGREE_SWITCH4(d, GD_LV, {
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
                    })
#undef GD_LV
                }
            __syncthreads();
            // ---- check phase: owner of check c ----
            if (worker)
                for (int c = r; c < C; c += R) {
                    const int b = chk_ptr[c], d = chk_ptr[c + 1] - b;
                    float4 s4 = make_float4(1.f, 1.f, 1.f, 1.f);
                    if constexpr (kSign) s4 = lds4(xT + (V + c) * tile + l4);
                    const uint16_t* edges = chk_edges + b;
#define GD_LC(D) light_chk_node<PROG, NPAD, D>(nm, t_st + l4, m_st + l4, tile, edges, s4)
                    GD_DEGREE_SWITCH4(d, GD_LC, {
                        const float sg[4] = {s4.x, s4.y, s4.z, s4.w};
                        float acc[4] = {0.f, 0.f, 0.f, 0.f};
                        int cnt[4] = {0, 0, 0, 0};
                        for (int k = 0; k < d; ++k) {
                            const float4 tv = lds4(t_st + edges[k] * tile + l4);
                            const float t4[4] = {tv.x, tv.y, tv.z, tv.w};
                            _Pragma("unroll")
                            for (int j = 0; j < 4; ++j) {
                                if constexpr (kIsBP) {
                                    acc[j] -= fabsf(t4[j]);
                                    cnt[j] += t4[j] > 0.f ? 1 : 0;
                                } else {
                                    acc[j] += t4[j];
                                }
                            }
                        }
                        if constexpr (PROG == GD_PROG_BP_QUANTUM) {
                            _Pragma("unroll")
                            for (int j = 0; j < 4; ++j) cnt[j] += sg[j] < 0.f ? 1 : 0;
                        }
                        for (int k = 0; k < d; ++k) {
                            const int eo = edges[k] * tile + l4;
                            const float4 tv = lds4(t_st + eo);
                            const float t4[4] = {tv.x, tv.y, tv.z, tv.w};
                            float out[4];
                            if constexpr (kIsBP) {
                                _Pragma("unroll")
                                for (int j = 0; j < 4; ++j) {
                                    const int q = cnt[j] - (t4[j] > 0.f ? 1 : 0);
                                    out[j] = bp_check_out(acc[j] + fabsf(t4[j]), q & 1, NM::kEps2);
                                }
                            } else {
                                float ext[4], oo[4];
                                _Pragma("unroll")
                                for (int j = 0; j < 4; ++j) ext[j] = acc[j] - t4[j];
                                nm.chk_mlp(ext, oo);
                                const float4 mo = lds4(m_st + eo);
                                out[0] = fmaf(oo[0], sg[0], mo.x);
                                out[1] = fmaf(oo[1], sg[1], mo.y);
                                out[2] = fmaf(oo[2], sg[2], mo.z);
                                out[3] = fmaf(oo[3], sg[3], mo.w);
                            }
                            stg4(m_st + eo, out);
                        }
                    })
#undef GD_LC
                }
            __syncthreads();
            if constexpr (STASH) {   // m^{it+1}: [E][tile] rows -> stash[it][E][B]; the next writer of m_st is behind a barrier
                const int q4 = tile / 4;
                float* dst = p.stash + (size_t)it * E * (size_t)p.B + s0;
                for (int i = tid; i < E * q4; i += nthr) {
                    const int e = i / q4, c = (i - e * q4) * 4;
                    if (c >= nvalid) continue;
                    const float4 v = lds4(m_st + e * tile + c);
                    float* d = dst + (size_t)e * p.B + c;
                    if ((p.B & 3) == 0) {
                        __stcg(reinterpret_cast<float4*>(d), v);
                    } else {
                        const float vv[4] = {v.x, v.y, v.z, v.w};
                        for (int j = 0; j < 4 && c + j < nvalid; ++j) __stcg(d + j, vv[j]);
                    }
                }
            }
        }

        // ---- read-out (variable owner): logit rows into the t region as lg[V][tile] ----
        if (worker)
            for (int v = r; v < V; v += R) {
                const int b = var_ptr[v], d = var_ptr[v + 1] - b;
                const float4 pr = lds4(xT + v * tile + l4);
                float acc[4] = {0.f, 0.f, 0.f, 0.f};
                for (int k = 0; k < d; ++k) {
                    const float4 mv = lds4(m_st + (b + k) * tile + l4);
                    acc[0] += mv.x; acc[1] += mv.y; acc[2] += mv.z; acc[3] += mv.w;
                }
                float lg[4] = {acc[0] + pr.x, acc[1] + pr.y, acc[2] + pr.z, acc[3] + pr.w};
                nm.readout_mlp(lg);
                stg4(t_st + v * tile + l4, lg);
            }
        __syncthreads();
        // ---- outputs: prob / logit / hard [tile][V], coalesced over v ----
        {
            const long long g0 = s0 * V;
            const int pitch = V | 1;
            const bool via_m = E >= pitch;                // transpose lg[V][tile] -> [tile][pitch] through the dead m region
            if (via_m) {
                for (int i = tid; i < V * tile; i += nthr) {
                    const int v = i / tile, si = i - v * tile;
                    m_st[si * pitch + v] = t_st[i];
                }
                __syncthreads();
            }
            for (int i = tid; i < nvalid * V; i += nthr) {
                const int si = i / V, v = i - si * V;
                const float lg = via_m ? m_st[si * pitch + v] : t_st[v * tile + si];
                float pr = sigmoid_neg(lg);
                if (kClamp) pr = fminf(fmaxf(pr, 1e-7f), 1.0f - 1e-7f);
                if (p.prob) p.prob[g0 + i] = pr;
                if (p.logit) p.logit[g0 + i] = lg;
                if (p.hard) p.hard[g0 + i] = pr > 0.5f;
            }
        }
        __syncthreads();
        if (p.gate_out && tid == 0) {   // gated launch: publish the tile so the chunk's device->host copy can go
            __threadfence_system();
            atomicAdd(p.gate_out + tix / p.gate_chunk_tiles, 1u);
        }
    }
}

// ---- the "next" programs on the same mapping: neural BP (quantum/neural_BP.py, quantum/decoder_v1_1.py: per-edge weights,
// un-tied layers, + alpha * m_p) and the GRU decoder (quantum/QGNNNI_ca.py: MLP + GRUCell(1,1) per phase, m updated in place).
// Same layout, phases and barriers as decode_light_kernel; node loops over the runtime degree (registers for d <= 4).
template <int PROG, int NPAD>
__global__ void __launch_bounds__(512, 2) decode_light_ext_kernel(const LightParams p) {
    extern __shared__ __align__(128) unsigned char smem[];
    constexpr bool kNBP = PROG == GD_PROG_NEURAL_BP;
    const int tile = p.tile, E = p.E, V = p.V, C = p.C, N = p.N, R = p.R;
    const int tid = threadIdx.x, nthr = blockDim.x;
    const int l4 = (tid % p.lanes) * 4, r = tid / p.lanes;
    const bool worker = r < R;
    float* const xT = reinterpret_cast<float*>(smem + p.off_x);
    float* const m_st = reinterpret_cast<float*>(smem + p.off_m);
    float* const t_st = reinterpret_cast<float*>(smem + p.off_t);
    uint16_t* const var_ptr = reinterpret_cast<uint16_t*>(smem + p.off_tab);
    uint16_t* const chk_ptr = var_ptr + (V + 1);
    uint16_t* const chk_edges = chk_ptr + (C + 1);
    for (int i = tid; i <= V; i += nthr) var_ptr[i] = (uint16_t)p.tb.var_ptr[i];
    for (int i = tid; i <= C; i += nthr) chk_ptr[i] = (uint16_t)p.tb.chk_ptr[i];
    for (int i = tid; i < E; i += nthr) chk_edges[i] = (uint16_t)p.tb.chk_edges[i];
    PwlSmem P1{}, P2{}, P3{};
    const float* gru = nullptr;
    if constexpr (!kNBP) {      // GRU_CA: ggc1.mlp1 | ggc1.rnn | ggc2.mlp2 | ggc2.rnn | mlp  (packed order)
        float* wsm = reinterpret_cast<float*>(smem + p.off_w);
        const int h = p.hid, warp = tid >> 5, nwarp = (nthr + 31) >> 5;
        for (int k = warp; k < 3; k += nwarp) {
            const float* w = p.weights + k * (3 * h + 1) + k * 12;
            float* t = wsm + k * pwl_smem_floats(NPAD);
            pwl_build(t, reinterpret_cast<float2*>(t + NPAD), NPAD, w, w + h, w + 2 * h, w[3 * h], h, tid & 31);
        }
        float* gs = wsm + 3 * pwl_smem_floats(NPAD);
        if (tid < 24) gs[tid] = p.weights[(tid < 12 ? 3 * h + 1 : 2 * (3 * h + 1)) + tid];
        gru = gs;
        P1 = PwlSmem{wsm, reinterpret_cast<const float2*>(wsm + NPAD)};
        P2 = PwlSmem{wsm + pwl_smem_floats(NPAD), reinterpret_cast<const float2*>(wsm + pwl_smem_floats(NPAD) + NPAD)};
        P3 = PwlSmem{wsm + 2 * pwl_smem_floats(NPAD), reinterpret_cast<const float2*>(wsm + 2 * pwl_smem_floats(NPAD) + NPAD)};
    }
    __syncthreads();

    for (int tix = blockIdx.x; tix < p.n_tiles; tix += gridDim.x) {
        const long long s0 = (long long)tix * tile;
        const int nvalid = (int)min((long long)tile, p.B - s0);
        if (p.gate_in) {   // gated launch: this tile's chunk may still be on its way from the host
            if (tid == 0) gate_wait(p.gate_in + tix / p.gate_chunk_tiles, p.gate_epoch, p.gate_err);
            __syncthreads();
        }
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
            for (int i = tid; i < E * tile; i += nthr) m_st[i] = 0.f;
        }
        __syncthreads();

        for (int it = 0; it < p.T; ++it) {
            const float* wl = kNBP ? p.weights + (size_t)it * 2 * E : nullptr;      // this layer's W[E] | W_p[E]
            // ---- variable phase ----
            if (worker)
                for (int v = r; v < V; v += R) {
                    const int b = var_ptr[v], d = var_ptr[v + 1] - b;
                    const float4 pr4 = lds4(xT + v * tile + l4);
                    const float pr[4] = {pr4.x, pr4.y, pr4.z, pr4.w};
                    float acc[4] = {0.f, 0.f, 0.f, 0.f};
                    for (int k = 0; k < d; ++k) {                  // ascending edge id
                        const float4 mv = lds4(m_st + (b + k) * tile + l4);
                        const float wk = kNBP ? __ldg(wl + b + k) : 1.f;
                        acc[0] = fmaf(mv.x, wk, acc[0]); acc[1] = fmaf(mv.y, wk, acc[1]);
                        acc[2] = fmaf(mv.z, wk, acc[2]); acc[3] = fmaf(mv.w, wk, acc[3]);
                    }
                    for (int k = 0; k < d; ++k) {
                        float* mp = m_st + (b + k) * tile + l4;
                        const float4 mv = lds4(mp);
                        const float m4[4] = {mv.x, mv.y, mv.z, mv.w};
                        float out[4];
                        if constexpr (kNBP) {       // neural_BP.py:244-258: t from (sum of m W) - m W + prior W_p; m itself stays = m_p
                            const float wk = __ldg(wl + b + k), wpk = __ldg(wl + E + b + k);
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const float a = acc[j] - m4[j] * wk + pr[j] * wpk;
                                const float tv = bp_log_abs_tanh_half<false>(a, -46.0517019f);
                                out[j] = a < 0.f ? -tv : tv;
                            }
                            stg4(t_st + (b + k) * tile + l4, out);
                        } else {                    // QGNNNI_ca.py:103-106,197-198,208-209
#pragma unroll
                            for (int j = 0; j < 4; ++j)
                                out[j] = gru_cell(gru, m4[j], pwl_eval<NPAD>(P1, acc[j] - m4[j] + pr[j]));
                            stg4(t_st + (b + k) * tile + l4, out);      // staged in t: siblings still need the old m
                        }
                    }
                    if constexpr (!kNBP)
                        for (int k = 0; k < d; ++k) {
                            const float4 nv = lds4(t_st + (b + k) * tile + l4);
                            *reinterpret_cast<float4*>(m_st + (b + k) * tile + l4) = nv;
                        }
                }
            __syncthreads();
            // ---- check phase ----
            if (worker)
                for (int c = r; c < C; c += R) {
                    const int b = chk_ptr[c], d = chk_ptr[c + 1] - b;
                    const float4 s4 = lds4(xT + (V + c) * tile + l4);
                    const float sg[4] = {s4.x, s4.y, s4.z, s4.w};
                    const uint16_t* edges = chk_edges + b;
                    float acc[4] = {0.f, 0.f, 0.f, 0.f};
                    int cnt[4] = {0, 0, 0, 0};
                    for (int k = 0; k < d; ++k) {
                        const float4 tv = lds4((kNBP ? t_st : m_st) + edges[k] * tile + l4);
                        const float t4[4] = {tv.x, tv.y, tv.z, tv.w};
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            if constexpr (kNBP) {
                                acc[j] -= fabsf(t4[j]);
                                cnt[j] += t4[j] > 0.f ? 1 : 0;
                            } else {
                                acc[j] += t4[j];
                            }
                        }
                    }
                    if constexpr (kNBP) {
#pragma unroll
                        for (int j = 0; j < 4; ++j) cnt[j] += sg[j] < 0.f ? 1 : 0;
                        const float alpha = __ldg(p.weights + (size_t)(2 * p.T + 2) * E);
                        for (int k = 0; k < d; ++k) {
                            const int eo = edges[k] * tile + l4;
                            const float4 tv = lds4(t_st + eo), mo = lds4(m_st + eo);
                            const float t4[4] = {tv.x, tv.y, tv.z, tv.w}, m4[4] = {mo.x, mo.y, mo.z, mo.w};
                            float out[4];
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const int q = cnt[j] - (t4[j] > 0.f ? 1 : 0);
                                out[j] = fmaf(alpha, m4[j], bp_check_out(acc[j] + fabsf(t4[j]), q & 1, 1e-15f));
                            }
                            stg4(m_st + eo, out);
                        }
                    } else {                        // QGNNNI_ca.py:109,197-198,206-207: new values staged in t, then copied
                        for (int k = 0; k < d; ++k) {
                            const int eo = edges[k] * tile + l4;
                            const float4 mo = lds4(m_st + eo);
                            const float m4[4] = {mo.x, mo.y, mo.z, mo.w};
                            float out[4];
#pragma unroll
                            for (int j = 0; j < 4; ++j)
                                out[j] = gru_cell(gru + 12, m4[j], pwl_eval<NPAD>(P2, (acc[j] - m4[j]) * sg[j]));
                            stg4(t_st + eo, out);
                        }
                        for (int k = 0; k < d; ++k) {
                            const int eo = edges[k] * tile + l4;
                            *reinterpret_cast<float4*>(m_st + eo) = lds4(t_st + eo);
                        }
                    }
                }
            __syncthreads();
        }

        // ---- read-out ----
        if (worker)
            for (int v = r; v < V; v += R) {
                const int b = var_ptr[v], d = var_ptr[v + 1] - b;
                const float4 pr4 = lds4(xT + v * tile + l4);
                const float pr[4] = {pr4.x, pr4.y, pr4.z, pr4.w};
                float acc[4] = {0.f, 0.f, 0.f, 0.f}, accp[4] = {0.f, 0.f, 0.f, 0.f};
                const float* wo = kNBP ? p.weights + (size_t)p.T * 2 * E : nullptr;
                for (int k = 0; k < d; ++k) {
                    const float4 mv = lds4(m_st + (b + k) * tile + l4);
                    const float m4[4] = {mv.x, mv.y, mv.z, mv.w};
                    const float wk = kNBP ? __ldg(wo + b + k) : 1.f, wpk = kNBP ? __ldg(wo + E + b + k) : 0.f;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        acc[j] = fmaf(m4[j], wk, acc[j]);
                        accp[j] = fmaf(pr[j], wpk, accp[j]);
                    }
                }
                float lg[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) lg[j] = kNBP ? acc[j] + accp[j] : pwl_eval<(NPAD > 0 ? NPAD : 16)>(P3, acc[j]);
                stg4(t_st + v * tile + l4, lg);
            }
        __syncthreads();
        {
            const long long g0 = s0 * V;
            const int pitch = V | 1;
            const bool via_m = E >= pitch;
            if (via_m) {
                for (int i = tid; i < V * tile; i += nthr) {
                    const int v = i / tile, si = i - v * tile;
                    m_st[si * pitch + v] = t_st[i];
                }
                __syncthreads();
            }
            for (int i = tid; i < nvalid * V; i += nthr) {
                const int si = i / V, v = i - si * V;
                const float lg = via_m ? m_st[si * pitch + v] : t_st[v * tile + si];
                float pr = sigmoid_neg(lg);
                if (!kNBP) pr = fminf(fmaxf(pr, 1e-7f), 1.0f - 1e-7f);      // QGNNNI_ca.py:247
                if (p.prob) p.prob[g0 + i] = pr;
                if (p.logit) p.logit[g0 + i] = lg;
                if (p.hard) p.hard[g0 + i] = pr > 0.5f;
            }
        }
        __syncthreads();
        if (p.gate_out && tid == 0) {   // gated launch: publish the tile so the chunk's device->host copy can go
            __threadfence_system();
            atomicAdd(p.gate_out + tix / p.gate_chunk_tiles, 1u);
        }
    }
}

static int align_up_l(int x, int a) { return (x + a - 1) / a * a; }

void plan_light(const gd_graph* g, const gd_model* m, int64_t B, LightPlan* out, bool train, int extra_rows, int extra_bytes) {
    LightParams& p = out->p;
    memset(&p, 0, sizeof(p));
    out->ok = false;
    out->why = "program has no node-owner kernel";
    const int prog = m->program;
    const bool ext = prog == GD_PROG_NEURAL_BP || prog == GD_PROG_GRU_CA;
    const bool force = train || opt_on(OPT_FORCE_LIGHT);
    if (prog != GD_PROG_CGNNI && prog != GD_PROG_QGNNI && prog != GD_PROG_BP_QUANTUM && prog != GD_PROG_BP_CLASSICAL && !ext) return;
    if (prog == GD_PROG_GRU_CA && (m->hidden >= 32 || (m->flags & GD_FLAG_ALL_ITERS) || opt_on(OPT_NO_PWL))) return;
    if (prog == GD_PROG_NEURAL_BP && m->hidden != g->E) return;      // the caller's argument check reports it
    if (train && m->hidden >= 32) { out->why = "hidden >= 32: the MLPs have no piecewise-linear table"; return; }
    if (!train && (opt_on(OPT_NO_LIGHT) || opt_on(OPT_FORCE_STREAMED))) return;
    if ((B + 15) / 16 < g->sm_count && !force) return;   // cannot fill the GPU at any tile size: skip the search
    out->why = "code too large for the node-owner kernel (E >= 65536 or V, C >= 65535)";
    if (g->E >= 65536 || g->V >= 65535 || g->C >= 65535) return;
    out->why = "edge order is not the canonical variable-sorted order (H.to_sparse())";
    for (size_t i = 0; i < g->h_var_edges.size(); ++i)
        if (g->h_var_edges[i] != (int32_t)i) return;           // needs the canonical variable-sorted edge order
    const bool bp = prog == GD_PROG_BP_QUANTUM || prog == GD_PROG_BP_CLASSICAL || prog == GD_PROG_NEURAL_BP;
    p.B = B; p.T = m->iters; p.V = g->V; p.C = g->C; p.E = (int)g->E; p.N = g->N; p.tb = g->t;
    p.hid = bp ? 0 : m->hidden;
    p.hp = align_up_l(p.hid, 4);
    out->npad = (!bp && m->hidden < 32 && (train || !opt_on(OPT_NO_PWL))) ? (m->hidden < 16 ? 16 : 32) : 0;
    p.trows = g->E > g->V ? (int)g->E : g->V;                  // the t region doubles as the logit rows lg[V][tile]
    int off = 0;
    p.off_w = off;
    off += bp ? 0 : (prog == GD_PROG_GRU_CA ? (3 * pwl_smem_floats(32) + 24) * 4
                                             : (out->npad ? 2 * pwl_smem_floats(out->npad) * 4 : 2 * 4 * p.hp * 4));
    off = align_up_l(off, 16);
    p.off_tab = off; off += (g->V + 1 + g->C + 1 + (int)g->E) * 2;
    off = align_up_l(off, 128);
    const int fixed = off;
    const int64_t per_syn = ((int64_t)g->N + g->E + p.trows + extra_rows) * 4;
    // Geometry: tile in {16, 32, 64, 128} (lanes = tile / 4 divides a warp), R thread groups of `lanes` threads, and as
    // many co-resident CTAs as shared memory and the 64-register build allow (one CTA's barriers overlap another's
    // arithmetic).  Node-owner phases are only as fast as their busiest group, so every candidate is scored by
    //   rounds * tile / (sqrt(balance) * occupancy),  balance = ideal / actual work of the busiest group over both phases;
    // graphs whose balance falls below 0.3 keep the edge-owner kernel.
    int best_tile = 0, best_cps = 1, best_R = 1;
    double best_cost = 1e300, best_bal = 0.0;
    const long long et = opt_int(OPT_LTILE, 0), er = opt_int(OPT_LR, 0);
    const int maxn = g->V > g->C ? g->V : g->C;
    std::vector<int> load;
    for (int t = 16; t <= 128; t *= 2) {
        if (et > 0 && et != t) continue;
        const int64_t smem = fixed + per_syn * t + extra_bytes;
        if (smem > g->max_smem_optin) break;
        const int lanes = t / 4;
        int r_max = 512 / lanes;
        if (r_max > maxn) r_max = maxn;
        const int cand[8] = {r_max, g->C, (g->C + 1) / 2, g->V, (g->V + 1) / 2, (g->V + 2) / 3, (g->V + 3) / 4, (g->C + 2) / 3};
        for (int ci = 0; ci < 8; ++ci) {
            const int R = cand[ci];
            if (R < 1 || R > r_max) continue;
            if (er > 0 && er != R) continue;
            bool dup = false;
            for (int cj = 0; cj < ci; ++cj) dup = dup || cand[cj] == R;
            if (dup) continue;
            int max_v = 0, max_c = 0;
            load.assign((size_t)R, 0);
            for (int v = 0; v < g->V; ++v) load[(size_t)(v % R)] += g->h_var_ptr[(size_t)v + 1] - g->h_var_ptr[(size_t)v] + 1;
            for (int q = 0; q < R; ++q) max_v = load[(size_t)q] > max_v ? load[(size_t)q] : max_v;
            load.assign((size_t)R, 0);
            for (int c = 0; c < g->C; ++c) load[(size_t)(c % R)] += g->h_chk_ptr[(size_t)c + 1] - g->h_chk_ptr[(size_t)c] + 1;
            for (int q = 0; q < R; ++q) max_c = load[(size_t)q] > max_c ? load[(size_t)q] : max_c;
            const double bal = ((double)(2 * g->E + g->V + g->C) / R) / (double)(max_v + max_c);
            const int threads = align_up_l(R * lanes, 32);
            int cps = (int)(g->max_smem_sm / (smem + 1024));
            if (cps > 1024 / threads) cps = 1024 / threads;      // 64 registers per thread
            if (cps > 16) cps = 16;
            if (cps < 1) cps = 1;
            const double occ = (double)(threads * cps) / 1024.0;
            const int64_t n_t = (B + t - 1) / t;
            const int64_t slots = (int64_t)g->sm_count * cps;
            const int64_t rounds = (n_t + slots - 1) / slots;
            // measured (toric L=5, BCH, toy LDPC; profiles/r01g_light_geometry.txt): resident threads matter linearly,
            // group balance roughly as its square root (idle groups leave issue slots to the busy warps)
            const double cost = (double)rounds * t * cps / (sqrt(bal) * occ) * (t >= 32 ? 1.0 : 1.1);
            if (cost < best_cost * (1.0 - 1e-12)) { best_cost = cost; best_tile = t; best_cps = cps; best_R = R; best_bal = bal; }
        }
    }
    out->why = "code too large for shared memory (the node-owner kernel keeps a tile's edge state on chip)";
    if (!best_tile || (best_bal < 0.3 && !force)) return;
    p.tile = best_tile;
    p.lanes = best_tile / 4;
    p.R = best_R;
    out->threads = align_up_l(best_R * p.lanes, 32);
    out->cps = best_cps;
    p.off_x = fixed;
    p.off_m = p.off_x + g->N * best_tile * 4;
    p.off_t = p.off_m + (int)g->E * best_tile * 4;
    out->smem = p.off_t + p.trows * best_tile * 4;      // + extra_rows * tile * 4 + extra_bytes: the caller lays them out
    p.n_tiles = (int)((B + best_tile - 1) / best_tile);
    const int slots = g->sm_count * best_cps;
    // Small batches are latency-bound: four syndromes per lane leave 4x fewer threads than the edge-owner kernel's
    // one-syndrome-per-lane mapping (toy LDPC, B = 1024: 48 vs 35 us).  Take over only when the GPU is filled.
    if (p.n_tiles < slots && !force) return;
    out->grid = p.n_tiles < slots ? p.n_tiles : slots;
    out->ok = true;
    out->why = nullptr;
}

bool light_launch_info(const gd_graph* g, const gd_model* model, int64_t B, gd_launch_info* out) {
    LightPlan pl;
    plan_light(g, model, B, &pl);
    if (!pl.ok) return false;
    out->tile = pl.p.tile; out->threads = pl.threads; out->grid = pl.grid; out->smem_bytes = pl.smem;
    out->resident = 1; out->n_tiles = pl.p.n_tiles;
    return true;
}

// rc < 0: not applicable (the caller keeps the edge-owner kernel); otherwise a gd_status.
int light_decode(const gd_graph* g, const gd_model* model, const float* weights_dev, const float* x_dev, float* prob_dev,
                 float* logit_dev, uint8_t* hard_dev, int64_t B, cudaStream_t st, const Gate* gate, float* stash_dev) {
    LightPlan pl;
    plan_light(g, model, B, &pl, stash_dev != nullptr);
    if (stash_dev) {   // CGNNI training: this kernel is the only one the backward mirrors
        if (model->program != GD_PROG_CGNNI) {
            set_error("gd_decode_fwd_train: program %d has no node-owner backward", model->program);
            return GD_ERR_UNSUPPORTED;
        }
        if (!pl.ok) {
            set_error("gd_decode_fwd_train: CGNNI training needs the node-owner kernel: %s", pl.why);
            return GD_ERR_UNSUPPORTED;
        }
        pl.p.x = x_dev; pl.p.prob = prob_dev; pl.p.logit = logit_dev; pl.p.hard = hard_dev; pl.p.weights = weights_dev;
        pl.p.stash = stash_dev;
        void (*k)(const LightParams) = pl.npad == 16 ? decode_light_kernel<GD_PROG_CGNNI, 16, true> : decode_light_kernel<GD_PROG_CGNNI, 32, true>;
        GD_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, pl.smem));
        k<<<pl.grid, pl.threads, pl.smem, st>>>(pl.p);
        GD_CUDA(cudaGetLastError());
        return GD_OK;
    }
    if (!pl.ok) return -1;
    if (gate) {
        pl.p.gate_in = gate->in_flags; pl.p.gate_out = gate->out_counts; pl.p.gate_err = gate->err;
        pl.p.gate_epoch = gate->epoch; pl.p.gate_chunk_tiles = gate->chunk_tiles;
    }
    pl.p.x = x_dev; pl.p.prob = prob_dev; pl.p.logit = logit_dev; pl.p.hard = hard_dev; pl.p.weights = weights_dev;
    void (*k)(const LightParams);
    switch (model->program) {
        case GD_PROG_CGNNI:
            k = pl.npad == 16 ? decode_light_kernel<GD_PROG_CGNNI, 16>
                : pl.npad == 32 ? decode_light_kernel<GD_PROG_CGNNI, 32> : decode_light_kernel<GD_PROG_CGNNI, 0>;
            break;
        case GD_PROG_QGNNI:
            k = pl.npad == 16 ? decode_light_kernel<GD_PROG_QGNNI, 16>
                : pl.npad == 32 ? decode_light_kernel<GD_PROG_QGNNI, 32> : decode_light_kernel<GD_PROG_QGNNI, 0>;
            break;
        case GD_PROG_BP_QUANTUM: k = decode_light_kernel<GD_PROG_BP_QUANTUM, 0>; break;
        case GD_PROG_NEURAL_BP: k = decode_light_ext_kernel<GD_PROG_NEURAL_BP, 0>; break;
        case GD_PROG_GRU_CA: k = decode_light_ext_kernel<GD_PROG_GRU_CA, 32>; break;
        default: k = decode_light_kernel<GD_PROG_BP_CLASSICAL, 0>; break;
    }
    GD_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, pl.smem));
    k<<<pl.grid, pl.threads, pl.smem, st>>>(pl.p);
    GD_CUDA(cudaGetLastError());
    return GD_OK;
}

}  // namespace gd
