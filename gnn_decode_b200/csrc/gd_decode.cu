// The fused decoder: GNNI.forward of the reference (quantum/decoder_v2_4.py:272-294,
// classical/CGNNI.py:259-284, quantum/QGNNI.py:228-252, quantum/BP.py:199-219,
// classical/BP.py:239-259) as ONE persistent kernel.
//
// Design (B200-first, not a translation of the reference's ~25 eager ops per iteration):
//   * one CTA per SM loops over tiles of `tile` syndromes; the tile's edge state m[E][tile],
//     t[E][tile] lives in shared memory for all T iterations (codes whose state does not fit
//     227 KB take the streamed global-memory kernel in gd_streamed.cu instead);
//   * lanes of a warp are SYNDROMES (the batch dimension): every shared/global access of the
//     state is unit-stride across lanes (conflict-free / coalesced), the graph tables and MLP
//     weights are warp-uniform broadcasts, and there is no divergence and no atomic anywhere;
//   * thread (s, r) owns syndrome s and the edges / nodes e == r (mod R): node sums are
//     computed in ascending edge order (deterministic, same order as the CPU index_add_ of
//     the reference), the per-edge MLPs are evaluated for EB edges at a time in registers;
//   * the tile's input slab x[tile][V+C] is fetched with one bulk async copy (TMA, UBLKCP)
//     completing on an mbarrier; outputs go out as 128-bit coalesced stores;
//   * the scalar (1 -> h -> 1) MLPs are not summed per hidden unit: the ReLU ones are evaluated
//     as the piecewise-linear functions they are (exact), decoder_v2_4's two Softplus ones from
//     per-launch cubic tables on their compact domains with an in-kernel error bound and automatic
//     fall-back (gd_math.cuh: PwlSmem, CubicTab); what remains MUFU-bound is the 2-input
//     variable-phase MLP (1 ex2 + half an lg2 per hidden unit, the other half on the FMA pipe);
//   * messages of degree-1 variables are iteration-invariant and are computed once.
#include "gd_common.cuh"
#include "gd_math.cuh"
#include "gd_decode.cuh"
#include "gd_lean.cuh"
#include "gd_options.cuh"
#include <stdlib.h>
#include <string.h>
#include <algorithm>

namespace gd {

constexpr int kMaxThreads = 1024;   // largest CTA; kernels are instantiated for 512 (<=128 regs) and 1024 (<=64 regs)

// ---------------- PTX helpers: mbarrier + bulk async copy (TMA 1-D) ----------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

// Graph tables: 16-bit copies in shared memory (warp-uniform reads: broadcast, conflict-free).
struct Tables {
    const uint16_t *edge_var, *edge_chk, *var_ptr, *var_edges, *chk_ptr, *chk_edges, *vlist;
    const uint16_t *vsib, *csib;     // [E] sibling edge on the same variable, [E][3] sibling edges on the same check (0xFFFF = none)
    __device__ __forceinline__ static int ld(const uint16_t* p, int i) { return p[i]; }
};

__device__ __forceinline__ void stage_mlp(float* dst, int hp, int hid, const float* w1, int w1_stride,
                                          bool two_in, const float* b1, const float* w2, float s1, float s2,
                                          int tid, int nthr) {
    // dst rows: w1a[hp] | w1b[hp] | b1[hp] | w2[hp]
    for (int k = tid; k < hp; k += nthr) {
        const bool in = k < hid;
        dst[k] = in ? w1[k * w1_stride] * s1 : 0.f;
        dst[hp + k] = (in && two_in) ? w1[k * w1_stride + 1] * s1 : 0.f;
        dst[2 * hp + k] = in ? b1[k] * s1 : 0.f;
        dst[3 * hp + k] = in ? w2[k] * s2 : 0.f;
    }
}

// kEB = edges evaluated together per thread (register blocking of the MLP: weights are loaded
// once per 4 hidden units and reused for kEB edges).
template <int PROG, int MAXT, int kEB, int NPOLY>
__global__ void __launch_bounds__(MAXT, 1) decode_kernel(const DecodeParams p) {
    extern __shared__ __align__(128) unsigned char smem[];
    // (the deferred pass of the table kernel is launched with programmatic stream serialisation: a no-op otherwise)
    gd::pdl_enter();
    constexpr bool kIsBP = (PROG == GD_PROG_BP_QUANTUM || PROG == GD_PROG_BP_CLASSICAL);
    constexpr bool kSoftplus = (PROG == GD_PROG_V2_4);
    constexpr bool kNBP = (PROG == GD_PROG_NEURAL_BP);   // sum-product + per-edge weights (quantum/neural_BP.py)
    constexpr bool kGRU = (PROG == GD_PROG_GRU_CA);      // MLP + GRUCell updates (quantum/QGNNNI_ca.py)
    constexpr bool kV3 = (PROG == GD_PROG_V3_0);         // 2-input ReLU MLPs + GRUCell updates, second read-out at the checks (quantum/decoder_v3_0.py)
    constexpr bool kV122 = (PROG == GD_PROG_V1_2_2);     // Tanh-MLP variable phase, sum-product check phase, a read-out per iteration (quantum/decoder_v1_2_2.py)
    constexpr bool kV241 = (PROG == GD_PROG_V2_4_1);     // decoder_v2_4 with un-tied layers, per-edge-type weights, gated residual (quantum/decoder_v2_4_1.py)
    // ReLU programs: NPOLY carries NPAD -- > 0 evaluates their 1->h->1 MLPs as piecewise-linear tables (gd_math.cuh)
    constexpr int kNPAD = (PROG == GD_PROG_CGNNI || PROG == GD_PROG_QGNNI || kGRU) ? (NPOLY > 0 ? NPOLY : 0) : 0;

    uint64_t* bar = reinterpret_cast<uint64_t*>(smem);
    float* wsm = reinterpret_cast<float*>(smem + p.off_w);
    float* xs = reinterpret_cast<float*>(smem + p.off_x);
    float* node = reinterpret_cast<float*>(smem + p.off_node);
    const int tile = p.tile, R = p.R, E = p.E, V = p.V, C = p.C, N = p.N, hp = p.hp;
    float* node2 = node + (size_t)p.maxvc * tile;  // sum-product programs only (allocated only then)
    float* m_st = reinterpret_cast<float*>(smem + p.off_m);
    float* t_st = reinterpret_cast<float*>(smem + p.off_t);
    const int tid = threadIdx.x, nthr = blockDim.x;
    const int s = tid % tile, r = tid / tile;
    long long B_eff = p.B;
    int n_tiles = p.n_tiles;
    const int* didx = nullptr;
    if (p.defer_count) {
        const int cnt = *p.defer_count;
        if (cnt == 0) return;                                  // nothing was deferred: no prologue either
        if (cnt > 0) {
            B_eff = cnt;
            didx = p.defer_idx;
            n_tiles = (cnt + tile - 1) / tile;
        }
    }

    // ---- prologue: tables and (pre-scaled) weights into shared memory ----
    Tables tb;
    {
        uint16_t* tab = reinterpret_cast<uint16_t*>(smem + p.off_tab);
        uint16_t* d_ev = tab;
        uint16_t* d_ec = d_ev + E;
        uint16_t* d_vp = d_ec + E;
        uint16_t* d_ve = d_vp + (V + 1);
        uint16_t* d_cp = d_ve + E;
        uint16_t* d_ce = d_cp + (C + 1);
        uint16_t* d_vl = d_ce + E;
        for (int i = tid; i < E; i += nthr) {
            d_vl[i] = (uint16_t)p.tb.vlist[i];
            d_ev[i] = (uint16_t)p.tb.edge_var[i];
            d_ec[i] = (uint16_t)p.tb.edge_chk[i];
            d_ve[i] = (uint16_t)p.tb.var_edges[i];
            d_ce[i] = (uint16_t)p.tb.chk_edges[i];
        }
        for (int i = tid; i <= V; i += nthr) d_vp[i] = (uint16_t)p.tb.var_ptr[i];
        for (int i = tid; i <= C; i += nthr) d_cp[i] = (uint16_t)p.tb.chk_ptr[i];
        tb.edge_var = d_ev; tb.edge_chk = d_ec; tb.var_ptr = d_vp;
        tb.var_edges = d_ve; tb.chk_ptr = d_cp; tb.chk_edges = d_ce; tb.vlist = d_vl;
        tb.vsib = d_vl + E; tb.csib = d_vl + 2 * E;
    }
    // decoder_v2_4 on low-degree graphs (every surface / toric code: variable degree <= 2, check degree <= 4): the
    // "sum over siblings minus self" is just the one sibling message (variables) or the sum of <= 3 of them (checks), read
    // directly -- no node-sum passes, no node arrays, two barriers per iteration instead of four.
    const bool vdir = PROG == GD_PROG_V2_4 && p.vdirect, cdir = PROG == GD_PROG_V2_4 && p.cdirect;
    if (vdir || cdir) {
        __syncthreads();                                   // the 16-bit graph tables are complete
        uint16_t* vs = const_cast<uint16_t*>(tb.vsib);
        uint16_t* cs = const_cast<uint16_t*>(tb.csib);
        for (int e = tid; e < E; e += nthr) {
            const int v = tb.edge_var[e], vb = tb.var_ptr[v], vd = tb.var_ptr[v + 1] - vb;
            vs[e] = vd == 2 ? (tb.var_edges[vb] == e ? tb.var_edges[vb + 1] : tb.var_edges[vb]) : (uint16_t)0xFFFF;
            const int c = tb.edge_chk[e], cb = tb.chk_ptr[c], ce = tb.chk_ptr[c + 1];
            int n = 0;
            for (int i = cb; i < ce && n < 3; ++i)
                if (tb.chk_edges[i] != e) cs[3 * e + n++] = tb.chk_edges[i];       // ascending edge id
            for (; n < 3; ++n) cs[3 * e + n] = (uint16_t)0xFFFF;
        }
    }
    MlpSmem W1{}, W2{}, W3{};
    const float* gru = nullptr;   // GRU_CA: the two GRUCell(1,1) parameter sets, [2][12] in shared memory
    PwlSmem P1{}, P2{}, P3{};
    if constexpr (kNPAD > 0) {
        // MLP k of the packed weights: CGNNI/QGNNI  k = 0 check phase, 1 read-out;  GRU_CA  k = 0 ggc1.mlp1, 1 ggc2.mlp2, 2 mlp
        constexpr int kM = kGRU ? 3 : 2;
        const int h = p.hid, warp = tid >> 5, nwarp = nthr >> 5;
        for (int k = warp; k < kM; k += nwarp) {
            const float* w = p.weights + k * (3 * h + 1) + (kGRU ? k * 12 : 0);
            float* t = wsm + k * p.wslot;
            pwl_build(t, reinterpret_cast<float2*>(t + kNPAD), kNPAD, w, w + h, w + 2 * h, w[3 * h], h, tid & 31);
        }
        const PwlSmem Pa{wsm, reinterpret_cast<const float2*>(wsm + kNPAD)};
        const PwlSmem Pb{wsm + p.wslot, reinterpret_cast<const float2*>(wsm + p.wslot + kNPAD)};
        const PwlSmem Pc{wsm + 2 * p.wslot, reinterpret_cast<const float2*>(wsm + 2 * p.wslot + kNPAD)};
        if constexpr (kGRU) {
            P1 = Pa; P2 = Pb; P3 = Pc;
            float* gs = wsm + 3 * p.wslot;
            if (tid < 24) gs[tid] = p.weights[(tid < 12 ? 3 * h + 1 : 2 * (3 * h + 1)) + tid];
            gru = gs;
        } else {
            P2 = Pa; P3 = Pb;
        }
    } else if constexpr (kGRU) {
        const float* w = p.weights;
        const int h = p.hid;
        float* slot = wsm;
        float* gs = wsm + 3 * p.wslot;
        for (int k = 0; k < 3; ++k) {       // ggc1.mlp1 | ggc1.rnn | ggc2.mlp2 | ggc2.rnn | mlp
            stage_mlp(slot, hp, h, w, 1, false, w + h, w + 2 * h, 1.f, 1.f, tid, nthr);
            const MlpSmem Wk{slot, slot + hp, slot + 2 * hp, slot + 3 * hp, w[3 * h]};
            if (k == 0) W1 = Wk; else if (k == 1) W2 = Wk; else W3 = Wk;
            w += 3 * h + 1;
            slot += p.wslot;
            if (k < 2) {
                if (tid < 12) gs[k * 12 + tid] = w[tid];
                w += 12;
            }
        }
        gru = gs;
    } else if constexpr (kV3) {
        // ggc1.mlp1 (2 -> h -> 1) | ggc1.rnn1 | ggc2.mlp2 (2 -> h -> 1) | ggc2.rnn2 | mlp (1 -> h -> 1)
        const float* w = p.weights;
        const int h = p.hid;
        float* slot = wsm;
        float* gs = wsm + 3 * p.wslot;
        for (int k = 0; k < 2; ++k) {
            stage_mlp(slot, hp, h, w, 2, true, w + 2 * h, w + 3 * h, 1.f, 1.f, tid, nthr);
            const MlpSmem Wk{slot, slot + hp, slot + 2 * hp, slot + 3 * hp, w[4 * h]};
            if (k == 0) W1 = Wk; else W2 = Wk;
            w += 4 * h + 1;
            slot += p.wslot;
            if (tid < 12) gs[k * 12 + tid] = w[tid];
            w += 12;
        }
        stage_mlp(slot, hp, h, w, 1, false, w + h, w + 2 * h, 1.f, 1.f, tid, nthr);
        W3 = MlpSmem{slot, slot + hp, slot + 2 * hp, slot + 3 * hp, w[3 * h]};
        gru = gs;
    } else if constexpr (kV241) {
        // per iteration (staged at its start): layers.{2l}.mlp1 | W[8] | W_p[8] | layers.{2l+1}.mlp; once: mlp | W[8] | W_p[8] | alpha | beta
        const int h = p.hid;
        const float* w = p.weights + (size_t)p.T * (6 * h + 18);
        float* slot = wsm + 2 * p.wslot;
        stage_mlp(slot, hp, h, w, 1, false, w + h, w + 2 * h, kLog2e, kLn2, tid, nthr);
        W3 = MlpSmem{slot, slot + hp, slot + 2 * hp, slot + 3 * hp, w[3 * h]};
        float* tw = wsm + 3 * p.wslot;                 // [0..15] this layer's W | W_p, [16..31] the read-out's, [32..33] the gates
        if (tid < 16) tw[16 + tid] = w[3 * h + 1 + tid];
        if (tid < 2) tw[32 + tid] = sigmoid_fast(w[3 * h + 17 + tid]);
        // edge types (decoder_v2_4_1.py:211-236): rank of the edge among its check's edges in ascending variable order, + 4 for
        // the second half of the checks (`idx > cols / 2 - 1`)
        __syncthreads();                               // the 16-bit graph tables are complete
        uint16_t* et = const_cast<uint16_t*>(tb.csib);
        for (int e = tid; e < E; e += nthr) {
            const int c = tb.edge_chk[e], v = tb.edge_var[e];
            int rank = 0;
            for (int i = tb.chk_ptr[c]; i < tb.chk_ptr[c + 1]; ++i) {
                const int e2 = tb.chk_edges[i], v2 = tb.edge_var[e2];
                rank += (v2 < v || (v2 == v && e2 < e)) ? 1 : 0;
            }
            et[e] = (uint16_t)((rank & 3) + (2 * c > C - 2 ? 4 : 0));
        }
    } else if constexpr (kV122) {
        // ggc1.mlp | mlp, both 2 -> h -> 1 Tanh: first layers pre-scaled by 2 log2(e) (mlp_tanh2)
        const float* w = p.weights;
        const int h = p.hid;
        const float s1 = 2.0f * kLog2e;
        stage_mlp(wsm, hp, h, w, 2, true, w + 2 * h, w + 3 * h, s1, 1.f, tid, nthr);
        W1 = MlpSmem{wsm, wsm + hp, wsm + 2 * hp, wsm + 3 * hp, w[4 * h]};
        w += 4 * h + 1;
        float* slot = wsm + p.wslot;
        stage_mlp(slot, hp, h, w, 2, true, w + 2 * h, w + 3 * h, s1, 1.f, tid, nthr);
        W3 = MlpSmem{slot, slot + hp, slot + 2 * hp, slot + 3 * hp, w[4 * h]};
    } else if constexpr (!kIsBP && !kNBP) {
        const float* w = p.weights;
        const int h = p.hid;
        const float s1 = kSoftplus ? kLog2e : 1.f, s2 = kSoftplus ? kLn2 : 1.f;
        float* slot = wsm;
        if constexpr (PROG == GD_PROG_V2_4) {  // ggc1.mlp: 2 -> h -> 1
            stage_mlp(slot, hp, h, w, 2, true, w + 2 * h, w + 3 * h, s1, s2, tid, nthr);
            W1 = MlpSmem{slot, slot + hp, slot + 2 * hp, slot + 3 * hp, w[4 * h]};
            w += 4 * h + 1;
            slot += 4 * hp;
        }
        stage_mlp(slot, hp, h, w, 1, false, w + h, w + 2 * h, s1, s2, tid, nthr);  // check-phase MLP
        W2 = MlpSmem{slot, slot + hp, slot + 2 * hp, slot + 3 * hp, w[3 * h]};
        w += 3 * h + 1;
        slot += 4 * hp;
        stage_mlp(slot, hp, h, w, 1, false, w + h, w + 2 * h, s1, s2, tid, nthr);  // read-out MLP
        W3 = MlpSmem{slot, slot + hp, slot + 2 * hp, slot + 3 * hp, w[3 * h]};
    }
    // V2_4: tabulate the 1 -> h -> 1 check-phase MLP on its compact domain (gd_math.cuh, CubicTab)
    // V2_4: the two 1 -> h -> 1 Softplus MLPs as cubic tables on their compact domains (gd_math.cuh, CubicTab).
    //   check phase (decoder_v2_4.py:257): |ext| <= max check degree - 1 (a sum of tanh values minus one of them);
    //   read-out (decoder_v2_4.py:291, per edge on m): m starts at 0 and every iteration adds mlp2(ext) * (+-1), so
    //     |m| <= T * max|mlp2| -- known once the check table exists; lanes outside it (possible only when the
    //     caller's check inputs are not +-1) take the direct path.
    // Node values come from the same packed MUFU/FMA evaluation the direct path uses, node derivatives from 4th-order
    // central differences of them; the interpolation-error bound h^4/384 * 0.125 * sum|w2| w1^4 is checked from the
    // raw weights (identical arithmetic in every thread -> a uniform decision), else the direct evaluation stays.
    CubicTab ctab{}, rtab{};
    bool use_ctab = false, use_rtab = false;
    float rtab_R = 0.f;
    if constexpr (PROG == GD_PROG_V2_4) {
        float* const F = reinterpret_cast<float*>(smem + p.off_x);        // scratch: the state regions are idle here
        const int scratch_floats = p.scratch_bytes >> 2;
        if (p.ctab_n > 0 && p.ctab_n + 8 <= scratch_floats) {
            __syncthreads();                                              // the staged (pre-scaled) weights are visible
            const float step = 2.0f * p.ctab_R / (float)p.ctab_n;
            use_ctab = cubic_tab_bound(p.weights + 4 * p.hid + 1, p.hid, step) <= 1e-7f;
            if (use_ctab) {
                float4* dst = reinterpret_cast<float4*>(smem + p.off_ctab);
                const float fm = cubic_tab_build(W2, hp, p.ctab_R, p.ctab_n, dst, F, tid, nthr);
                ctab = CubicTab{dst, 1.0f / step, p.ctab_R / step, (float)p.ctab_n - 0.001f};
                if (p.rtab_n > 0 && p.T > 0 && p.rtab_n + 8 <= scratch_floats) {
                    unsigned int* fmax_bits = reinterpret_cast<unsigned int*>(smem + 8);     // after the 8-byte mbarrier
                    if (tid == 0) *fmax_bits = 0u;
                    __syncthreads();
                    atomicMax(fmax_bits, __float_as_uint(fm));            // non-negative floats order like uints
                    __syncthreads();
                    // 1.02: a cubic piece may overshoot its end values slightly inside an interval
                    rtab_R = (float)p.T * (__uint_as_float(*fmax_bits) * 1.02f + 1e-6f);
                    const float rstep = 2.0f * rtab_R / (float)p.rtab_n;
                    use_rtab = cubic_tab_bound(p.weights + 7 * p.hid + 2, p.hid, rstep) <= 4e-6f;   // feeds the logit directly (x degree <= 4), not the iteration: 1000x below the parity bar
                    if (use_rtab) {
                        float4* rdst = reinterpret_cast<float4*>(smem + p.off_rtab);
                        cubic_tab_build(W3, hp, rtab_R, p.rtab_n, rdst, F, tid, nthr);
                        rtab = CubicTab{rdst, 1.0f / rstep, rtab_R / rstep, (float)p.rtab_n - 0.001f};
                    }
                }
            }
        }
    }
    // V2_4 variable phase (decoder_v2_4.py:254-255, mlp([ext, prior])): when every variable of a syndrome carries the same
    // prior (the reference's gen_syn: x = log((1-p)/p) for all of them) the update is a function of ext alone, f_p(ext).
    // A CTA keeps cubic tables of f_p for the distinct p it meets (up to vtab_k; later tiles reuse them); syndromes with
    // non-uniform priors, more distinct values than slots, or |ext| beyond the tabulated domain take the direct path.
    // Domain half-width: the largest R whose interpolation-error bound (same formula, first-input weights) is <= 2e-7.
    bool use_vtab = false;
    float vtab_R = 0.f, vtab_inv_h = 0.f;
    float* const vt_vals = reinterpret_cast<float*>(smem + p.off_vmeta + 16);      // [16] prior of table k
    int* const vt_cnt = reinterpret_cast<int*>(smem + p.off_vmeta);               // tables built so far
    int* const vt_lane = reinterpret_cast<int*>(smem + p.off_vmeta + 16 + 16 * 4); // [tile] table of lane s (-1: direct)
    if constexpr (PROG == GD_PROG_V2_4) {
        // (a deferred LIST is evaluated directly, per item: its results must not depend on what else was deferred)
        if (p.vtab_n > 0 && use_ctab && tile <= 128 && E * tile >= p.vtab_n + 8 && !didx) {
            float m4 = 0.f;
            for (int k = 0; k < p.hid; ++k) {
                float a = __ldg(p.weights + 2 * k);                       // w1[k][0]: the ext input
                a *= a;
                m4 = fmaf(fabsf(__ldg(p.weights + 3 * p.hid + k)), a * a, m4);
            }
            const float hmax = sqrtf(sqrtf(2e-7f * 384.0f / (0.125f * fmaxf(m4, 1e-20f))));
            vtab_R = fminf(0.5f * (float)p.vtab_n * hmax, 1e4f);
            use_vtab = vtab_R >= 0.5f;                                    // a narrower domain would mostly fall back
            if (use_rtab && rtab_R > 0.f) vtab_R = fminf(vtab_R, rtab_R * (float)(p.vdirect ? 1 : 8));   // |m| <= rtab_R: no need to go wider
            vtab_inv_h = 0.5f * (float)p.vtab_n / vtab_R;
            if (tid == 0) *vt_cnt = 0;
        }
    }
    fence_proxy_async();   // the prologue used the slab region as generic-proxy scratch; the bulk copies (async proxy) come next
    if (tid == 0) {
        mbar_init(bar, 1);
        fence_mbar_init();
    }
    __syncthreads();

    uint32_t parity = 0;
    const int n_iter = (E + R - 1) / R;  // edges per thread (interleaved ownership e = r + i*R)

    for (int tix = blockIdx.x; tix < n_tiles; tix += gridDim.x) {
        const long long s0 = (long long)tix * tile;
        const int nvalid = (int)min((long long)tile, B_eff - s0);
        const float* xg = p.x + s0 * N;
        const int n_in = nvalid * N;
        const uint32_t bulk_bytes = didx ? 0u : ((uint32_t)n_in * 4u) & ~15u;
        // ---- input slab: one bulk async copy (TMA) + scalar tail; zero the state ----
        if (tid == 0) {
            fence_proxy_async();  // order earlier generic reads of xs before the async write
            mbar_arrive_expect_tx(bar, bulk_bytes);
            if (bulk_bytes) bulk_g2s(xs, xg, bulk_bytes, bar);
        }
        if (didx) {                                            // listed syndromes: gather their rows
            for (int i = tid; i < tile * N; i += nthr) {
                const int q = i / N;
                xs[i] = q < nvalid ? __ldcg(p.x + (long long)__ldg(didx + s0 + q) * N + (i - q * N)) : 0.f;
            }
        } else {
            for (int i = (int)(bulk_bytes >> 2) + tid; i < tile * N; i += nthr) xs[i] = i < n_in ? __ldcg(xg + i) : 0.f;
        }
        for (int i = 0; i < n_iter; ++i) {
            const int e = r + i * R;
            if (e < E) m_st[(size_t)e * tile + s] = 0.f;
        }
        mbar_wait(bar, parity);
        parity ^= 1u;
        __syncthreads();
        const float* xrow = xs + (size_t)s * N;  // prior = xrow[0..V), check input = xrow[V..V+C)
        int my_vtab = -1;
        if constexpr (PROG == GD_PROG_V2_4) {
            if (use_vtab) {
                const int old_cnt = *vt_cnt;
                float* const lane_prior = t_st;                              // t is idle until the first variable phase
                if (r == 0) {
                    const float pv = xrow[0];
                    bool uni = s < nvalid;
                    for (int v = 1; v < V; ++v) uni = uni && (__float_as_uint(xrow[v]) == __float_as_uint(pv));
                    int k = -1;                                           // -1: direct (non-uniform priors / padding lane)
                    if (uni) {                                            // every lane searches the cache itself, in parallel
                        k = 0;
                        while (k < old_cnt && __float_as_uint(vt_vals[k]) != __float_as_uint(pv)) ++k;
                        if (k == old_cnt) k = -2;                         // -2: uniform, but its prior has no table yet
                    }
                    lane_prior[s] = pv;
                    vt_lane[s] = k;
                }
                __syncthreads();
                if (tid == 0) {                                           // only priors met for the first time are inserted serially
                    int cnt = old_cnt;
                    bool overflow = false;
                    for (int q = 0; q < tile && !overflow; ++q) {
                        if (vt_lane[q] != -2) continue;
                        const unsigned int pb = __float_as_uint(lane_prior[q]);
                        int k = old_cnt;
                        while (k < cnt && __float_as_uint(vt_vals[k]) != pb) ++k;
                        if (k == cnt) {
                            if (cnt < p.vtab_k) vt_vals[cnt++] = lane_prior[q];
                            else overflow = true;
                        }
                        vt_lane[q] = k;
                    }
                    if (overflow) {       // more distinct priors than slots: the whole tile goes direct (warps would diverge otherwise)
                        cnt = old_cnt;
                        for (int q = 0; q < tile; ++q) vt_lane[q] = -1;
                    }
                    *vt_cnt = cnt;
                }
                __syncthreads();
                const int new_cnt = *vt_cnt;
                for (int k = old_cnt; k < new_cnt; ++k)                       // CTA-uniform bounds
                    cubic_tab_build<true>(W1, hp, vtab_R, p.vtab_n, reinterpret_cast<float4*>(smem + p.off_vtab) + (size_t)k * p.vtab_n,
                                          t_st, tid, nthr, vt_vals[k]);
                my_vtab = vt_lane[s];
                __syncthreads();
            }
        }
        const CubicTab vtab{reinterpret_cast<const float4*>(smem + p.off_vtab) + (size_t)(my_vtab > 0 ? my_vtab : 0) * p.vtab_n,
                            vtab_inv_h, vtab_R * vtab_inv_h, (float)p.vtab_n - 0.001f};

        // read-out as a callable: GRU_CA with GD_FLAG_ALL_ITERS emits one prediction per iteration
        auto emit = [&](const long long out_off) {
            // ---- read-out: logits staged as [tile][V] in the node region ----
            if constexpr (kV241) {                 // decoder_v2_4_1.py:341-345: mlp(m) W[type], summed at the variable with prior W_p[type]
                const float* tw = wsm + 3 * p.wslot;
                const uint16_t* et = tb.csib;
                for (int i0 = 0; i0 < n_iter; i0 += kEB) {
                    float x0[kEB], o[kEB];
                    int ee[kEB];
#pragma unroll
                    for (int j = 0; j < kEB; ++j) {
                        const int e = r + (i0 + j) * R;
                        ee[j] = e;
                        x0[j] = m_st[(size_t)(e < E ? e : E - 1) * tile + s];
                    }
                    mlp_softplus<kEB, false>(W3, hp, x0, x0, o);
#pragma unroll
                    for (int j = 0; j < kEB; ++j)
                        if (ee[j] < E) {
                            const int ty = et[ee[j]];
                            t_st[(size_t)ee[j] * tile + s] = fmaf(o[j], tw[16 + ty], xrow[tb.ld(tb.edge_var, ee[j])] * tw[24 + ty]);
                        }
                }
                __syncthreads();
            }
            if constexpr (PROG == GD_PROG_V2_4) {  // per-EDGE MLP, then sum at the variable
                for (int i0 = 0; i0 < n_iter; i0 += kEB) {
                    float x0[kEB], o[kEB];
                    int ee[kEB];
    #pragma unroll
                    for (int j = 0; j < kEB; ++j) {
                        const int e = r + (i0 + j) * R;
                        ee[j] = e;
                        x0[j] = m_st[(size_t)(e < E ? e : E - 1) * tile + s];
                        if (p.stash && e < E && s < nvalid) p.stash[((size_t)p.T * 2 * E + e) * (size_t)p.B + s0 + s] = x0[j];
                    }
                    bool in_range = use_rtab;
    #pragma unroll
                    for (int j = 0; j < kEB; ++j) in_range = in_range && fabsf(x0[j]) <= rtab_R;
                    if (in_range) {
    #pragma unroll
                        for (int j = 0; j < kEB; ++j) o[j] = cubic_tab_eval(rtab, x0[j]);
                    } else if constexpr (NPOLY >= 0) mlp_softplus_x2<kEB, false, (NPOLY > 0 ? NPOLY : 0)>(W3, hp, x0, x0, o);
                    else mlp_softplus<kEB, false>(W3, hp, x0, x0, o);
    #pragma unroll
                    for (int j = 0; j < kEB; ++j)
                        if (ee[j] < E) t_st[(size_t)ee[j] * tile + s] = o[j];
                }
                __syncthreads();
            }
            float* stage = node;  // [tile][V]
            for (int v = r; v < V; v += R) {
                const int b = tb.ld(tb.var_ptr, v), e_end = tb.ld(tb.var_ptr, v + 1);
                const float* src = (PROG == GD_PROG_V2_4 || kV241) ? t_st : m_st;
                float acc = 0.f, acc_p = 0.f;
                for (int i = b; i < e_end; ++i) {
                    const int e = tb.ld(tb.var_edges, i);
                    if constexpr (kNBP) {   // neural_BP.py:308-312: scatter(m W) + scatter(prior W_p), no bare prior
                        const float* wo = p.weights + (size_t)p.T * 2 * E;
                        acc += src[(size_t)e * tile + s] * __ldg(wo + e);
                        acc_p += xrow[v] * __ldg(wo + E + e);
                    } else {
                        acc += src[(size_t)e * tile + s];
                    }
                }
                float lg = kNBP ? acc + acc_p : ((kGRU || kV3 || kV122 || kV241) ? acc : acc + xrow[v]);   // QGNNNI_ca.py:241-245: mlp(sum), no prior
                if constexpr (kV3) {            // decoder_v3_0.py:275: mlp(sum) + x
                    float xi[1] = {lg}, oo[1];
                    mlp_relu<1>(W3, hp, xi, oo);
                    lg = oo[0] + xrow[v];
                }
                if constexpr (kV122) {          // decoder_v1_2_2.py:275-278: mlp([sum, prior])
                    float xi[1] = {lg}, xp[1] = {xrow[v]}, oo[1];
                    mlp_tanh2<1>(W3, hp, xi, xp, oo);
                    lg = oo[0];
                }
                if constexpr (kGRU) {
                    float xi[1] = {lg}, oo[1];
                    if constexpr (kNPAD > 0) oo[0] = pwl_eval<kNPAD>(P3, xi[0]);
                    else mlp_relu<1>(W3, hp, xi, oo);
                    lg = oo[0];
                }
                if constexpr (PROG == GD_PROG_CGNNI || PROG == GD_PROG_QGNNI) {
                    float xi[1] = {lg}, oo[1];
                    if constexpr (kNPAD > 0) oo[0] = pwl_eval<kNPAD>(P3, xi[0]);
                    else mlp_relu<1>(W3, hp, xi, oo);
                    lg = oo[0];
                }
                stage[(size_t)s * V + v] = lg;
            }
            __syncthreads();
            // ---- outputs: coalesced 128-bit stores of prob / logit, 32-bit stores of hard bytes ----
            {
                const int total = nvalid * V;
                const long long g0 = out_off + s0 * V;  // s0 * V is a multiple of 8 elements: tile % 8 == 0
                const bool vec_ok = (g0 & 3) == 0 && !didx;
                constexpr bool kClamp = (PROG == GD_PROG_CGNNI || PROG == GD_PROG_BP_CLASSICAL || PROG == GD_PROG_GRU_CA);
                for (int i = tid * 4; i < total; i += nthr * 4) {
                    float l[4], pr[4];
                    const int n = min(4, total - i);
    #pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        l[j] = j < n ? stage[i + j] : 0.f;
                        pr[j] = sigmoid_neg(l[j]);
                        if (kClamp) pr[j] = fminf(fmaxf(pr[j], 1e-7f), 1.0f - 1e-7f);
                    }
                    if (n == 4 && vec_ok) {
                        if (p.prob) *reinterpret_cast<float4*>(p.prob + g0 + i) = make_float4(pr[0], pr[1], pr[2], pr[3]);
                        if (p.logit) *reinterpret_cast<float4*>(p.logit + g0 + i) = make_float4(l[0], l[1], l[2], l[3]);
                        if (p.hard)
                            *reinterpret_cast<uchar4*>(p.hard + g0 + i) =
                                make_uchar4(pr[0] > 0.5f, pr[1] > 0.5f, pr[2] > 0.5f, pr[3] > 0.5f);
                    } else {
                        for (int j = 0; j < n; ++j) {
                            long long o = g0 + i + j;
                            if (didx) {                        // scatter back to the listed rows
                                const int q = (i + j) / V;
                                o = out_off + (long long)__ldg(didx + s0 + q) * V + (i + j - q * V);
                            }
                            if (p.prob) p.prob[o] = pr[j];
                            if (p.logit) p.logit[o] = l[j];
                            if (p.hard) p.hard[o] = pr[j] > 0.5f;
                        }
                    }
                }
                if (p.hard_bits) {
                    const int vw = (V + 31) >> 5;
                    for (int i = tid; i < nvalid * vw; i += nthr) {
                        const int q = i / vw, w = i - q * vw;
                        uint32_t word = 0u;
                        for (int b = 0; b < 32 && w * 32 + b < V; ++b)
                            word |= (sigmoid_neg(stage[q * V + w * 32 + b]) > 0.5f ? 1u : 0u) << b;
                        const long long row = didx ? (long long)__ldg(didx + s0 + q) : s0 + q;
                        p.hard_bits[row * vw + w] = word;     // (single read-out only: not combined with GD_FLAG_ALL_ITERS)
                    }
                }
            }
            __syncthreads();  // xs / node / state are rewritten by the next tile
        };
        for (int it = 0; it < p.T; ++it) {
            // NEURAL_BP: this layer's per-edge weights W_l[E] | W_p,l[E] (warp-uniform reads)
            const float* wl = kNBP ? p.weights + (size_t)it * 2 * E : nullptr;
            if constexpr (kV241) {     // un-tied layers: this iteration's two MLPs and type tables (the last readers of the old ones are behind a barrier)
                const int h = p.hid;
                const float* w = p.weights + (size_t)it * (6 * h + 18);
                stage_mlp(wsm, hp, h, w, 1, false, w + h, w + 2 * h, kLog2e, kLn2, tid, nthr);
                W1 = MlpSmem{wsm, wsm + hp, wsm + 2 * hp, wsm + 3 * hp, w[3 * h]};
                float* tw = wsm + 3 * p.wslot;
                if (tid < 16) tw[tid] = w[3 * h + 1 + tid];
                w += 3 * h + 17;
                float* slot = wsm + p.wslot;
                stage_mlp(slot, hp, h, w, 1, false, w + h, w + 2 * h, kLog2e, kLn2, tid, nthr);
                W2 = MlpSmem{slot, slot + hp, slot + 2 * hp, slot + 3 * hp, w[3 * h]};
                __syncthreads();
            }
            // ---- V1: per-variable sums of m (ascending edge id) ----
            if (!vdir) {
            for (int v = r; v < V; v += R) {
                const int b = tb.ld(tb.var_ptr, v), e_end = tb.ld(tb.var_ptr, v + 1);
                float acc = 0.f;
                for (int i = b; i < e_end; ++i) {
                    const int e = tb.ld(tb.var_edges, i);
                    float mv = m_st[(size_t)e * tile + s];
                    if constexpr (kNBP) mv *= __ldg(wl + e);
                    if constexpr (kV241) mv *= (wsm + 3 * p.wslot)[tb.csib[e]];
                    acc += mv;
                }
                node[v * tile + s] = acc;
            }
            __syncthreads();
            }
            // ---- V2: variable-phase message + the `pre` of the check phase, per edge ----
            if constexpr (PROG == GD_PROG_V2_4) {
                // A degree-1 variable has no sibling edge: ext == 0 in every iteration, so its message
                // mlp([0, prior]) is computed in the first iteration only (vlist puts those edges last).
                // Training keeps all edges: the backward kernel wants every iteration's stash.
                const int n_act = (it == 0 || p.stash) ? E : p.n_vact;
                const int n_it_act = (n_act + R - 1) / R;
                for (int i0 = 0; i0 < n_it_act; i0 += kEB) {
                    float x0[kEB], x1[kEB], o[kEB], mo[kEB];
                    int ee[kEB];
#pragma unroll
                    for (int j = 0; j < kEB; ++j) {
                        const int li = r + (i0 + j) * R;
                        const int e = li < n_act ? tb.ld(tb.vlist, li) : E;
                        ee[j] = e;
                        const int ec = e < E ? e : E - 1;
                        const int v = tb.ld(tb.edge_var, ec);
                        mo[j] = m_st[(size_t)ec * tile + s];
                        if (vdir) {
                            const int sb = tb.ld(tb.vsib, ec);
                            x0[j] = sb != 0xFFFF ? m_st[(size_t)sb * tile + s] : 0.f;
                        } else {
                            x0[j] = node[v * tile + s] - mo[j];
                        }
                        x1[j] = xrow[v];
                    }
                    bool vt_ok = my_vtab >= 0;
#pragma unroll
                    for (int j = 0; j < kEB; ++j) vt_ok = vt_ok && fabsf(x0[j]) <= vtab_R;
                    if (!vt_ok) {
                        if constexpr (NPOLY >= 0) mlp_softplus_x2<kEB, true, (NPOLY > 0 ? NPOLY : 0)>(W1, hp, x0, x1, o);
                        else mlp_softplus<kEB, true>(W1, hp, x0, x1, o);
                    }
                    if (my_vtab >= 0) {     // per item, so a result never depends on which items share a register batch
#pragma unroll
                        for (int j = 0; j < kEB; ++j)
                            if (vt_ok || fabsf(x0[j]) <= vtab_R) o[j] = cubic_tab_eval(vtab, x0[j]);
                    }
#pragma unroll
                    for (int j = 0; j < kEB; ++j)
                        if (ee[j] < E) {
                            t_st[(size_t)ee[j] * tile + s] = tanh_half_fast(o[j]);
                            if (p.stash && s < nvalid) {   // training: keep (m_it, a_it) for the backward kernel
                                float* st = p.stash + ((size_t)it * 2 * E + ee[j]) * (size_t)p.B + s0 + s;
                                st[0] = mo[j];
                                st[(size_t)E * p.B] = o[j];
                            }
                        }
                }
            } else {
                for (int i = 0; i < n_iter; ++i) {
                    const int e = r + i * R;
                    if (e < E) {
                        const int v = tb.ld(tb.edge_var, e);
                        if constexpr (kNBP) {          // neural_BP.py:244-258: (m W) summed, + prior W_p; m itself stays = m_p
                            const float mw = m_st[(size_t)e * tile + s] * __ldg(wl + e);
                            const float a = node[v * tile + s] - mw + xrow[v] * __ldg(wl + E + e);
                            const float tv = bp_log_abs_tanh_half<false>(a, -46.0517019f);    // < 0 always
                            t_st[(size_t)e * tile + s] = a < 0.f ? -tv : tv;                 // sign flag rides in the sign bit
                            continue;
                        }
                        if constexpr (kV241) {         // decoder_v2_4_1.py:275-276, 283-286: mlp1(sum of (m W) - own) + prior W_p; m itself stays = m_p
                            const float* tw = wsm + 3 * p.wslot;
                            const int ty = tb.csib[e];
                            float ai[1] = {node[v * tile + s] - m_st[(size_t)e * tile + s] * tw[ty]}, oo[1];
                            mlp_softplus<1, false>(W1, hp, ai, ai, oo);
                            t_st[(size_t)e * tile + s] = tanh_half_fast(fmaf(xrow[v], tw[8 + ty], oo[0]));
                            continue;
                        }
                        if constexpr (kV3) {           // decoder_v3_0.py:103-108,229-232,246-247: rnn1(m, mlp1([sum - m, prior]))
                            const float mo = m_st[(size_t)e * tile + s];
                            float ai[1] = {node[v * tile + s] - mo}, ap[1] = {xrow[v]}, oo[1];
                            mlp_relu2<1>(W1, hp, ai, ap, oo);
                            m_st[(size_t)e * tile + s] = gru_cell(gru, mo, oo[0]);
                            continue;
                        }
                        if constexpr (kV122) {         // decoder_v1_2_2.py:120-124,232-233: mlp([sum - m, prior]); m itself stays = m_p
                            float ai[1] = {node[v * tile + s] - m_st[(size_t)e * tile + s]}, ap[1] = {xrow[v]}, oo[1];
                            mlp_tanh2<1>(W1, hp, ai, ap, oo);
                            const float tv = bp_log_abs_tanh_half<false>(oo[0], -46.0517019f);  // < 0 always
                            t_st[(size_t)e * tile + s] = oo[0] < 0.f ? -tv : tv;                 // sign flag rides in the sign bit
                            continue;
                        }
                        if constexpr (kGRU) {          // QGNNNI_ca.py:103-106,197-198,208-209
                            const float mo = m_st[(size_t)e * tile + s];
                            float ai[1] = {node[v * tile + s] - mo + xrow[v]}, oo[1];
                            if constexpr (kNPAD > 0) oo[0] = pwl_eval<kNPAD>(P1, ai[0]);
                            else mlp_relu<1>(W1, hp, ai, oo);
                            m_st[(size_t)e * tile + s] = gru_cell(gru, mo, oo[0]);
                            continue;
                        }
                        const float a = node[v * tile + s] - m_st[(size_t)e * tile + s] + xrow[v];
                        if constexpr (kIsBP) {
                            const float le1 = PROG == GD_PROG_BP_QUANTUM ? -46.0517019f : -16.1180957f;
                            t_st[(size_t)e * tile + s] = bp_log_abs_tanh_half(a, le1);
                            m_st[(size_t)e * tile + s] = a < 0.f ? 1.f : 0.f;  // sign flag (m is dead here)
                        } else {
                            t_st[(size_t)e * tile + s] = tanh_half_fast(a);   // ex2 + rcp, abs. error ~2e-7 (libm tanhf: ~25 instructions)
                        }
                    }
                }
            }
            __syncthreads();
            // ---- C1: per-check sums ----
            if (!cdir) {
            for (int c = r; c < C; c += R) {
                const int b = tb.ld(tb.chk_ptr, c), e_end = tb.ld(tb.chk_ptr, c + 1);
                float acc = 0.f, cnt = 0.f;
                for (int i = b; i < e_end; ++i) {
                    const int e = tb.ld(tb.chk_edges, i);
                    if constexpr (kNBP || kV122) {
                        const float tv = t_st[(size_t)e * tile + s];
                        acc -= fabsf(tv);
                        cnt += tv > 0.f ? 1.f : 0.f;
                    } else if constexpr (kGRU || kV3) {
                        acc += m_st[(size_t)e * tile + s];          // no tanh in this script's check phase
                    } else {
                        acc += t_st[(size_t)e * tile + s];
                        if constexpr (kIsBP) cnt += m_st[(size_t)e * tile + s];
                    }
                }
                node[c * tile + s] = acc;
                if constexpr (kIsBP || kNBP || kV122) node2[c * tile + s] = cnt;
            }
            __syncthreads();
            }
            if constexpr (kV3) {
                // the second read-out (decoder_v3_0.py:267-268, 276): mlp(sum at the check of the messages after the LAST variable phase)
                if (it == p.T - 1 && (p.aux_prob || p.aux_logit)) {
                    for (int c = r; c < C; c += R) {
                        float xi[1] = {node[c * tile + s]}, oo[1];
                        mlp_relu<1>(W3, hp, xi, oo);
                        if (s < nvalid) {
                            const long long row = didx ? (long long)__ldg(didx + s0 + s) : s0 + s;
                            if (p.aux_logit) p.aux_logit[row * C + c] = oo[0];
                            if (p.aux_prob) p.aux_prob[row * C + c] = sigmoid_neg(oo[0]);
                        }
                    }
                }
            }
            // ---- C2: check-phase message, residual ----
            if constexpr (kNBP) {          // neural_BP.py:108-122 (eps2 = 1e-15) and :304 (+ alpha * m_p)
                const float alpha = __ldg(p.weights + (size_t)(2 * p.T + 2) * E);
                for (int i = 0; i < n_iter; ++i) {
                    const int e = r + i * R;
                    if (e < E) {
                        const int c = tb.ld(tb.edge_chk, e);
                        const float tv = t_st[(size_t)e * tile + s];
                        int cnt = (int)(node2[c * tile + s] - (tv > 0.f ? 1.f : 0.f));
                        cnt += xrow[V + c] < 0.f ? 1 : 0;
                        float* mp = m_st + (size_t)e * tile + s;
                        *mp = fmaf(alpha, *mp, bp_check_out(node[c * tile + s] + fabsf(tv), cnt & 1, 1e-15f));
                    }
                }
            } else if constexpr (kV241) {  // decoder_v2_4_1.py:287-288 (mlp(sum - own) * sign) and :337-339 (gated residual)
                const float* tw = wsm + 3 * p.wslot;
                const float ga = tw[32], gb = tw[33];
                for (int i0 = 0; i0 < n_iter; i0 += kEB) {
                    float x0[kEB], o[kEB];
                    int ee[kEB];
#pragma unroll
                    for (int j = 0; j < kEB; ++j) {
                        const int e = r + (i0 + j) * R;
                        ee[j] = e;
                        const int ec = e < E ? e : E - 1;
                        x0[j] = node[tb.ld(tb.edge_chk, ec) * tile + s] - t_st[(size_t)ec * tile + s];
                    }
                    mlp_softplus<kEB, false>(W2, hp, x0, x0, o);
#pragma unroll
                    for (int j = 0; j < kEB; ++j)
                        if (ee[j] < E) {
                            float* mp = m_st + (size_t)ee[j] * tile + s;
                            *mp = fmaf(o[j] * xrow[V + tb.ld(tb.edge_chk, ee[j])], ga, *mp * gb);
                        }
                }
            } else if constexpr (kV122) {  // decoder_v1_2_2.py:105-119 (eps 1e-20 / 1e-12, no input clamp) and :266 (+ m_p)
                for (int i = 0; i < n_iter; ++i) {
                    const int e = r + i * R;
                    if (e < E) {
                        const int c = tb.ld(tb.edge_chk, e);
                        const float tv = t_st[(size_t)e * tile + s];
                        int cnt = (int)(node2[c * tile + s] - (tv > 0.f ? 1.f : 0.f));
                        cnt += xrow[V + c] < 0.f ? 1 : 0;
                        float* mp = m_st + (size_t)e * tile + s;
                        *mp = *mp + bp_check_out(node[c * tile + s] + fabsf(tv), cnt & 1, 1e-12f);
                    }
                }
            } else if constexpr (kV3) {    // decoder_v3_0.py:109-112,229-231,242-243: rnn2(m, mlp2([sum - m, syndrome]))
                for (int i = 0; i < n_iter; ++i) {
                    const int e = r + i * R;
                    if (e < E) {
                        const int c = tb.ld(tb.edge_chk, e);
                        float* mp = m_st + (size_t)e * tile + s;
                        const float mo = *mp;
                        float ai[1] = {node[c * tile + s] - mo}, ap[1] = {xrow[V + c]}, oo[1];
                        mlp_relu2<1>(W2, hp, ai, ap, oo);
                        *mp = gru_cell(gru + 12, mo, oo[0]);
                    }
                }
            } else if constexpr (kGRU) {   // QGNNNI_ca.py:109,197-198,206-207
                for (int i = 0; i < n_iter; ++i) {
                    const int e = r + i * R;
                    if (e < E) {
                        const int c = tb.ld(tb.edge_chk, e);
                        float* mp = m_st + (size_t)e * tile + s;
                        const float mo = *mp;
                        float ai[1] = {(node[c * tile + s] - mo) * xrow[V + c]}, oo[1];
                        if constexpr (kNPAD > 0) oo[0] = pwl_eval<kNPAD>(P2, ai[0]);
                        else mlp_relu<1>(W2, hp, ai, oo);
                        *mp = gru_cell(gru + 12, mo, oo[0]);
                    }
                }
            } else if constexpr (kIsBP) {
                for (int i = 0; i < n_iter; ++i) {
                    const int e = r + i * R;
                    if (e < E) {
                        const int c = tb.ld(tb.edge_chk, e);
                        const float ext = node[c * tile + s] - t_st[(size_t)e * tile + s];
                        int cnt = (int)(node2[c * tile + s] - m_st[(size_t)e * tile + s]);
                        if constexpr (PROG == GD_PROG_BP_QUANTUM) cnt += xrow[V + c] < 0.f ? 1 : 0;
                        const float eps2 = PROG == GD_PROG_BP_QUANTUM ? 1e-12f : 1e-7f;
                        m_st[(size_t)e * tile + s] = bp_check_out(ext, cnt & 1, eps2);
                    }
                }
            } else {
                for (int i0 = 0; i0 < n_iter; i0 += kEB) {
                    float x0[kEB], o[kEB], sg[kEB];
                    int ee[kEB];
#pragma unroll
                    for (int j = 0; j < kEB; ++j) {
                        const int e = r + (i0 + j) * R;
                        ee[j] = e;
                        const int ec = e < E ? e : E - 1;
                        const int c = tb.ld(tb.edge_chk, ec);
                        if (cdir) {
                            float a3 = 0.f;
#pragma unroll
                            for (int q = 0; q < 3; ++q) {
                                const int sb = tb.ld(tb.csib, 3 * ec + q);
                                a3 += sb != 0xFFFF ? t_st[(size_t)sb * tile + s] : 0.f;
                            }
                            x0[j] = a3;
                        } else {
                            x0[j] = node[c * tile + s] - t_st[(size_t)ec * tile + s];
                        }
                        sg[j] = PROG == GD_PROG_CGNNI ? 1.f : xrow[V + c];
                    }
                    if (kSoftplus && use_ctab) {
#pragma unroll
                        for (int j = 0; j < kEB; ++j) o[j] = cubic_tab_eval(ctab, x0[j]);
                    } else if constexpr (kSoftplus && NPOLY >= 0) mlp_softplus_x2<kEB, false, (NPOLY > 0 ? NPOLY : 0)>(W2, hp, x0, x0, o);
                    else if constexpr (kSoftplus) mlp_softplus<kEB, false>(W2, hp, x0, x0, o);
                    else if constexpr (kNPAD > 0) {
#pragma unroll
                        for (int j = 0; j < kEB; ++j) o[j] = pwl_eval<kNPAD>(P2, x0[j]);
                    } else mlp_relu<kEB>(W2, hp, x0, o);
#pragma unroll
                    for (int j = 0; j < kEB; ++j)
                        if (ee[j] < E) {
                            float* mp = m_st + (size_t)ee[j] * tile + s;
                            *mp = o[j] * sg[j] + *mp;
                        }
                }
            }
            __syncthreads();
            if constexpr (kGRU || kV122) {
                if (p.all_iters) emit((long long)it * p.B * V);
            }
        }
        if (!((kGRU || kV122) && p.all_iters)) emit(0);
    }
}

// ---------------------------------------------------------------------------------------------
static int align_up(int x, int a) { return (x + a - 1) / a * a; }

// A (tile, R, EB) candidate of the geometry search with its model score
struct GeomCand {
    int tile, R, eb;
    double score;
};

// force: use exactly this geometry (autotuner / tuned cache); collect: gather every candidate with its score instead
static int plan_decode(const gd_graph* g, const gd_model* m, int64_t B, DecodePlan* out, const GeomCand* force = nullptr,
                       std::vector<GeomCand>* collect = nullptr) {
    GeomCand tuned_hit;
    if (!force && !collect && !g->tuned.empty()) {
        std::lock_guard<std::mutex> lk(const_cast<gd_graph*>(g)->mu);
        for (const auto& tg : g->tuned)
            if (tg.program == m->program && tg.hidden == m->hidden && tg.iters == m->iters && tg.flags == m->flags && tg.B == B) {
                tuned_hit = GeomCand{tg.tile, tg.R, tg.eb, 0.0};
                force = &tuned_hit;
                break;
            }
    }
    const int V = g->V, C = g->C, N = g->N, Cn = g->C;
    const int64_t E64 = g->E;
    // "bp" here = the sum-product family: no MLP slots, a second node array for the sign counts
    const bool bp = m->program == GD_PROG_BP_QUANTUM || m->program == GD_PROG_BP_CLASSICAL || m->program == GD_PROG_NEURAL_BP;
    const int hid = bp ? 0 : m->hidden;
    const int hp = align_up(hid, 8);
    const bool gru = m->program == GD_PROG_GRU_CA || m->program == GD_PROG_V3_0 || m->program == GD_PROG_V2_4_1;   // three MLP slots + 24 (V2_4_1: 34) extra floats
    const bool sp2 = bp || m->program == GD_PROG_V1_2_2;                             // sum-product check phase: a second node array (sign counts)
    const int n_slots = bp ? 0 : ((m->program == GD_PROG_V2_4 || gru) ? 3 : 2);
    const int maxvc = V > C ? V : C;
    DecodeParams& p = out->p;
    memset(&p, 0, sizeof(p));
    out->eb = 4;
    p.B = B; p.T = m->iters; p.V = V; p.C = C; p.E = (int)E64; p.N = N; p.hid = hid; p.hp = hp; p.maxvc = maxvc;
    p.tb = g->t;
    p.all_iters = (m->flags & GD_FLAG_ALL_ITERS) ? 1 : 0;
    p.n_vact = opt_on(OPT_NO_VSKIP) ? (int)g->E : g->n_vact;
    p.vdirect = g->max_var_deg <= 2 ? 1 : 0;
    p.cdirect = g->max_chk_deg <= 4 ? 1 : 0;
    int off = 16;                                  // mbarrier
    // ReLU programs with h < 32: piecewise-linear tables (3 * NPAD floats per MLP) instead of the SoA weight rows
    const bool relu_prog = m->program == GD_PROG_CGNNI || m->program == GD_PROG_QGNNI || m->program == GD_PROG_GRU_CA;   // 1-input ReLU MLPs
    out->npad = (relu_prog && hid < 32) ? (hid < 16 ? 16 : 32) : 0;
    p.wslot = 4 * hp > 3 * out->npad ? 4 * hp : 3 * out->npad;
    p.off_w = off; off += n_slots * p.wslot * 4 + (gru ? 40 * 4 : 0); off = align_up(off, 16);
    if (m->program == GD_PROG_V2_4 && !opt_on(OPT_NO_CTAB)) {
        p.rtab_n = kRtabN;
        p.off_rtab = off;
        off += p.rtab_n * 16;
        p.ctab_n = kCtabN;
        p.ctab_R = (float)(g->max_chk_deg > 1 ? g->max_chk_deg - 1 : 1);
        p.off_ctab = off;
        off += p.ctab_n * 16;
    }
    const bool fits16 = E64 < 65536 && V < 65535 && C < 65535;
    const int tab_bytes = (int)(9 * E64 + V + C + 2) * 2;
    if (p.ctab_n > 0 && !opt_on(OPT_NO_VTAB)) {
        // 12 tables x 512 intervals (96 KB): the reference draws p from a list of 10 (decoder_v2_4.py:187).  Measured on B200,
        // rotated d=5, B=65536, 10 distinct priors: direct 3.43 ms; 4 x 1024 3.68 (6 of 10 priors overflow the slots);
        // 12 x 384 1.21; 10..12 x 512..640 0.81 ms.  With 4 distinct priors 4 x 1024 takes 0.69 ms.
        const int64_t per_syn_est = ((int64_t)N + maxvc + 2 * E64) * 4;
        const int64_t t_without = fits16 ? (g->max_smem_optin - align_up(off + tab_bytes, 128)) / per_syn_est / 8 * 8 : 0;
        // slots: as many (12, 8, 6) as still leave tiles as large as the code gets anyway, up to 16 syndromes (rotated d = 5 / 7
        // and toric L = 5 take 12; rotated d = 11 takes 8, toric L = 11 takes 6).  A tile whose syndromes carry more distinct
        // priors than there are slots takes the direct evaluation as a whole (no mixed warps).
        static const int ks[] = {12, 8, 6};
        for (int ki = 0; ki < 3 && t_without >= 8; ++ki) {
            const int vk = ks[ki];
            const int vbytes = vk * kVtabN * 16 + 16 + 16 * 4 + 128 * 4;
            const int64_t t_with = (g->max_smem_optin - align_up(off + vbytes + tab_bytes, 128)) / per_syn_est / 8 * 8;
            if (t_with >= 8 && t_with >= (t_without < 16 ? t_without : 16)) {
                p.vtab_n = kVtabN; p.vtab_k = vk;
                p.off_vtab = off; off += vk * kVtabN * 16;
                p.off_vmeta = off; off += 16 + 16 * 4 + 128 * 4;
                break;
            }
        }
    }
    // resident layout first
    int tile = 0, resident = 0, R = 0;
    if (fits16 && off + tab_bytes < g->max_smem_optin) {
        const int fixed = align_up(off + tab_bytes, 128);
        const int64_t per_syn = ((int64_t)N + (int64_t)maxvc * (sp2 ? 2 : 1) + 2 * E64) * 4;
        const int64_t tmax = (g->max_smem_optin - fixed) / per_syn;
        if (tmax >= 8) {
            // Pick (tile, R, EB): tile = syndromes per CTA, R = threads per syndrome.  Score =
            //   (fraction of the SMs' tile slots doing useful work over all rounds)
            // x (fraction of the EB-blocked edge slots of a thread that hold a real edge)
            // x w(threads): measured sensitivity of the MUFU-bound inner loop to resident warps
            //   and to the register blocking (profiles/r01_geometry_sweep.txt).
            const int E = (int)E64;
            static const int wx[] = {32, 128, 256, 384, 512, 640, 896, 1024};
            static const double wy[] = {0.20, 0.62, 0.80, 0.90, 0.96, 0.985, 1.0, 1.0};
            double best = -1.0;
            for (int t = 8; t <= tmax && t <= kMaxThreads; t += 8) {
                if (force && force->tile != t) continue;
                if (t < 32 && (32 % t)) continue;
                const int64_t n_t = (B + t - 1) / t;
                const int64_t rounds = (n_t + g->sm_count - 1) / g->sm_count;
                const double eff_round = (double)B / ((double)rounds * (double)g->sm_count * t);
                for (int r = 1; r * t <= kMaxThreads && r <= E; ++r) {
                    if (force && force->R != r) continue;
                    const int thr = r * t;
                    if (thr % 32) continue;
                    double w = wy[7];
                    for (int i = 1; i < 8; ++i)
                        if (thr <= wx[i]) { w = wy[i - 1] + (wy[i] - wy[i - 1]) * (thr - wx[i - 1]) / (wx[i] - wx[i - 1]); break; }
                    const int n_iter = (E + r - 1) / r;
                    // per-thread cost of one iteration in issue slots: EB-blocked per-edge update
                    // (c_edge each) + the node sums this thread owns (c_ld per summed edge)
                    const double c_edge = (m->program == GD_PROG_V2_4 || m->program == GD_PROG_V1_2_2 || m->program == GD_PROG_V2_4_1) ? 16.0 * hp : (bp ? 200.0 : 40.0 + 6.0 * hp);
                    const double c_ld = 4.0;
                    const double node_cost = (double)((V + r - 1) / r) * g->max_var_deg + (double)((Cn + r - 1) / r) * g->max_chk_deg;
                    const double ideal = E * c_edge + 2.0 * E * c_ld;
                    for (int ebk = 4; ebk >= 2; ebk -= 2) {
                        if (force && force->eb != ebk) continue;
                        const int blocks = (n_iter + ebk - 1) / ebk;
                        const double per_thread = (bp ? n_iter : blocks * ebk) * c_edge + node_cost * c_ld;
                        const double eff_bal = ideal / (r * per_thread);
                        const double score = eff_round * eff_bal * w * (ebk == 2 ? (thr >= 384 ? 1.0 : 0.92) : (thr >= 384 ? 0.985 : 1.0));
                        if (collect) collect->push_back(GeomCand{t, r, ebk, score});
                        if (score > best + 1e-9) { best = score; tile = t; R = r; out->eb = ebk; }
                    }
                }
            }
        }
        if (tile) {
            resident = 1;
            p.off_tab = off;
            int o2 = fixed;
            p.off_x = o2; o2 += tile * N * 4; o2 = align_up(o2, 16);
            p.off_node = o2; o2 += maxvc * tile * 4 * (sp2 ? 2 : 1);
            p.off_m = o2; o2 += (int)E64 * tile * 4;
            p.off_t = o2; o2 += (int)E64 * tile * 4;
            out->smem = o2;
            p.scratch_bytes = o2 - p.off_x;
        }
    }
    if (!resident || opt_on(OPT_FORCE_STREAMED)) {
        out->resident = 0;
        return GD_OK;           // caller takes the streamed kernel (gd_streamed.cu)
    }
    p.tile = tile;
    p.R = R;
    out->threads = R * tile;
    p.n_tiles = (int)((B + tile - 1) / tile);
    out->grid = p.n_tiles < g->sm_count ? p.n_tiles : g->sm_count;
    out->resident = resident;
    return GD_OK;
}

template <int PROG>
static int launch_decode(const DecodePlan& pl, cudaStream_t st) {
    void (*k)(const DecodeParams);
    if constexpr (PROG == GD_PROG_V2_4) {
        // NPOLY = 2 of every 4 hidden-unit pairs take the FMA-pipe polynomial lg2.  Measured on B200
        // (profiles/r01_npoly_sweep.txt): 8.70 M syndromes/s against 6.84 M for the scalar MUFU loop.
        if (pl.threads > 512) k = pl.eb == 2 ? decode_kernel<PROG, 1024, 2, 2> : decode_kernel<PROG, 1024, 4, 2>;   // the <= 64-register build
        else k = pl.eb == 2 ? decode_kernel<PROG, 512, 2, 2> : decode_kernel<PROG, 512, 4, 2>;
    } else if constexpr (PROG == GD_PROG_CGNNI || PROG == GD_PROG_QGNNI || PROG == GD_PROG_GRU_CA) {
        if (pl.npad == 16) k = pl.threads > 512 ? decode_kernel<PROG, 1024, 2, 16> : decode_kernel<PROG, 512, 2, 16>;
        else if (pl.npad == 32) k = pl.threads > 512 ? decode_kernel<PROG, 1024, 2, 32> : decode_kernel<PROG, 512, 2, 32>;
        else if (pl.threads > 512) k = pl.eb == 2 ? decode_kernel<PROG, 1024, 2, -1> : decode_kernel<PROG, 1024, 4, -1>;
        else k = pl.eb == 2 ? decode_kernel<PROG, 512, 2, -1> : decode_kernel<PROG, 512, 4, -1>;
    } else {
        if (pl.threads > 512) k = pl.eb == 2 ? decode_kernel<PROG, 1024, 2, -1> : decode_kernel<PROG, 1024, 4, -1>;
        else k = pl.eb == 2 ? decode_kernel<PROG, 512, 2, -1> : decode_kernel<PROG, 512, 4, -1>;
    }
    GD_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, pl.smem));
    if (pl.p.defer_count) {          // deferred pass of the table kernel: overlap its launch with that kernel's tail
        GD_CUDA(gd::pdl_launch(k, dim3(pl.grid), dim3(pl.threads), (size_t)pl.smem, st, pl.p));
    } else {
        k<<<pl.grid, pl.threads, pl.smem, st>>>(pl.p);
        GD_CUDA(cudaGetLastError());
    }
    return GD_OK;
}

int edge_decode(const gd_graph* g, const gd_model* model, DecodePlan pl, const DecodeIO& io, cudaStream_t st,
                const DeferList* dl) {
    pl.p.x = io.x; pl.p.prob = io.prob; pl.p.logit = io.logit; pl.p.hard = io.hard; pl.p.weights = io.weights;
    pl.p.stash = io.stash; pl.p.hard_bits = io.hard_bits;
    pl.p.aux_prob = io.aux_prob; pl.p.aux_logit = io.aux_logit;
    if (dl) { pl.p.defer_count = dl->count; pl.p.defer_idx = dl->idx; }
    switch (model->program) {
        case GD_PROG_CGNNI: return launch_decode<GD_PROG_CGNNI>(pl, st);
        case GD_PROG_QGNNI: return launch_decode<GD_PROG_QGNNI>(pl, st);
        case GD_PROG_V2_4: return launch_decode<GD_PROG_V2_4>(pl, st);
        case GD_PROG_BP_QUANTUM: return launch_decode<GD_PROG_BP_QUANTUM>(pl, st);
        case GD_PROG_NEURAL_BP: return launch_decode<GD_PROG_NEURAL_BP>(pl, st);
        case GD_PROG_GRU_CA: return launch_decode<GD_PROG_GRU_CA>(pl, st);
        case GD_PROG_V3_0: return launch_decode<GD_PROG_V3_0>(pl, st);
        case GD_PROG_V1_2_2: return launch_decode<GD_PROG_V1_2_2>(pl, st);
        case GD_PROG_V2_4_1: return launch_decode<GD_PROG_V2_4_1>(pl, st);
        default: return launch_decode<GD_PROG_BP_CLASSICAL>(pl, st);
    }
}

int route_decode(const gd_graph* gc, const gd_model* m, int64_t B, Use use, Route* r) {
    gd_graph* g = const_cast<gd_graph*>(gc);
    r->lean.clear();
    if (use == Use::Train || use == Use::TrainBwd) {     // (the callers take GD_PROG_V2_4, GD_PROG_CGNNI and GD_PROG_NEURAL_BP)
        if (m->program == GD_PROG_NEURAL_BP) {
            // the TMA-staged streamed forward on every code (its exclusive sums are the accurate arithmetic); its backward
            // (gd_backward_nbp.cu) plans its own layout.  A graph the planner declines is refused, nothing falls back.
            GD_CHECK_ARG(m->hidden == g->E, "%s: GD_PROG_NEURAL_BP needs model.hidden == E (%lld per-edge weights), got %d",
                         use == Use::Train ? "gd_decode_fwd_train" : "gd_decode_bwd", (long long)g->E, m->hidden);
            r->family = Family::StreamedTma;
            if (use == Use::TrainBwd) return GD_OK;
            plan_streamed_tma(g, m, B, &r->tma, true);
            if (!r->tma.ok) {
                set_error("gd_decode_fwd_train: neural BP trains on the streamed kernel, which cannot take this graph: %s",
                          r->tma.why);
                return GD_ERR_UNSUPPORTED;
            }
            return GD_OK;
        }
        if (m->program == GD_PROG_CGNNI) {
            // the node-owner kernel is the only one with a CGNNI backward; that backward plans its own layout
            r->family = Family::Light;
            if (use == Use::TrainBwd) return GD_OK;
            plan_light(g, m, B, &r->light, true);
            if (!r->light.ok) {
                set_error("gd_decode_fwd_train: CGNNI training needs the node-owner kernel: %s", r->light.why);
                return GD_ERR_UNSUPPORTED;
            }
            return GD_OK;
        }
        // decoder_v2_4: where the edge-owner kernel is resident, the table kernel over the whole graph when it plans, and the
        // edge-owner pair in any case -- the header at the end of the stash tells the device which of them runs (gd_lean.cuh).
        // Elsewhere (and under GD_FORCE_STREAMED) the TMA-staged streamed kernel writes the edge-owner stash layout.  The
        // backward plans the table kernel as the forward did; the edge-owner backward has its own planner (gd_backward.cu),
        // which takes its shared-memory or its global-memory variant independently of the forward.
        if (opt_on(OPT_FORCE_STREAMED)) {
            r->family = Family::StreamedTma;
        } else {
            const bool lean = lean_plan(g, m, B, &r->lean, true);
            if (lean || use == Use::Train) {         // the table kernel needs the resident edge-owner kernel (its deferred pass)
                const int rc = plan_decode(g, m, B, &r->edge);
                if (rc != GD_OK) return rc;
                r->family = !r->edge.resident ? Family::StreamedTma : lean ? Family::Lean : Family::EdgeOwner;
            } else {
                r->family = Family::EdgeOwner;
            }
        }
        if (use == Use::Train && r->family == Family::StreamedTma) {
            if (g->E >= 65536) {
                set_error("gd_decode_fwd_train: E=%lld edges; the backward's graph tables hold 16-bit edge ids (E < 65536)",
                          (long long)g->E);
                return GD_ERR_UNSUPPORTED;
            }
            plan_streamed_tma(g, m, B, &r->tma, true);
            if (!r->tma.ok) {
                set_error("gd_decode_fwd_train: the streamed training forward cannot take this graph: %s", r->tma.why);
                return GD_ERR_UNSUPPORTED;
            }
        }
        return GD_OK;
    }
    if (m->program == GD_PROG_V2_4_1) {
        bool all4 = true;
        for (int c = 0; c < g->C && all4; ++c) all4 = g->h_chk_ptr[c + 1] - g->h_chk_ptr[c] == 4;
        GD_CHECK_ARG(all4, "gd_decode_fwd: GD_PROG_V2_4_1 needs every check to have exactly 4 edges (decoder_v2_4_1.py:211-236)");
    }
    GD_CHECK_ARG(m->program != GD_PROG_NEURAL_BP || m->hidden == g->E,
                 "gd_decode_fwd: GD_PROG_NEURAL_BP needs model.hidden == E (%lld per-edge weights), got %d", (long long)g->E,
                 m->hidden);
    // Residency first: a code whose edge state does not fit shared memory (or GD_FORCE_STREAMED) takes a streamed kernel
    // and nothing else.  Every resident route keeps this plan: it is the table kernel's deferred pass.
    const int rc = plan_decode(g, m, B, &r->edge);
    if (rc != GD_OK) return rc;
    if (!r->edge.resident) {
        if (use == Use::Packed) {
            set_error("gd_decode_packed_fwd: this code's edge state does not fit shared memory (streamed path has no packed form)");
            return GD_ERR_UNSUPPORTED;
        }
        if (m->program == GD_PROG_GRU_CA || m->program == GD_PROG_V3_0 || m->program == GD_PROG_V1_2_2 ||
            m->program == GD_PROG_V2_4_1) {
            set_error("gd_decode_fwd: program %d has a resident kernel only and this code's edge state does not fit "
                      "shared memory", m->program);
            return GD_ERR_UNSUPPORTED;
        }
        plan_streamed_tma(g, m, B, &r->tma);
        if (r->tma.ok) {
            r->family = Family::StreamedTma;
            return GD_OK;
        }
        if (m->program == GD_PROG_NEURAL_BP) {       // the register-batched kernel (gd_streamed.cu) has no neural BP program
            set_error("gd_decode_fwd: neural BP on a code whose edge state does not fit shared memory needs the TMA-staged "
                      "streamed kernel, which cannot take this graph: %s", r->tma.why);
            return GD_ERR_UNSUPPORTED;
        }
        r->family = Family::Streamed;
        return plan_streamed(g, m, B, &r->streamed);
    }
    if (lean_plan(g, m, B, &r->lean)) {
        r->family = Family::Lean;                        // decoder_v2_4 on surface / toric codes
        return GD_OK;
    }
    plan_light(g, m, B, &r->light);                      // the light programs, when the batch fills the GPU
    r->family = r->light.ok ? Family::Light : Family::EdgeOwner;
    return GD_OK;
}

gd_launch_info route_launch_info(const Route& r) {
    gd_launch_info li;
    memset(&li, 0, sizeof(li));
    li.resident = 1;
    switch (r.family) {
        case Family::Lean: {
            const LeanPlan& pl = r.lean[0];              // (parts: the first launch's geometry; tiles of all launches)
            li.tile = 32 * pl.p.G; li.threads = pl.threads; li.grid = pl.grid; li.smem_bytes = pl.smem;
            li.n_tiles = (int)r.lean.size() * ((pl.n_tiles + pl.p.G - 1) / pl.p.G);
        } break;
        case Family::Light:
            li.tile = r.light.p.tile; li.threads = r.light.threads; li.grid = r.light.grid; li.smem_bytes = r.light.smem;
            li.n_tiles = r.light.p.n_tiles;
            break;
        case Family::EdgeOwner:
            li.tile = r.edge.p.tile; li.threads = r.edge.threads; li.grid = r.edge.grid; li.smem_bytes = r.edge.smem;
            li.n_tiles = r.edge.p.n_tiles;
            break;
        case Family::StreamedTma:
            li.tile = r.tma.p.tile; li.threads = r.tma.threads; li.grid = r.tma.grid; li.smem_bytes = r.tma.smem;
            li.resident = 0; li.n_tiles = r.tma.p.n_tiles;
            break;
        case Family::Streamed:
            li.tile = r.streamed.p.tile; li.threads = r.streamed.threads; li.grid = r.streamed.grid;
            li.smem_bytes = r.streamed.smem; li.resident = 0; li.n_tiles = r.streamed.p.n_tiles;
            break;
    }
    return li;
}

namespace {
struct PackedRun {
    const gd_graph* g; const gd_model* model; const DecodePlan* plan; const DecodeIO* io; cudaStream_t st;
};
int packed_run(void* ctx, const float* x_dev) {
    const PackedRun* r = static_cast<const PackedRun*>(ctx);
    DecodeIO io = *r->io;
    io.x = x_dev;
    return edge_decode(r->g, r->model, *r->plan, io, r->st);
}
}  // namespace

int decode_routed(gd_graph* g, const gd_model* model, const Route& r, const DecodeIO& io, int64_t B, cudaStream_t st) {
    switch (r.family) {
        case Family::Lean: {
            bool no_resources = false;
            const int rc = lean_decode(g, model, r.lean, r.edge, io, B, st, &no_resources);
            if (!no_resources) return rc;
            // The one decline only a launch can discover: the table kernel got no memory pool or table set on this device.
            // The edge-owner kernel decodes the whole batch instead.
            break;
        }
        case Family::Light: return light_decode(r.light, model, io, st);
        case Family::StreamedTma: return streamed_tma_decode(g, r.tma, model, io, st);
        case Family::Streamed: return streamed_decode(g, r.streamed, model, io, st);
        case Family::EdgeOwner: break;
    }
    if (!io.x) {             // packed inputs: expand them for the edge-owner kernel
        PackedRun run{g, model, &r.edge, &io, st};
        return packed_via_unpack(g, io.prior, io.synd, B, st, packed_run, &run);
    }
    return edge_decode(g, model, r.edge, io, st);
}

}  // namespace gd

extern "C" int gd_decode_launch_info(const gd_graph* g, const gd_model* model, int64_t B, gd_launch_info* out) {
    GD_CHECK_ARG(g && out, "gd_decode_launch_info: NULL argument");
    GD_CHECK_ARG(gd_model_valid(model), "gd_decode_launch_info: invalid model");
    GD_CHECK_ARG(B > 0, "gd_decode_launch_info: B must be positive");
    gd::DeviceGuard dg(g->device);
    GD_CUDA(dg.status());
    gd::Route r;
    const int rc = gd::route_decode(g, model, B, gd::Use::Infer, &r);
    if (rc != GD_OK) return rc;
    *out = gd::route_launch_info(r);
    return GD_OK;
}

extern "C" int gd_decode_tables_info(const gd_graph* g, const gd_model* model, int64_t B, int32_t* out4) {
    GD_CHECK_ARG(g && out4, "gd_decode_tables_info: NULL argument");
    GD_CHECK_ARG(gd_model_valid(model) && B > 0, "gd_decode_tables_info: invalid model / B");
    out4[0] = out4[1] = out4[2] = out4[3] = 0;
    gd::DeviceGuard dg(g->device);
    GD_CUDA(dg.status());
    gd::Route r;
    const int rc = gd::route_decode(g, model, B, gd::Use::Infer, &r);
    if (rc != GD_OK) return rc;
    if (r.family != gd::Family::Lean && r.family != gd::Family::EdgeOwner) return GD_OK;
    const gd::DecodeParams& p = r.edge.p;        // the edge-owner kernel's tables (the table kernel's deferred pass)
    out4[0] = p.ctab_n; out4[1] = p.rtab_n; out4[2] = p.vtab_n; out4[3] = p.vtab_k;
    return GD_OK;
}

// Argument checks, then the route and its launch on the graph's device.
static int decode_fwd_impl(const gd_graph* gc, const gd_model* model, const gd::DecodeIO& io, int64_t B, void* stream,
                           gd::Use use = gd::Use::Infer) {
    gd_graph* g = const_cast<gd_graph*>(gc);
    GD_CHECK_ARG(g != nullptr, "gd_decode_fwd: graph is NULL");
    GD_CHECK_ARG(gd_model_valid(model), "gd_decode_fwd: invalid model (program=%d hidden=%d iters=%d)",
                 model ? model->program : -1, model ? model->hidden : -1, model ? model->iters : -1);
    GD_CHECK_ARG(B >= 0 && B < ((int64_t)1 << 31), "gd_decode_fwd: B=%lld out of range", (long long)B);
    if (B == 0) return GD_OK;  // empty batch: nothing to do (the reference would crash; we return cleanly)
    GD_CHECK_ARG(io.x != nullptr, "gd_decode_fwd: x is NULL");
    GD_CHECK_ARG(gd_weights_size(model) == 0 || io.weights != nullptr, "gd_decode_fwd: weights is NULL");
    GD_CHECK_ARG(((uintptr_t)io.x & 15) == 0, "gd_decode_fwd: x must be 16-byte aligned");
    GD_CHECK_ARG(((uintptr_t)io.prob & 15) == 0 && ((uintptr_t)io.logit & 15) == 0 && ((uintptr_t)io.hard & 3) == 0,
                 "gd_decode_fwd: outputs must be 16-byte (prob, logit) / 4-byte (hard) aligned");
    gd::DeviceGuard dg(g->device);
    GD_CUDA(dg.status());
    gd::Route r;
    const int rc = gd::route_decode(g, model, B, use, &r);
    if (rc != GD_OK) return rc;
    return gd::decode_routed(g, model, r, io, B, (cudaStream_t)stream);
}

extern "C" int gd_decode_fwd(const gd_graph* gc, const gd_model* model, const float* weights_dev,
                             const float* x_dev, float* prob_dev, float* logit_dev, uint8_t* hard_dev, int64_t B,
                             void* stream) {
    gd::DecodeIO io{};
    io.weights = weights_dev; io.x = x_dev; io.prob = prob_dev; io.logit = logit_dev; io.hard = hard_dev;
    return decode_fwd_impl(gc, model, io, B, stream);
}

extern "C" int gd_decode_fwd_aux(const gd_graph* gc, const gd_model* model, const float* weights_dev, const float* x_dev,
                                 float* prob_dev, float* logit_dev, uint8_t* hard_dev, float* aux_prob_dev, float* aux_logit_dev,
                                 int64_t B, void* stream) {
    if ((aux_prob_dev || aux_logit_dev) && (!model || model->program != GD_PROG_V3_0)) {
        gd::set_error("gd_decode_fwd_aux: program %d has no second read-out (GD_PROG_V3_0 only)", model ? model->program : -1);
        return GD_ERR_UNSUPPORTED;
    }
    gd::DecodeIO io{};
    io.weights = weights_dev; io.x = x_dev; io.prob = prob_dev; io.logit = logit_dev; io.hard = hard_dev;
    io.aux_prob = aux_prob_dev; io.aux_logit = aux_logit_dev;
    return decode_fwd_impl(gc, model, io, B, stream);
}

// ---- packed form of the same decode (include/gnn_decode.h): what the reference's x actually carries per syndrome is ONE
// prior value and C check signs (gen_syn, quantum/error_generate.py:258, 270-276) ----
extern "C" int gd_decode_packed_fwd(const gd_graph* gc, const gd_model* model, const float* weights_dev, const float* prior_dev,
                                    const uint32_t* synd_dev, float* prob_dev, uint32_t* hard_bits_dev, int64_t B, void* stream) {
    gd_graph* g = const_cast<gd_graph*>(gc);
    GD_CHECK_ARG(g != nullptr, "gd_decode_packed_fwd: graph is NULL");
    GD_CHECK_ARG(gd_model_valid(model), "gd_decode_packed_fwd: invalid model");
    GD_CHECK_ARG(B >= 0 && B < ((int64_t)1 << 31), "gd_decode_packed_fwd: B=%lld out of range", (long long)B);
    if (B == 0) return GD_OK;
    GD_CHECK_ARG(prior_dev && synd_dev, "gd_decode_packed_fwd: prior / syndrome bits are NULL");
    GD_CHECK_ARG(prob_dev || hard_bits_dev, "gd_decode_packed_fwd: no output requested");
    GD_CHECK_ARG(gd_weights_size(model) == 0 || weights_dev != nullptr, "gd_decode_packed_fwd: weights is NULL");
    GD_CHECK_ARG(((uintptr_t)prob_dev & 15) == 0 && ((uintptr_t)hard_bits_dev & 3) == 0 && ((uintptr_t)synd_dev & 3) == 0,
                 "gd_decode_packed_fwd: prob must be 16-byte, bit arrays 4-byte aligned");
    if (model->program != GD_PROG_V2_4) {
        gd::set_error("gd_decode_packed_fwd: packed inputs are implemented for GD_PROG_V2_4 only");
        return GD_ERR_UNSUPPORTED;
    }
    gd::DeviceGuard dg(g->device);
    GD_CUDA(dg.status());
    gd::Route r;
    const int rc = gd::route_decode(g, model, B, gd::Use::Packed, &r);
    if (rc != GD_OK) return rc;
    gd::DecodeIO io{};
    io.weights = weights_dev; io.prior = prior_dev; io.synd = synd_dev; io.prob = prob_dev; io.hard_bits = hard_bits_dev;
    return gd::decode_routed(g, model, r, io, B, (cudaStream_t)stream);
}

extern "C" int64_t gd_stash_floats(const gd_graph* g, const gd_model* model, int64_t B) {
    if (!g || !gd_model_valid(model) || B < 0) {
        gd::set_error("gd_stash_floats: invalid argument");
        return -1;
    }
    // m after every iteration (gd_light.cuh; neural BP: the streamed forward, gd_streamed_tma.cu)
    if (model->program == GD_PROG_CGNNI || model->program == GD_PROG_NEURAL_BP) return (int64_t)model->iters * g->E * B;
    return (int64_t)(model->iters + 1) * 2 * g->E * B + gd::kLeanTrainTailFloats + B;   // + the header and sorted list of gd_lean.cuh
}

extern "C" int gd_decode_fwd_train(const gd_graph* gc, const gd_model* model, const float* weights_dev,
                                   const float* x_dev, float* prob_dev, float* logit_dev, float* stash_dev, int64_t B,
                                   void* stream) {
    GD_CHECK_ARG(model && (model->program == GD_PROG_V2_4 || model->program == GD_PROG_CGNNI || model->program == GD_PROG_NEURAL_BP),
                 "gd_decode_fwd_train: only GD_PROG_V2_4, GD_PROG_CGNNI and GD_PROG_NEURAL_BP have a backward kernel");
    GD_CHECK_ARG(stash_dev != nullptr || B == 0, "gd_decode_fwd_train: stash is NULL");
    gd::DecodeIO io{};
    io.weights = weights_dev; io.x = x_dev; io.prob = prob_dev; io.logit = logit_dev; io.stash = stash_dev;
    return decode_fwd_impl(gc, model, io, B, stream, gd::Use::Train);
}

// ---- geometry autotuner: measure, don't guess ------------------------------------------------------------------------
// The (tile, R, EB) model above ranks hundreds of geometries; its top picks are usually within a few percent of each
// other and occasionally mis-ordered (rotated d = 11: the model's pick is 15 % slower than its 4th candidate).  This
// entry point times the best few candidates on the caller's own batch and remembers the winner per
// (graph, model, B); gd_decode_fwd then uses it.  One-time cost: ~2 launches per candidate.
extern "C" int gd_decode_autotune(const gd_graph* gc, const gd_model* model, const float* weights_dev, const float* x_dev,
                                  int64_t B, int32_t max_candidates, void* stream, gd_launch_info* chosen) {
    gd_graph* g = const_cast<gd_graph*>(gc);
    GD_CHECK_ARG(g != nullptr && gd_model_valid(model) && x_dev != nullptr && B > 0, "gd_decode_autotune: bad argument");
    GD_CHECK_ARG(gd_weights_size(model) == 0 || weights_dev != nullptr, "gd_decode_autotune: weights is NULL");
    cudaStream_t st = (cudaStream_t)stream;
    gd::DeviceGuard dg(g->device);
    GD_CUDA(dg.status());
    gd::Route r;
    int rc = gd::route_decode(g, model, B, gd::Use::Infer, &r);
    if (rc != GD_OK) return rc;
    if (chosen) *chosen = gd::route_launch_info(r);
    // only the edge-owner resident kernel has a geometry to tune; the other families plan themselves
    if (r.family != gd::Family::EdgeOwner) return GD_OK;
    std::vector<gd::GeomCand> cands;
    gd::DecodePlan pl;
    rc = gd::plan_decode(g, model, B, &pl, nullptr, &cands);
    if (rc != GD_OK || cands.empty()) return rc;
    std::sort(cands.begin(), cands.end(), [](const gd::GeomCand& a, const gd::GeomCand& b) { return a.score > b.score; });
    // keep the best-scored candidate of each distinct (tile, R), EB = 2 and 4 compete inside it
    std::vector<gd::GeomCand> pick;
    const int K = max_candidates > 0 ? max_candidates : 24;
    for (const auto& c : cands) {
        bool dup = false;
        for (const auto& q : pick) dup = dup || (q.tile == c.tile && q.R == c.R && q.eb == c.eb);
        if (!dup) pick.push_back(c);
        if ((int)pick.size() >= K) break;
    }
    gd::DeviceBuffer<float> prob;
    gd::Event e0, e1;
    cudaError_t e = gd::device_alloc(prob, (size_t)B * g->V * sizeof(float));
    if (e == cudaSuccess) e = gd::create(e0, cudaEventCreateWithFlags, cudaEventDefault);
    if (e == cudaSuccess) e = gd::create(e1, cudaEventCreateWithFlags, cudaEventDefault);
    gd::GeomCand best{0, 0, 0, 0.0};
    float best_ms = 1e30f;
    for (size_t i = 0; i < pick.size() && e == cudaSuccess && rc == GD_OK; ++i) {
        {
            std::lock_guard<std::mutex> lk(g->mu);
            for (size_t q = 0; q < g->tuned.size(); ++q)       // drop a previous entry for this key
                if (g->tuned[q].program == model->program && g->tuned[q].hidden == model->hidden &&
                    g->tuned[q].iters == model->iters && g->tuned[q].flags == model->flags && g->tuned[q].B == B) {
                    g->tuned.erase(g->tuned.begin() + q);
                    break;
                }
            g->tuned.push_back(gd_graph::TunedGeom{model->program, model->hidden, model->iters, model->flags, B, pick[i].tile,
                                                   pick[i].R, pick[i].eb});
        }
        float ms = 1e30f;
        for (int rep = 0; rep < 3 && rc == GD_OK && e == cudaSuccess; ++rep) {       // first launch warms up
            cudaEventRecord(e0.get(), st);
            rc = gd_decode_fwd(g, model, weights_dev, x_dev, prob.get(), nullptr, nullptr, B, st);
            cudaEventRecord(e1.get(), st);
            e = cudaEventSynchronize(e1.get());
            float t = 0.f;
            if (e == cudaSuccess) cudaEventElapsedTime(&t, e0.get(), e1.get());
            if (rep > 0 && t < ms) ms = t;
        }
        if (ms < best_ms) { best_ms = ms; best = pick[i]; }
    }
    if (best.tile) {
        std::lock_guard<std::mutex> lk(g->mu);
        for (size_t q = 0; q < g->tuned.size(); ++q)
            if (g->tuned[q].program == model->program && g->tuned[q].hidden == model->hidden && g->tuned[q].iters == model->iters &&
                g->tuned[q].flags == model->flags && g->tuned[q].B == B) {
                g->tuned[q].tile = best.tile; g->tuned[q].R = best.R; g->tuned[q].eb = best.eb;
            }
    }
    if (rc != GD_OK) return rc;
    GD_CUDA(e);
    if (chosen) gd_decode_launch_info(g, model, B, chosen);
    return GD_OK;
}
