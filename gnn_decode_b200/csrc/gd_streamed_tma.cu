// Streamed decoder, TMA-staged (the default path for codes whose edge state does not fit shared
// memory -- BASELINE config 5: hypergraph-product [[1600,64]], V = 3200, C = 1536, E = 10752).
// Same arithmetic as gd_decode.cu (reference GNNI.forward: quantum/decoder_v2_4.py:272-294,
// quantum/QGNNI.py:228-252, quantum/BP.py:199-219, classical/CGNNI.py:259-284,
// classical/BP.py:239-259); what differs is the data movement, which is what bounds this path:
//
//   * each persistent CTA owns a slab in HBM   xT[N][tile] | m[E][tile] | t[E][tile] | lg[V][tile]
//     (batch-minor: one message of `tile` syndromes is one contiguous ROW of tile*4 bytes);
//   * a lane owns FOUR syndromes (one float4 of every row), a warp owns whole nodes:
//       variable phase: a warp takes a chunk of consecutive variables; in the canonical edge order
//         (H.to_sparse(): sorted by variable) their messages are ONE contiguous block of rows
//         -> one bulk async copy (TMA, cp.async.bulk) for the messages + one for the priors;
//       check phase:    a warp takes one check; lane k issues the bulk copy of the k-th sibling
//         row of t (and of m, for the residual) -> a gather of full rows, no sector waste;
//   * every warp runs its own 2-stage mbarrier pipeline in shared memory: the rows of the NEXT
//     node are in flight while the lanes evaluate the current one from shared memory, so HBM
//     latency is decoupled from the arithmetic (the register-batched kernel in gd_streamed.cu
//     alternates load bursts with compute and stalls 45% of its cycles on long_scoreboard);
//   * results leave as 128-bit coalesced stores straight from registers; no node-sum arrays, two
//     CTA barriers per iteration;
//   * HBM traffic per edge and iteration (fp32): learned programs 20 B (m: R,R,W; t: W,R),
//     sum-product 16 B -- log|tanh| <= 0 always, so the sign flag the check phase needs rides in
//     the sign bit of the stored value instead of a second array.
#include "gd_common.cuh"
#include "gd_math.cuh"
#include "gd_options.cuh"
#include "gd_decode.cuh"
#include "gd_nodemath.cuh"
#include <stdlib.h>
#include <string.h>

namespace gd {

namespace tma {
__device__ __forceinline__ uint32_t s32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void bar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(s32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_bar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
// generic-proxy accesses before, async-proxy (bulk copy) accesses after: shared and global
__device__ __forceinline__ void fence_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(s32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(s32(dst)),
                 "l"(src), "r"(bytes), "r"(s32(bar))
                 : "memory");
}
__device__ __forceinline__ void wait(uint64_t* bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n.reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n}\n"
            : "=r"(done)
            : "r"(s32(bar)), "r"(parity)
            : "memory");
    } while (!done);
}
}  // namespace tma

// STASH: decoder_v2_4's training forward -- also writes (m_it, a_it) of every edge and iteration and the final m into
// p.stash, in the edge-owner kernel's layout [(T+1)][2][E][B], so either backward kernel (gd_backward.cu) can take it.
template <int PROG, int NPAD, bool STASH = false>
__global__ void __launch_bounds__(512, 1) decode_streamed_tma_kernel(const StreamTmaParams p) {
    static_assert(!STASH || PROG == GD_PROG_V2_4, "the training stash exists for decoder_v2_4 only");
    extern __shared__ __align__(128) unsigned char smem[];
    using NM = NodeMath<PROG, NPAD>;
    constexpr bool kIsBP = NM::kIsBP;
    constexpr bool kSoftplus = NM::kSoftplus;
    constexpr bool kSign = NM::kSign;
    constexpr bool kClamp = (PROG == GD_PROG_CGNNI || PROG == GD_PROG_BP_CLASSICAL);

    const int tile = p.tile, E = p.E, V = p.V, C = p.C, N = p.N, W = p.W;
    const int tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31, w = tid >> 5;
    const uint32_t row_bytes = (uint32_t)tile * 4u;
    const int stage_floats = p.stage_rows * tile;
    float* const scratch = reinterpret_cast<float*>(smem + p.off_stage);     // all stages, as one array
    const int S = p.S;
    const int scratch_floats = W * S * stage_floats;
    float* const stg0 = scratch + (w * S) * stage_floats;
    uint64_t* const bar0 = reinterpret_cast<uint64_t*>(smem) + w * 4;
    uint32_t parbits = 0;                 // bit s = phase parity of this warp's stage s
    const bool active = lane < p.lanes;
    const int l4 = active ? lane * 4 : 0;
    const GraphTables tb = p.tb;

    float* const xT = p.slab + (size_t)blockIdx.x * p.slab_floats;
    float* const m_st = xT + (size_t)N * tile;
    float* const t_st = m_st + (size_t)E * tile;
    float* const lg_st = t_st + (size_t)E * tile;

    NM nm{};
    nm.hp = p.hp;
    if constexpr (!kIsBP) {
        float* wsm = reinterpret_cast<float*>(smem + p.off_w);
        const float* wt = p.weights;
        const int h = p.hid, hp = p.hp;
        const float s1 = kSoftplus ? kLog2e : 1.f, s2 = kSoftplus ? kLn2 : 1.f;
        float* slot = wsm;
        if constexpr (PROG == GD_PROG_V2_4) {
            stage_mlp_t(slot, hp, h, wt, 2, true, wt + 2 * h, wt + 3 * h, s1, s2, tid, nthr);
            nm.W1 = MlpSmem{slot, slot + hp, slot + 2 * hp, slot + 3 * hp, wt[4 * h]};
            wt += 4 * h + 1;
            slot += 4 * hp;
        }
        if constexpr (NPAD > 0) {   // 1 -> h -> 1 ReLU MLPs as piecewise-linear tables (gd_math.cuh)
            float* t2 = slot;
            float* t3 = slot + pwl_smem_floats(NPAD);
            if (w == 0) pwl_build(t2, reinterpret_cast<float2*>(t2 + NPAD), NPAD, wt, wt + h, wt + 2 * h, wt[3 * h], h, lane);
            if (w == 1 || (W == 1 && w == 0)) {
                const float* w3 = wt + 3 * h + 1;
                pwl_build(t3, reinterpret_cast<float2*>(t3 + NPAD), NPAD, w3, w3 + h, w3 + 2 * h, w3[3 * h], h, lane);
            }
            nm.P2 = PwlSmem{t2, reinterpret_cast<const float2*>(t2 + NPAD)};
            nm.P3 = PwlSmem{t3, reinterpret_cast<const float2*>(t3 + NPAD)};
        } else {
            stage_mlp_t(slot, hp, h, wt, 1, false, wt + h, wt + 2 * h, s1, s2, tid, nthr);
            nm.W2 = MlpSmem{slot, slot + hp, slot + 2 * hp, slot + 3 * hp, wt[3 * h]};
            wt += 3 * h + 1;
            slot += 4 * hp;
            stage_mlp_t(slot, hp, h, wt, 1, false, wt + h, wt + 2 * h, s1, s2, tid, nthr);
            nm.W3 = MlpSmem{slot, slot + hp, slot + 2 * hp, slot + 3 * hp, wt[3 * h]};
        }
    }
    if (lane == 0) {
        for (int q = 0; q < S; ++q) tma::bar_init(bar0 + q, 1);
        tma::fence_bar_init();
    }
    __syncthreads();
    nm.use_ctab = nm.use_rtab = false;
    nm.rtab_R = 0.f;
    if constexpr (PROG == GD_PROG_V2_4) {
        // the same tables, bounds and decisions as the resident kernel (gd_decode.cu): check phase on |ext| <= max check degree - 1,
        // read-out on |m| <= T max|mlp2|; the stage area is idle here and serves as scratch
        if (p.ctab_n > 0 && p.ctab_n + 8 <= scratch_floats) {
            const float step = 2.0f * p.ctab_R / (float)p.ctab_n;
            nm.use_ctab = cubic_tab_bound(p.weights + 4 * p.hid + 1, p.hid, step) <= 1e-7f;
            if (nm.use_ctab) {
                float4* dst = reinterpret_cast<float4*>(smem + p.off_ctab);
                const float fm = cubic_tab_build(nm.W2, nm.hp, p.ctab_R, p.ctab_n, dst, scratch, tid, nthr);
                nm.ctab = CubicTab{dst, 1.0f / step, p.ctab_R / step, (float)p.ctab_n - 0.001f};
                if (p.rtab_n > 0 && p.T > 0 && p.rtab_n + 8 <= scratch_floats) {
                    __shared__ unsigned int fmax_bits;
                    if (tid == 0) fmax_bits = 0u;
                    __syncthreads();
                    atomicMax(&fmax_bits, __float_as_uint(fm));           // non-negative floats order like uints
                    __syncthreads();
                    nm.rtab_R = (float)p.T * (__uint_as_float(fmax_bits) * 1.02f + 1e-6f);
                    const float rstep = 2.0f * nm.rtab_R / (float)p.rtab_n;
                    nm.use_rtab = cubic_tab_bound(p.weights + 7 * p.hid + 2, p.hid, rstep) <= 4e-6f;
                    if (nm.use_rtab) {
                        float4* rdst = reinterpret_cast<float4*>(smem + p.off_rtab);
                        cubic_tab_build(nm.W3, nm.hp, nm.rtab_R, p.rtab_n, rdst, scratch, tid, nthr);
                        nm.rtab = CubicTab{rdst, 1.0f / rstep, nm.rtab_R / rstep, (float)p.rtab_n - 0.001f};
                    }
                }
            }
            __syncthreads();                                              // tables complete; the scratch is free again
        }
    }

    const int K = p.vchunk, n_vchunks = (V + K - 1) / K;

    // ---- per-warp pipeline pieces ----
    // variable-phase item ci: variables [ci*K, ci*K+K): message rows var_ptr[v0]..var_ptr[v1] (contiguous) + prior rows
    auto issue_var = [&](int ci, int sidx, bool with_m) {
        if (lane == 0) {
            const int v0 = ci * K, v1 = min(V, v0 + K);
            const int e0 = __ldg(tb.var_ptr + v0), e1 = __ldg(tb.var_ptr + v1);
            float* dst = stg0 + sidx * stage_floats;
            const uint32_t bm = with_m ? (uint32_t)(e1 - e0) * row_bytes : 0u, bp = (uint32_t)(v1 - v0) * row_bytes;
            tma::fence_async_smem();
            tma::expect_tx(bar0 + sidx, bm + bp);
            if (bm) tma::g2s(dst, m_st + (size_t)e0 * tile, bm, bar0 + sidx);
            tma::g2s(dst + p.vrows * tile, xT + (size_t)v0 * tile, bp, bar0 + sidx);
        }
    };
    // check-phase item c: row k of the stage = t of the k-th edge of c, row d+k = m of that edge, last row = syndrome sign
    auto issue_chk = [&](int c, int sidx, bool with_m) {
        const int b = __ldg(tb.chk_ptr + c), d = __ldg(tb.chk_ptr + c + 1) - b;
        float* dst = stg0 + sidx * stage_floats;
        if (lane == 0) {
            tma::fence_async_smem();
            tma::expect_tx(bar0 + sidx, (uint32_t)(d * (with_m ? 2 : 1) + (kSign ? 1 : 0)) * row_bytes);
        }
        __syncwarp();
        for (int k = lane; k < d; k += 32) {
            const size_t e = (size_t)__ldg(tb.chk_edges + b + k);
            tma::g2s(dst + k * tile, t_st + e * tile, row_bytes, bar0 + sidx);
            if (with_m) tma::g2s(dst + (d + k) * tile, m_st + e * tile, row_bytes, bar0 + sidx);
        }
        if (kSign && lane == 0)
            tma::g2s(dst + (with_m ? 2 * d : d) * tile, xT + (size_t)(V + c) * tile, row_bytes, bar0 + sidx);
    };
    auto wait_stage = [&](int sidx) {
        tma::wait(bar0 + sidx, (parbits >> sidx) & 1u);
        parbits ^= 1u << sidx;
    };
    // training: this lane's float4 of stash row `row` (syndromes s0 + l4 ..); past s0 + nvalid the row runs into the next one
    const bool stash_vec = STASH && (p.B & 3) == 0 && ((uintptr_t)p.stash & 15) == 0;
    auto stash4 = [&](size_t row, long long s0, int nvalid, const float (&v)[4]) {
        float* d = p.stash + row * (size_t)p.B + s0 + l4;
        if (stash_vec) {
            if (l4 < nvalid) __stcg(reinterpret_cast<float4*>(d), make_float4(v[0], v[1], v[2], v[3]));
        } else {
            for (int j = 0; j < 4 && l4 + j < nvalid; ++j) __stcg(d + j, v[j]);
        }
    };

    for (int tix = blockIdx.x; tix < p.n_tiles; tix += gridDim.x) {
        const long long s0 = (long long)tix * tile;
        const int nvalid = (int)min((long long)tile, p.B - s0);
        // ---- x[tile][N] -> xT[N][tile]: transposed through shared memory, both sides coalesced ----
        {
            const int pitch = tile | 1;
            const int NC = scratch_floats / pitch;
            const float* xg = p.x + s0 * N;
            for (int n0 = 0; n0 < N; n0 += NC) {
                const int nc = min(NC, N - n0);
                for (int i = tid; i < tile * nc; i += nthr) {
                    const int si = i / nc, j = i - si * nc;
                    scratch[j * pitch + si] = si < nvalid ? __ldg(xg + (size_t)si * N + n0 + j) : 0.f;
                }
                __syncthreads();
                for (int i = tid; i < nc * tile; i += nthr) {
                    const int j = i / tile, si = i - j * tile;
                    xT[(size_t)(n0 + j) * tile + si] = scratch[j * pitch + si];
                }
                __syncthreads();
            }
        }
        tma::fence_async_all();
        __syncthreads();

        for (int it = 0; it <= p.T; ++it) {
            const bool with_m = it > 0;           // m == 0 before the first iteration: nothing to fetch
            const bool readout = it == p.T;       // the read-out is one more variable-owner pass over m
            // ---- variable phase (or read-out) ----
            {
                int ci = w, sidx = 0;
                for (int q = 0; q < S - 1; ++q)                       // prologue: S - 1 items in flight
                    if (ci + q * W < n_vchunks) issue_var(ci + q * W, q, with_m);
                for (; ci < n_vchunks; ci += W, sidx = sidx + 1 == S ? 0 : sidx + 1) {
                    if (ci + (S - 1) * W < n_vchunks) issue_var(ci + (S - 1) * W, sidx == 0 ? S - 1 : sidx - 1, with_m);
                    wait_stage(sidx);
                    const float* st = stg0 + sidx * stage_floats + l4;
                    const int v0 = ci * K, v1 = min(V, v0 + K);
                    const int e0 = __ldg(tb.var_ptr + v0);
                    if (active) {
                        int b = e0;
                        for (int v = v0; v < v1; ++v) {
                            const int b_next = __ldg(tb.var_ptr + v + 1), d = b_next - b;
                            const float4 pr = lds4(st + (p.vrows + v - v0) * tile);
                            const float* rows = st + (b - e0) * tile;
                            if (readout) {
                                float acc[4] = {0.f, 0.f, 0.f, 0.f};
                                if (with_m) {
                                    for (int k = 0; k < d; ++k) {
                                        const float4 mv = lds4(rows + k * tile);
                                        if constexpr (PROG == GD_PROG_V2_4) {     // per-EDGE read-out MLP, then the sum
                                            float xi[4] = {mv.x, mv.y, mv.z, mv.w}, oo[4];
                                            if constexpr (STASH) stash4((size_t)p.T * 2 * E + b + k, s0, nvalid, xi);   // m_T
                                            nm.readout_edge(xi, oo);
#pragma unroll
                                            for (int j = 0; j < 4; ++j) acc[j] += oo[j];
                                        } else {
                                            acc[0] += mv.x; acc[1] += mv.y; acc[2] += mv.z; acc[3] += mv.w;
                                        }
                                    }
                                } else if constexpr (PROG == GD_PROG_V2_4) {      // T == 0: mlp(0) per edge
                                    float xi[4] = {0.f, 0.f, 0.f, 0.f}, oo[4];
                                    mlp_softplus_x2<4, false, 2>(nm.W3, nm.hp, xi, xi, oo);
                                    for (int k = 0; k < d; ++k) {
                                        if constexpr (STASH) stash4((size_t)b + k, s0, nvalid, xi);
#pragma unroll
                                        for (int j = 0; j < 4; ++j) acc[j] += oo[j];
                                    }
                                }
                                float lg[4] = {acc[0] + pr.x, acc[1] + pr.y, acc[2] + pr.z, acc[3] + pr.w};
                                nm.readout_mlp(lg);
                                stg4(lg_st + (size_t)v * tile + l4, lg);
                            } else if constexpr (STASH) {
                                // training: the generic loop of the inference path below, with (m_it, a_it) of every edge
                                // (edge id b + k: canonical order) into the stash
                                float* tout = t_st + (size_t)b * tile + l4;
                                float acc[4] = {0.f, 0.f, 0.f, 0.f};
                                if (with_m)
                                    for (int k = 0; k < d; ++k) {      // ascending edge id
                                        const float4 mv = lds4(rows + k * tile);
                                        acc[0] += mv.x; acc[1] += mv.y; acc[2] += mv.z; acc[3] += mv.w;
                                    }
                                const float prv[4] = {pr.x, pr.y, pr.z, pr.w};
                                for (int k = 0; k < d; ++k) {
                                    float mo[4] = {0.f, 0.f, 0.f, 0.f};
                                    if (with_m) {
                                        const float4 mv = lds4(rows + k * tile);
                                        mo[0] = mv.x; mo[1] = mv.y; mo[2] = mv.z; mo[3] = mv.w;
                                    }
                                    const float ext[4] = {acc[0] - mo[0], acc[1] - mo[1], acc[2] - mo[2], acc[3] - mo[3]};
                                    float a[4], out[4];
                                    nm.var_update_a(ext, prv, a, out);
                                    stg4(tout + k * tile, out);
                                    stash4((size_t)it * 2 * E + b + k, s0, nvalid, mo);
                                    stash4((size_t)(it * 2 + 1) * E + b + k, s0, nvalid, a);
                                }
                            } else {
                                float* tout = t_st + (size_t)b * tile + l4;
#define GD_VAR_CALL(D) nm.template var_node<D>(rows, tile, pr, tout)
                                if (with_m) {
                                    GD_DEGREE_SWITCH(d, GD_VAR_CALL, {
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
                                } else {                                    // first iteration: every message is 0
                                    const float ext[4] = {0.f, 0.f, 0.f, 0.f}, prv[4] = {pr.x, pr.y, pr.z, pr.w};
                                    float out[4];
                                    nm.var_update(ext, prv, out);
                                    for (int k = 0; k < d; ++k) stg4(tout + k * tile, out);
                                }
#undef GD_VAR_CALL
                            }
                            b = b_next;
                        }
                    }
                    __syncwarp();     // every lane is done with this stage before it is refilled
                }
            }
            tma::fence_async_all();   // this thread's generic stores -> visible to the bulk copies of the next phase
            __syncthreads();
            if (readout) break;
            // ---- check phase ----
            {
                const bool ld_m = with_m && !kIsBP;
                int c = w, sidx = 0;
                for (int q = 0; q < S - 1; ++q)
                    if (c + q * W < C) issue_chk(c + q * W, q, ld_m);
                for (; c < C; c += W, sidx = sidx + 1 == S ? 0 : sidx + 1) {
                    if (c + (S - 1) * W < C) issue_chk(c + (S - 1) * W, sidx == 0 ? S - 1 : sidx - 1, ld_m);
                    wait_stage(sidx);
                    const float* st = stg0 + sidx * stage_floats + l4;
                    const int b = __ldg(tb.chk_ptr + c), d = __ldg(tb.chk_ptr + c + 1) - b;
                    if (active) {
                        float* m_out = m_st + l4;
                        const int32_t* edges = tb.chk_edges + b;
#define GD_CHK_CALL(D) nm.template chk_node<D>(st, tile, edges, m_out)
                        if (ld_m || kIsBP) {
                            GD_DEGREE_SWITCH(d, GD_CHK_CALL, {
                                float sg[4] = {1.f, 1.f, 1.f, 1.f};
                                if constexpr (kSign) {
                                    const float4 s4 = lds4(st + (ld_m ? 2 * d : d) * tile);
                                    sg[0] = s4.x; sg[1] = s4.y; sg[2] = s4.z; sg[3] = s4.w;
                                }
                                float acc[4] = {0.f, 0.f, 0.f, 0.f};
                                int cnt[4] = {0, 0, 0, 0};
                                for (int k = 0; k < d; ++k) {
                                    const float4 tv = lds4(st + k * tile);
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
                                    const size_t e = (size_t)__ldg(edges + k);
                                    const float4 tv = lds4(st + k * tile);
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
                                        const float4 mo = lds4(st + (d + k) * tile);
                                        out[0] = fmaf(oo[0], sg[0], mo.x);
                                        out[1] = fmaf(oo[1], sg[1], mo.y);
                                        out[2] = fmaf(oo[2], sg[2], mo.z);
                                        out[3] = fmaf(oo[3], sg[3], mo.w);
                                    }
                                    stg4(m_out + e * tile, out);
                                }
                            })
                        } else {
                            // first iteration of a learned program: no residual rows were fetched (m == 0)
                            if constexpr (!kIsBP) {
                            float sg[4] = {1.f, 1.f, 1.f, 1.f};
                            if constexpr (kSign) {
                                const float4 s4 = lds4(st + d * tile);
                                sg[0] = s4.x; sg[1] = s4.y; sg[2] = s4.z; sg[3] = s4.w;
                            }
                            float acc[4] = {0.f, 0.f, 0.f, 0.f};
                            for (int k = 0; k < d; ++k) {
                                const float4 tv = lds4(st + k * tile);
                                acc[0] += tv.x; acc[1] += tv.y; acc[2] += tv.z; acc[3] += tv.w;
                            }
                            for (int k = 0; k < d; ++k) {
                                const size_t e = (size_t)__ldg(edges + k);
                                const float4 tv = lds4(st + k * tile);
                                const float ext[4] = {acc[0] - tv.x, acc[1] - tv.y, acc[2] - tv.z, acc[3] - tv.w};
                                float oo[4];
                                nm.chk_mlp(ext, oo);
                                const float out[4] = {oo[0] * sg[0], oo[1] * sg[1], oo[2] * sg[2], oo[3] * sg[3]};
                                stg4(m_out + e * tile, out);
                            }
                            }
                        }
#undef GD_CHK_CALL
                    }
                    __syncwarp();
                }
            }
            tma::fence_async_all();
            __syncthreads();
        }

        // ---- outputs: lg[V][tile] -> prob / logit / hard [tile][V], transposed through shared memory ----
        {
            const int NC = ((scratch_floats / tile) - 1) & ~1;    // even -> odd pitch: conflict-free both ways
            const int pitch = NC + 1;
            for (int v0 = 0; v0 < V; v0 += NC) {
                const int nc = min(NC, V - v0);
                for (int i = tid; i < nc * tile; i += nthr) {
                    const int j = i / tile, si = i - j * tile;
                    scratch[si * pitch + j] = __ldcg(lg_st + (size_t)(v0 + j) * tile + si);
                }
                __syncthreads();
                for (int i = tid; i < nvalid * nc; i += nthr) {
                    const int si = i / nc, j = i - si * nc;
                    const float lg = scratch[si * pitch + j];
                    float pr = sigmoid_neg(lg);
                    if (kClamp) pr = fminf(fmaxf(pr, 1e-7f), 1.0f - 1e-7f);
                    const long long o = (s0 + si) * V + v0 + j;
                    if (p.prob) p.prob[o] = pr;
                    if (p.logit) p.logit[o] = lg;
                    if (p.hard) p.hard[o] = pr > 0.5f;
                }
                __syncthreads();
            }
        }
    }
}

static int align_up_i(int x, int a) { return (x + a - 1) / a * a; }

// Returns ok == false (and out->why) when the graph does not qualify (edges not in variable-sorted order, or a
// node's rows do not fit a pipeline stage): the caller then takes the register-batched kernel.
void plan_streamed_tma(const gd_graph* g, const gd_model* m, int64_t B, StreamTmaPlan* out, bool train) {
    StreamTmaParams& p = out->p;
    memset(&p, 0, sizeof(p));
    out->ok = false;
    out->why = "edges are not in the canonical variable-sorted order (H.to_sparse())";
    for (size_t i = 0; i < g->h_var_edges.size(); ++i)
        if (g->h_var_edges[i] != (int32_t)i) return;
    out->why = "a node's rows do not fit a pipeline stage in shared memory";
    const bool bp = m->program == GD_PROG_BP_QUANTUM || m->program == GD_PROG_BP_CLASSICAL;
    p.B = B; p.T = m->iters; p.V = g->V; p.C = g->C; p.E = (int)g->E; p.N = g->N;
    p.hid = bp ? 0 : m->hidden;
    p.hp = align_up_i(p.hid, m->program == GD_PROG_V2_4 ? 8 : 4);
    p.tb = g->t;
    const int n_slots = bp ? 0 : (m->program == GD_PROG_V2_4 ? 3 : 2);
    // The Softplus program is MUFU-bound, not HBM-bound: four syndromes per lane only pay when the
    // batch fills all 32 lanes of every SM; smaller batches take the register-batched kernel.
    if (m->program == GD_PROG_V2_4 && !train && B < (int64_t)128 * g->sm_count) {
        out->why = "batch too small to fill the SMs";
        return;
    }
    out->npad = 0;
    if ((m->program == GD_PROG_CGNNI || m->program == GD_PROG_QGNNI) && m->hidden < 32)
        out->npad = m->hidden < 16 ? 16 : 32;
    // tile: multiple of 4 (a lane owns one float4 of a row), <= 128.  Cost model: the kernel is
    // HBM-bound, a tile's time ~ its bytes ~ tile (with a floor: a warp instruction costs the
    // same for 12 active lanes as for 32), so minimise rounds * max(tile, floor); ties -> larger rows.
    int tile = 128;
    {
        double best = 1e300;
        for (int t = 8; t <= 128; t += 4) {
            const int64_t n_t = (B + t - 1) / t;
            const int64_t rounds = (n_t + g->sm_count - 1) / g->sm_count;
            const double cost = (double)rounds * (t > 48 ? t : 48);
            if (cost <= best * (1.0 + 1e-12)) { best = cost; tile = t; }
        }
    }
    p.tile = tile;
    p.lanes = tile / 4;
    const int vd = g->max_var_deg > 0 ? g->max_var_deg : 1;
    // rows per stage: a check item needs deg (+ deg residual rows for the learned programs) + 1; the sum-product family
    // could do with half, but bigger stages amortise the per-item cost better (variables per item K = rows / (vd + 1)):
    // measured on B200, sum-product / HGP-1600 / T = 50: 15 rows x 2 stages 28.4 ms, 8 rows x 2 / 3 / 4 stages 33.7 / 32.9 / 33.2 ms
    int rows = 2 * g->max_chk_deg + 1;
    if (rows < vd + 1) rows = vd + 1;
    int K = rows / (vd + 1);
    if (K > 8) K = 8;
    p.stage_rows = rows; p.vchunk = K; p.vrows = K * vd;
    const int stage_bytes = rows * tile * 4;
    int off = 16 * 4 * 8;                              // up to 16 warps x 4 mbarriers
    p.off_w = off; off += out->npad ? 2 * pwl_smem_floats(out->npad) * 4 : n_slots * 4 * p.hp * 4;
    off = align_up_i(off, 128);
    if (m->program == GD_PROG_V2_4 && !opt_on(OPT_NO_CTAB)) {
        // check-phase table on |ext| <= max check degree - 1 at the resident kernel's node spacing (512 pieces per +-3), read-out 2048
        p.ctab_R = (float)(g->max_chk_deg > 1 ? g->max_chk_deg - 1 : 1);
        p.ctab_n = (int)(512.0f * p.ctab_R / 3.0f + 0.5f);
        if (p.ctab_n < 512) p.ctab_n = 512;
        p.off_ctab = off; off += p.ctab_n * 16;
        p.rtab_n = 2048; p.off_rtab = off; off += p.rtab_n * 16;
    }
    p.off_stage = off;
    // stages per warp (2..4): 2 unless deeper still leaves room for all 16 warps at this stage size
    int S = 2;
    for (int q = 4; q > 2; --q)
        if ((g->max_smem_optin - off) / (q * stage_bytes) >= 16) { S = q; break; }
    p.S = S;
    int Wn = (g->max_smem_optin - off) / (S * stage_bytes);
    if (Wn > 16) Wn = 16;
    if (Wn < 2) return;
    if ((int64_t)Wn * S * rows * tile < 2 * (int64_t)(tile + 2) * 2) return;   // transposition scratch
    p.W = Wn;
    out->threads = Wn * 32;
    out->smem = off + Wn * S * stage_bytes;
    p.n_tiles = (int)((B + tile - 1) / tile);
    out->grid = p.n_tiles < g->sm_count ? p.n_tiles : g->sm_count;
    p.slab_floats = ((long long)g->N + 2 * g->E + g->V) * tile;
    out->ok = true;
}

int streamed_tma_decode(gd_graph* g, const StreamTmaPlan& plan, const gd_model* model, const DecodeIO& io, cudaStream_t st) {
    StreamTmaPlan pl = plan;
    pl.p.x = io.x; pl.p.prob = io.prob; pl.p.logit = io.logit; pl.p.hard = io.hard; pl.p.weights = io.weights;
    pl.p.stash = io.stash;
    pl.p.slab = streamed_slab(g, (size_t)pl.grid * (size_t)pl.p.slab_floats * sizeof(float));
    if (!pl.p.slab) return GD_ERR_CUDA;
    void (*k)(const StreamTmaParams);
    if (io.stash && model->program != GD_PROG_V2_4) {
        set_error("gd_decode_fwd_train: the streamed kernel writes a training stash for GD_PROG_V2_4 only");
        return GD_ERR_UNSUPPORTED;
    }
    switch (model->program) {
        case GD_PROG_CGNNI:
            k = pl.npad == 16 ? decode_streamed_tma_kernel<GD_PROG_CGNNI, 16>
                : pl.npad == 32 ? decode_streamed_tma_kernel<GD_PROG_CGNNI, 32> : decode_streamed_tma_kernel<GD_PROG_CGNNI, 0>;
            break;
        case GD_PROG_QGNNI:
            k = pl.npad == 16 ? decode_streamed_tma_kernel<GD_PROG_QGNNI, 16>
                : pl.npad == 32 ? decode_streamed_tma_kernel<GD_PROG_QGNNI, 32> : decode_streamed_tma_kernel<GD_PROG_QGNNI, 0>;
            break;
        case GD_PROG_V2_4:
            k = io.stash ? decode_streamed_tma_kernel<GD_PROG_V2_4, 0, true> : decode_streamed_tma_kernel<GD_PROG_V2_4, 0>;
            break;
        case GD_PROG_BP_QUANTUM: k = decode_streamed_tma_kernel<GD_PROG_BP_QUANTUM, 0>; break;
        default: k = decode_streamed_tma_kernel<GD_PROG_BP_CLASSICAL, 0>; break;
    }
    GD_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, pl.smem));
    k<<<pl.grid, pl.threads, pl.smem, st>>>(pl.p);
    GD_CUDA(cudaGetLastError());
    return GD_OK;
}

}  // namespace gd
