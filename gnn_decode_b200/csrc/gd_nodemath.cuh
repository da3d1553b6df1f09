// Per-node arithmetic of the phase programs on FOUR syndromes at a time (a lane owns one float4 of every
// batch-minor state row): shared by the TMA-staged streamed kernel (gd_streamed_tma.cu) and the node-owner
// resident kernel for the light programs (gd_decode_light.cu).
#pragma once
#include "gd_common.cuh"
#include "gd_math.cuh"

namespace gd {

__device__ __forceinline__ float4 lds4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void stg4(float* p, const float (&v)[4]) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
}

__device__ __forceinline__ void stage_mlp_t(float* dst, int hp, int hid, const float* w1, int w1_stride, bool two_in,
                                            const float* b1, const float* w2, float s1, float s2, int tid, int nthr) {
    for (int k = tid; k < hp; k += nthr) {
        const bool in = k < hid;
        dst[k] = in ? w1[k * w1_stride] * s1 : 0.f;
        dst[hp + k] = (in && two_in) ? w1[k * w1_stride + 1] * s1 : 0.f;
        dst[2 * hp + k] = in ? b1[k] * s1 : 0.f;
        dst[3 * hp + k] = in ? w2[k] * s2 : 0.f;
    }
}


// ---- per-node arithmetic on FOUR syndromes (one float4 of every row) --------------------------
template <int PROG, int NPAD>
struct NodeMath {
    static constexpr bool kIsBP = (PROG == GD_PROG_BP_QUANTUM || PROG == GD_PROG_BP_CLASSICAL);
    static constexpr bool kSoftplus = (PROG == GD_PROG_V2_4);
    // neural BP (quantum/neural_BP.py): the BP_QUANTUM check phase with eps1 = 1e-20, eps2 = 1e-15 and a residual alpha * m;
    // its per-edge weights are read by the kernel from global memory, not staged
    static constexpr bool kNBP = (PROG == GD_PROG_NEURAL_BP);
    static constexpr bool kSign = (PROG == GD_PROG_QGNNI || PROG == GD_PROG_V2_4 || PROG == GD_PROG_BP_QUANTUM || kNBP);
    static constexpr float kLogEps1 = (PROG == GD_PROG_BP_QUANTUM || kNBP) ? -46.0517019f : -16.1180957f;
    static constexpr float kEps2 = PROG == GD_PROG_BP_QUANTUM ? 1e-12f : kNBP ? 1e-15f : 1e-7f;
    MlpSmem W1, W2, W3;
    PwlSmem P2, P3;
    int hp;
    // decoder_v2_4 in the streamed kernel: the two 1 -> h -> 1 Softplus MLPs as cubic tables (gd_math.cuh, CubicTab), used when
    // the kernel's error bound allows; the 2-input variable-phase MLP stays a direct evaluation there
    CubicTab ctab, rtab;
    bool use_ctab, use_rtab;
    float rtab_R;
    float alpha;     // neural BP's residual weight

    // neural BP variable phase, one edge and syndrome (neural_BP.py:244-258): u = (sum of the variable's W m) - own W m +
    // W_p prior, and the value the check phase sums, log|tanh(u/2)| with no input clamp and the sign of u in its sign bit.
    // Past |u| ~ 87 exp(-|u|) underflows and log|tanh| would be 0, whose negation is not > 0, so the sign of u would be lost:
    // -FLT_MIN keeps it strictly negative (far below any rounding of the sums it enters).  The training backward
    // (gd_backward_nbp.cu) recomputes u and t with these two, so its clamp decisions and parities are the forward's.
    static __device__ __forceinline__ float nbp_u(float acc, float m, float wk, float pr, float wpk) { return acc - m * wk + pr * wpk; }
    static __device__ __forceinline__ float nbp_t(float a) {
        const float tv = fminf(bp_log_abs_tanh_half<false>(a, kLogEps1), -1.17549435e-38f);
        return a < 0.f ? -tv : tv;
    }

    // variable phase: ext = (sum of siblings) - own, prior -> the value the check phase sums
    __device__ __forceinline__ void var_update(const float (&ext)[4], const float (&pr)[4], float (&out)[4]) const {
        if constexpr (PROG == GD_PROG_V2_4) {
            float a[4];
            var_update_a(ext, pr, a, out);
        } else if constexpr (kIsBP) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float a = ext[j] + pr[j];
                const float tv = bp_log_abs_tanh_half(a, kLogEps1);   // < 0 always
                out[j] = a < 0.f ? -tv : tv;                         // stored > 0 <=> tanh(a/2) < 0
            }
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) out[j] = tanh_half_fast(ext[j] + pr[j]);
        }
    }
    // decoder_v2_4's variable phase that also returns a = mlp(ext, prior), the value before tanh(a/2): the training stash keeps it
    __device__ __forceinline__ void var_update_a(const float (&ext)[4], const float (&pr)[4], float (&a)[4],
                                                 float (&out)[4]) const {
        mlp_softplus_x2<4, true, 2>(W1, hp, ext, pr, a);
#pragma unroll
        for (int j = 0; j < 4; ++j) out[j] = tanh_half_fast(a[j]);
    }
    // check phase (learned programs): mlp(ext)
    __device__ __forceinline__ void chk_mlp(const float (&ext)[4], float (&oo)[4]) const {
        if constexpr (kSoftplus) {
            if (use_ctab) {                  // |ext| <= check degree - 1 by construction: always inside the table
#pragma unroll
                for (int j = 0; j < 4; ++j) oo[j] = cubic_tab_eval(ctab, ext[j]);
            } else {
                mlp_softplus_x2<4, false, 2>(W2, hp, ext, ext, oo);
            }
        } else if constexpr (NPAD > 0) {
#pragma unroll
            for (int j = 0; j < 4; ++j) oo[j] = pwl_eval<NPAD>(P2, ext[j]);
        } else {
            mlp_relu<4>(W2, hp, ext, oo);
        }
    }
    // decoder_v2_4's per-edge read-out mlp(m) (decoder_v2_4.py:291)
    __device__ __forceinline__ void readout_edge(const float (&m)[4], float (&oo)[4]) const {
        bool in_range = use_rtab;
#pragma unroll
        for (int j = 0; j < 4; ++j) in_range = in_range && fabsf(m[j]) <= rtab_R;
        if (in_range) {
#pragma unroll
            for (int j = 0; j < 4; ++j) oo[j] = cubic_tab_eval(rtab, m[j]);
        } else {
            mlp_softplus_x2<4, false, 2>(W3, hp, m, m, oo);
        }
    }
    __device__ __forceinline__ void readout_mlp(float (&lg)[4]) const {
        if constexpr (PROG == GD_PROG_CGNNI || PROG == GD_PROG_QGNNI) {
            if constexpr (NPAD > 0) {
#pragma unroll
                for (int j = 0; j < 4; ++j) lg[j] = pwl_eval<NPAD>(P3, lg[j]);
            } else {
                float oo[4];
                mlp_relu<4>(W3, hp, lg, oo);
#pragma unroll
                for (int j = 0; j < 4; ++j) lg[j] = oo[j];
            }
        }
    }

    // One variable of degree D, messages present (it > 0): rows[k*tile] = m of its k-th edge (shared),
    // tout[k*tile] = where t of that edge goes (global).  Fully unrolled, values stay in registers.
    template <int D>
    __device__ __forceinline__ void var_node(const float* rows, int tile, const float4 pr4, float* tout) const {
        float4 mv[D];
#pragma unroll
        for (int k = 0; k < D; ++k) mv[k] = lds4(rows + k * tile);
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int k = 0; k < D; ++k) {        // ascending edge id
            acc[0] += mv[k].x; acc[1] += mv[k].y; acc[2] += mv[k].z; acc[3] += mv[k].w;
        }
        const float pr[4] = {pr4.x, pr4.y, pr4.z, pr4.w};
#pragma unroll
        for (int k = 0; k < D; ++k) {
            const float ext[4] = {acc[0] - mv[k].x, acc[1] - mv[k].y, acc[2] - mv[k].z, acc[3] - mv[k].w};
            float out[4];
            var_update(ext, pr, out);
            stg4(tout + k * tile, out);
        }
    }
    // One check of degree D with the residual rows present: st rows [0,D) = t, [D,2D) = m, row 2D = sign.
    template <int D>
    __device__ __forceinline__ void chk_node(const float* st, int tile, const int32_t* edges, float* m_out) const {
        int e[D];
#pragma unroll
        for (int k = 0; k < D; ++k) e[k] = __ldg(edges + k);
        float4 tv[D];
#pragma unroll
        for (int k = 0; k < D; ++k) tv[k] = lds4(st + k * tile);
        float sg[4] = {1.f, 1.f, 1.f, 1.f};
        if constexpr (kSign) {
            const float4 s4 = lds4(st + (kIsBP ? D : 2 * D) * tile);
            sg[0] = s4.x; sg[1] = s4.y; sg[2] = s4.z; sg[3] = s4.w;
        }
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
        int cnt[4] = {0, 0, 0, 0};
#pragma unroll
        for (int k = 0; k < D; ++k) {
            const float t4[4] = {tv[k].x, tv[k].y, tv[k].z, tv[k].w};
#pragma unroll
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
#pragma unroll
            for (int j = 0; j < 4; ++j) cnt[j] += sg[j] < 0.f ? 1 : 0;
        }
#pragma unroll
        for (int k = 0; k < D; ++k) {
            const float t4[4] = {tv[k].x, tv[k].y, tv[k].z, tv[k].w};
            float out[4];
            if constexpr (kIsBP) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int q = cnt[j] - (t4[j] > 0.f ? 1 : 0);
                    out[j] = bp_check_out(acc[j] + fabsf(t4[j]), q & 1, kEps2);
                }
            } else {
                float ext[4], oo[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) ext[j] = acc[j] - t4[j];
                chk_mlp(ext, oo);
                const float4 mo = lds4(st + (D + k) * tile);
                out[0] = fmaf(oo[0], sg[0], mo.x);
                out[1] = fmaf(oo[1], sg[1], mo.y);
                out[2] = fmaf(oo[2], sg[2], mo.z);
                out[3] = fmaf(oo[3], sg[3], mo.w);
            }
            stg4(m_out + (size_t)e[k] * tile, out);
        }
    }

    // Neural BP, one check: st rows [0,d) = t, then (res: residual rows present) [d,2d) = m, then the sign row.  t carries
    // log|tanh| <= 0 with the sign flag in its sign bit.  Each edge's sum over its siblings is formed without subtracting its
    // own term: a message without input clamp saturates, its log|tanh| (down to log 1e-20 = -46) would swamp the tiny terms
    // of saturated siblings in fp32 (sum - own loses them), and those terms set the output's magnitude.
    __device__ __forceinline__ void nbp_chk_out(const float (&ext)[4], const float (&t4)[4], const int (&cnt)[4], const float* st,
                                                int tile, int d, int k, bool res, float* dst) const {
        float out[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int q = cnt[j] - (t4[j] > 0.f ? 1 : 0);
            out[j] = bp_check_out(ext[j], q & 1, kEps2);
        }
        if (res) {                                    // neural_BP.py:304: + alpha * m_p (m == 0 in the first iteration)
            const float4 mo = lds4(st + (d + k) * tile);
            out[0] = fmaf(alpha, mo.x, out[0]);
            out[1] = fmaf(alpha, mo.y, out[1]);
            out[2] = fmaf(alpha, mo.z, out[2]);
            out[3] = fmaf(alpha, mo.w, out[3]);
        }
        stg4(dst, out);
    }
    // the syndrome sign's share of the parity (the row after the t rows, and after the m rows when they are present)
    __device__ __forceinline__ void nbp_sign_count(const float* st, int tile, int d, bool res, int (&cnt)[4]) const {
        const float4 s4 = lds4(st + (res ? 2 * d : d) * tile);
        cnt[0] = s4.x < 0.f ? 1 : 0; cnt[1] = s4.y < 0.f ? 1 : 0; cnt[2] = s4.z < 0.f ? 1 : 0; cnt[3] = s4.w < 0.f ? 1 : 0;
    }
    // degree D: each edge's exclusive sum of -|t| as prefix + suffix, in registers; cnt += the edges whose t flags a negative u
    template <int D>
    static __device__ __forceinline__ void nbp_exclusive(const float4 (&tv)[D], float (&ext)[D][4], int (&cnt)[4]) {
        float run[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int k = 0; k < D; ++k) {
            const float t4[4] = {tv[k].x, tv[k].y, tv[k].z, tv[k].w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                ext[k][j] = run[j];
                run[j] -= fabsf(t4[j]);
                cnt[j] += t4[j] > 0.f ? 1 : 0;
            }
        }
        run[0] = run[1] = run[2] = run[3] = 0.f;
#pragma unroll
        for (int k = D - 1; k >= 0; --k) {
            const float t4[4] = {tv[k].x, tv[k].y, tv[k].z, tv[k].w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                ext[k][j] += run[j];
                run[j] -= fabsf(t4[j]);
            }
        }
    }
    // any degree: edge k's exclusive sum directly, ascending over the others; row(i) = t of the check's i-th edge
    template <class Row>
    static __device__ __forceinline__ void nbp_exclusive_any(const Row& row, int d, int k, float (&ext)[4]) {
        ext[0] = ext[1] = ext[2] = ext[3] = 0.f;
        for (int i = 0; i < d; ++i) {
            if (i == k) continue;
            const float4 tv = row(i);
            ext[0] -= fabsf(tv.x); ext[1] -= fabsf(tv.y); ext[2] -= fabsf(tv.z); ext[3] -= fabsf(tv.w);
        }
    }
    // degree D, unrolled: exclusive sums as prefix + suffix, in registers
    template <int D>
    __device__ __forceinline__ void nbp_chk_node(const float* st, int tile, const int32_t* edges, float* m_out, bool res) const {
        float4 tv[D];
#pragma unroll
        for (int k = 0; k < D; ++k) tv[k] = lds4(st + k * tile);
        int cnt[4];
        nbp_sign_count(st, tile, D, res, cnt);
        float ext[D][4];
        nbp_exclusive<D>(tv, ext, cnt);
#pragma unroll
        for (int k = 0; k < D; ++k) {
            const float t4[4] = {tv[k].x, tv[k].y, tv[k].z, tv[k].w};
            nbp_chk_out(ext[k], t4, cnt, st, tile, D, k, res, m_out + (size_t)__ldg(edges + k) * tile);
        }
    }
    // any degree (past the unrolled ones): each exclusive sum directly from shared memory, O(d^2)
    __device__ __forceinline__ void nbp_chk_any(const float* st, int tile, const int32_t* edges, float* m_out, int d, bool res) const {
        int cnt[4];
        nbp_sign_count(st, tile, d, res, cnt);
        for (int k = 0; k < d; ++k) {
            const float4 tv = lds4(st + k * tile);
            cnt[0] += tv.x > 0.f ? 1 : 0; cnt[1] += tv.y > 0.f ? 1 : 0; cnt[2] += tv.z > 0.f ? 1 : 0; cnt[3] += tv.w > 0.f ? 1 : 0;
        }
        const auto row = [&](int i) { return lds4(st + i * tile); };
        for (int k = 0; k < d; ++k) {
            float ext[4];
            nbp_exclusive_any(row, d, k, ext);
            const float4 tv = lds4(st + k * tile);
            const float t4[4] = {tv.x, tv.y, tv.z, tv.w};
            nbp_chk_out(ext, t4, cnt, st, tile, d, k, res, m_out + (size_t)__ldg(edges + k) * tile);
        }
    }
};

#define GD_DEGREE_SWITCH(d, CALL, ...)      \
    switch (d) {                            \
        case 1: { CALL(1); } break;         \
        case 2: { CALL(2); } break;         \
        case 3: { CALL(3); } break;         \
        case 4: { CALL(4); } break;         \
        case 5: { CALL(5); } break;         \
        case 6: { CALL(6); } break;         \
        case 7: { CALL(7); } break;         \
        case 8: { CALL(8); } break;         \
        default: { __VA_ARGS__; } break;    \
    }

}  // namespace gd
