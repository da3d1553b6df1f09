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
    static constexpr bool kSign = (PROG == GD_PROG_QGNNI || PROG == GD_PROG_V2_4 || PROG == GD_PROG_BP_QUANTUM);
    static constexpr float kLogEps1 = PROG == GD_PROG_BP_QUANTUM ? -46.0517019f : -16.1180957f;
    static constexpr float kEps2 = PROG == GD_PROG_BP_QUANTUM ? 1e-12f : 1e-7f;
    MlpSmem W1, W2, W3;
    PwlSmem P2, P3;
    int hp;
    // decoder_v2_4 in the streamed kernel: the two 1 -> h -> 1 Softplus MLPs as cubic tables (gd_math.cuh, CubicTab), used when
    // the kernel's error bound allows; the 2-input variable-phase MLP stays a direct evaluation there
    CubicTab ctab, rtab;
    bool use_ctab, use_rtab;
    float rtab_R;

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
