// Per-edge arithmetic of the phase programs: the k->h->1 MLPs (evaluated as FMA + MUFU in
// registers -- they are scalar->scalar functions, not GEMMs: SURVEY.md section 7 "hard parts"),
// tanh(m/2), and the sum-product check update.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace gd {

constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;

__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float lg2_approx(float x) {
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// One k->h->1 MLP staged in shared memory as SoA rows padded to a multiple of 4 hidden units
// (padding units have w2 == 0).  For Softplus MLPs the rows are PRE-SCALED when staged:
//   w1*log2(e), b1*log2(e), w2*ln(2)   so that
//   w2*softplus(w1 x + b1) == (w2 ln2) * [ max(z',0) + lg2(1 + 2^-|z'|) ],  z' = (w1 log2e) x + b1 log2e
// which needs exactly one ex2 and one lg2 (MUFU) per hidden unit.
struct MlpSmem {
    const float* w1a;  // [hp] weight of input 0
    const float* w1b;  // [hp] weight of input 1 (2-input MLPs only)
    const float* b1;   // [hp]
    const float* w2;   // [hp]
    float b2;
};

// floats needed in shared memory for one MLP slot
__host__ __device__ constexpr int mlp_smem_floats(int hp) { return 4 * hp; }

// Evaluate a Softplus MLP for EB independent edges at once (weights are loaded once per 4
// hidden units as 128-bit broadcast LDS and reused across the EB edges).
template <int EB, bool TWO_IN>
__device__ __forceinline__ void mlp_softplus(const MlpSmem& W, int hp, const float (&x0)[EB],
                                             const float (&x1)[EB], float (&out)[EB]) {
    float acc[EB];
#pragma unroll
    for (int j = 0; j < EB; ++j) acc[j] = 0.f;
#pragma unroll 1
    for (int k = 0; k < hp; k += 4) {
        const float4 a4 = *reinterpret_cast<const float4*>(W.w1a + k);
        const float4 b4 = *reinterpret_cast<const float4*>(W.b1 + k);
        const float4 c4 = *reinterpret_cast<const float4*>(W.w2 + k);
        float4 d4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (TWO_IN) d4 = *reinterpret_cast<const float4*>(W.w1b + k);
        const float a[4] = {a4.x, a4.y, a4.z, a4.w};
        const float b[4] = {b4.x, b4.y, b4.z, b4.w};
        const float c[4] = {c4.x, c4.y, c4.z, c4.w};
        const float d[4] = {d4.x, d4.y, d4.z, d4.w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
#pragma unroll
            for (int j = 0; j < EB; ++j) {
                float z = fmaf(a[u], x0[j], b[u]);
                if (TWO_IN) z = fmaf(d[u], x1[j], z);
                const float t = ex2_approx(-fabsf(z));
                const float l = lg2_approx(1.0f + t);
                const float s = fmaxf(z, 0.f) + l;
                acc[j] = fmaf(c[u], s, acc[j]);
            }
        }
    }
#pragma unroll
    for (int j = 0; j < EB; ++j) out[j] = acc[j] + W.b2;
}

// ---- packed (f32x2) Softplus MLP --------------------------------------------------------------
// The scalar loop above is bound by the MUFU pipe (2 MUFU = 16 pipe cycles per hidden unit per
// warp, 95% busy in ncu) while the FMA pipe idles at ~29% and only ~55% of the issue slots are
// used.  This version (a) packs two HIDDEN UNITS into one fma.rn.f32x2 / add.rn.f32x2 so the
// FMA-type work costs half the issue slots, and (b) for NPOLY of every 4 unit pairs evaluates
// lg2(1 + t), t = 2^-|z| in (0, 1], as t * q(t) with a degree-7 minimax polynomial q on the FMA
// pipe instead of MUFU.LG2 (max abs error 2.1e-7 in fp32 arithmetic, the same as
// lg2.approx(1 + t) whose 1 + t rounding alone costs 6e-8) -- shifting work from the saturated
// pipe to the idle one.
__device__ __forceinline__ unsigned long long pack2(float lo, float hi) {
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack2(unsigned long long v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ unsigned long long fma2(unsigned long long a, unsigned long long b, unsigned long long c) {
    unsigned long long d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ unsigned long long add2(unsigned long long a, unsigned long long b) {
    unsigned long long d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}

// q(t) ~= lg2(1 + t) / t on [0, 1], degree 7, fitted so that max |t q(t) - lg2(1 + t)| is minimal.
__device__ __constant__ float kLg2Poly[8] = {1.442689881f, -0.721165802f, 0.478683666f, -0.3473009499f,
                                             0.2418644786f, -0.1375209878f, 0.0520587736f, -0.0093091058f};

template <int EB, bool TWO_IN, int NPOLY>
__device__ __forceinline__ void mlp_softplus_x2(const MlpSmem& W, int hp, const float (&x0)[EB],
                                                const float (&x1)[EB], float (&out)[EB]) {
    unsigned long long acc[EB], xx[EB], yy[EB];
#pragma unroll
    for (int j = 0; j < EB; ++j) {
        acc[j] = 0ull;
        xx[j] = pack2(x0[j], x0[j]);
        yy[j] = pack2(x1[j], x1[j]);
    }
    unsigned long long cq[8];
    if (NPOLY > 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) cq[i] = pack2(kLg2Poly[i], kLg2Poly[i]);
    }
    const unsigned long long one2 = pack2(1.0f, 1.0f);
#pragma unroll 1
    for (int k = 0; k < hp; k += 8) {
        const ulonglong2 a01 = *reinterpret_cast<const ulonglong2*>(W.w1a + k);
        const ulonglong2 a23 = *reinterpret_cast<const ulonglong2*>(W.w1a + k + 4);
        const ulonglong2 b01 = *reinterpret_cast<const ulonglong2*>(W.b1 + k);
        const ulonglong2 b23 = *reinterpret_cast<const ulonglong2*>(W.b1 + k + 4);
        const ulonglong2 c01 = *reinterpret_cast<const ulonglong2*>(W.w2 + k);
        const ulonglong2 c23 = *reinterpret_cast<const ulonglong2*>(W.w2 + k + 4);
        ulonglong2 d01 = make_ulonglong2(0ull, 0ull), d23 = d01;
        if (TWO_IN) {
            d01 = *reinterpret_cast<const ulonglong2*>(W.w1b + k);
            d23 = *reinterpret_cast<const ulonglong2*>(W.w1b + k + 4);
        }
        const unsigned long long a[4] = {a01.x, a01.y, a23.x, a23.y};
        const unsigned long long b[4] = {b01.x, b01.y, b23.x, b23.y};
        const unsigned long long c[4] = {c01.x, c01.y, c23.x, c23.y};
        const unsigned long long d[4] = {d01.x, d01.y, d23.x, d23.y};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
#pragma unroll
            for (int j = 0; j < EB; ++j) {
                unsigned long long z2 = fma2(a[u], xx[j], b[u]);
                if (TWO_IN) z2 = fma2(d[u], yy[j], z2);
                float zl, zh;
                unpack2(z2, zl, zh);
                const float tl = ex2_approx(-fabsf(zl)), th = ex2_approx(-fabsf(zh));
                const unsigned long long m2 = pack2(fmaxf(zl, 0.f), fmaxf(zh, 0.f));
                const unsigned long long t2 = pack2(tl, th);
                unsigned long long s2;
                if (u < NPOLY) {
                    unsigned long long q2 = fma2(cq[7], t2, cq[6]);
#pragma unroll
                    for (int i = 5; i >= 0; --i) q2 = fma2(q2, t2, cq[i]);
                    s2 = fma2(t2, q2, m2);
                } else {
                    float ul, uh;
                    unpack2(add2(t2, one2), ul, uh);
                    s2 = add2(pack2(lg2_approx(ul), lg2_approx(uh)), m2);
                }
                acc[j] = fma2(c[u], s2, acc[j]);
            }
        }
    }
#pragma unroll
    for (int j = 0; j < EB; ++j) {
        float lo, hi;
        unpack2(acc[j], lo, hi);
        out[j] = (lo + hi) + W.b2;
    }
}

// ReLU MLP (CGNNI / QGNNI, hidden 10): 3 instructions per hidden unit, no MUFU.
template <int EB>
__device__ __forceinline__ void mlp_relu(const MlpSmem& W, int hp, const float (&x0)[EB], float (&out)[EB]) {
    float acc[EB];
#pragma unroll
    for (int j = 0; j < EB; ++j) acc[j] = 0.f;
#pragma unroll 1
    for (int k = 0; k < hp; k += 4) {
        const float4 a4 = *reinterpret_cast<const float4*>(W.w1a + k);
        const float4 b4 = *reinterpret_cast<const float4*>(W.b1 + k);
        const float4 c4 = *reinterpret_cast<const float4*>(W.w2 + k);
        const float a[4] = {a4.x, a4.y, a4.z, a4.w};
        const float b[4] = {b4.x, b4.y, b4.z, b4.w};
        const float c[4] = {c4.x, c4.y, c4.z, c4.w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
#pragma unroll
            for (int j = 0; j < EB; ++j) {
                const float z = fmaf(a[u], x0[j], b[u]);
                acc[j] = fmaf(c[u], fmaxf(z, 0.f), acc[j]);
            }
        }
    }
#pragma unroll
    for (int j = 0; j < EB; ++j) out[j] = acc[j] + W.b2;
}

// 2 -> h -> 1 ReLU MLP (decoder_v3_0.py:217-222: [sum over the other edges, node input]); W.w1b holds the second input's weights
template <int EB>
__device__ __forceinline__ void mlp_relu2(const MlpSmem& W, int hp, const float (&x0)[EB], const float (&x1)[EB], float (&out)[EB]) {
    float acc[EB];
#pragma unroll
    for (int j = 0; j < EB; ++j) acc[j] = 0.f;
#pragma unroll 1
    for (int k = 0; k < hp; k += 4) {
        const float4 a4 = *reinterpret_cast<const float4*>(W.w1a + k);
        const float4 d4 = *reinterpret_cast<const float4*>(W.w1b + k);
        const float4 b4 = *reinterpret_cast<const float4*>(W.b1 + k);
        const float4 c4 = *reinterpret_cast<const float4*>(W.w2 + k);
        const float a[4] = {a4.x, a4.y, a4.z, a4.w}, d[4] = {d4.x, d4.y, d4.z, d4.w};
        const float b[4] = {b4.x, b4.y, b4.z, b4.w}, c[4] = {c4.x, c4.y, c4.z, c4.w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
#pragma unroll
            for (int j = 0; j < EB; ++j) {
                const float z = fmaf(a[u], x0[j], fmaf(d[u], x1[j], b[u]));
                acc[j] = fmaf(c[u], fmaxf(z, 0.f), acc[j]);
            }
        }
    }
#pragma unroll
    for (int j = 0; j < EB; ++j) out[j] = acc[j] + W.b2;
}

__device__ __forceinline__ float rcp_fast(float x);
// 2 -> h -> 1 Tanh MLP (decoder_v1_2_2.py:216-220, 245-248; h = 256).  The staged first layer is pre-scaled by 2 log2(e), so that
// tanh(z) = 1 - 2 / (1 + 2^(z')) costs one ex2 and one rcp (abs. error ~2e-7, as tanh_half_fast); padded units have w2 = 0.
template <int EB>
__device__ __forceinline__ void mlp_tanh2(const MlpSmem& W, int hp, const float (&x0)[EB], const float (&x1)[EB], float (&out)[EB]) {
    float acc[EB];
#pragma unroll
    for (int j = 0; j < EB; ++j) acc[j] = 0.f;
#pragma unroll 1
    for (int k = 0; k < hp; k += 4) {
        const float4 a4 = *reinterpret_cast<const float4*>(W.w1a + k);
        const float4 d4 = *reinterpret_cast<const float4*>(W.w1b + k);
        const float4 b4 = *reinterpret_cast<const float4*>(W.b1 + k);
        const float4 c4 = *reinterpret_cast<const float4*>(W.w2 + k);
        const float a[4] = {a4.x, a4.y, a4.z, a4.w}, d[4] = {d4.x, d4.y, d4.z, d4.w};
        const float b[4] = {b4.x, b4.y, b4.z, b4.w}, c[4] = {c4.x, c4.y, c4.z, c4.w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
#pragma unroll
            for (int j = 0; j < EB; ++j) {
                const float z2 = fmaf(a[u], x0[j], fmaf(d[u], x1[j], b[u]));         // = 2 log2(e) z
                const float th = fmaf(-2.0f, rcp_fast(1.0f + ex2_approx(z2)), 1.0f);
                acc[j] = fmaf(c[u], th, acc[j]);
            }
        }
    }
#pragma unroll
    for (int j = 0; j < EB; ++j) out[j] = acc[j] + W.b2;
}

// ---- 1 -> h -> 1 ReLU MLP as the piecewise-linear function it is --------------------------------
// f(x) = b2 + sum_u c_u relu(a_u x + b_u) has at most h breakpoints t_u = -b_u / a_u; between two
// consecutive breakpoints it is one line S_j x + I_j.  One warp builds the sorted breakpoints and
// the (S_j, I_j) table once per CTA in double precision (exactly the reference's sum, rounded once),
// then every evaluation is a branch-free binary search (log2 NPAD shared-memory loads; the tables
// have <= 32 words, so two lanes on the same bank read the same word: conflict-free) + ONE FMA
// instead of 3h instructions.  f is continuous, so landing in the neighbouring segment within an
// ulp of a breakpoint changes nothing beyond rounding.  Used when h < NPAD <= 32 (the reference's
// CGNNI / QGNNI have h = 10: classical/CGNNI.py:217-222, quantum/QGNNI.py:190-194).
struct PwlSmem {
    const float* bp;    // [NPAD] ascending breakpoints, +inf padded (entries 0 .. NPAD-2 are searched)
    const float2* seg;  // [NPAD] (slope, intercept) of segment j = #{breakpoints < x}
};
__host__ __device__ constexpr int pwl_smem_floats(int npad) { return 3 * npad; }

// Called by ONE full warp.  w1[h], b1[h], w2[h] are the reference's Linear(1,h).weight/bias and
// Linear(h,1).weight (global memory), h < npad <= 32.
__device__ __forceinline__ void pwl_build(float* bp, float2* seg, int npad, const float* w1, const float* b1,
                                          const float* w2, float b2, int h, int lane) {
    const double a = lane < h ? (double)w1[lane] : 0.0, b = lane < h ? (double)b1[lane] : 0.0;
    const double c = lane < h ? (double)w2[lane] : 0.0;
    const float t = (lane < h && a != 0.0) ? (float)(-b / a) : __int_as_float(0x7f800000);
    int rank = 0;
    for (int v = 0; v < h; ++v) {
        const float tv = __shfl_sync(0xffffffffu, t, v);
        rank += (tv < t || (tv == t && v < lane)) ? 1 : 0;
    }
    if (lane < h) bp[rank] = t;
    else if (lane < npad) bp[lane] = __int_as_float(0x7f800000);
    double S = 0.0, I = (double)b2;
    for (int v = 0; v < h; ++v) {
        const double av = __shfl_sync(0xffffffffu, a, v), bv = __shfl_sync(0xffffffffu, b, v);
        const double cv = __shfl_sync(0xffffffffu, c, v);
        const int rv = __shfl_sync(0xffffffffu, rank, v);
        if (av == 0.0) {
            I += cv * (bv > 0.0 ? bv : 0.0);
        } else if (av > 0.0 ? (rv < lane) : (rv >= lane)) {   // unit v is active on segment `lane`
            S += cv * av;
            I += cv * bv;
        }
    }
    if (lane < npad) seg[lane] = make_float2((float)S, (float)I);
}

// The segment pwl_eval evaluates x on (the backward needs its index and slope).
template <int NPAD>
__device__ __forceinline__ int pwl_segment(const PwlSmem& P, float x) {
    int i = 0;
#pragma unroll
    for (int s = NPAD / 2; s >= 1; s >>= 1) i += (P.bp[i + s - 1] < x) ? s : 0;
    return i;
}

template <int NPAD>
__device__ __forceinline__ float pwl_eval(const PwlSmem& P, float x) {
    int i = 0;
#pragma unroll
    for (int s = NPAD / 2; s >= 1; s >>= 1) i += (P.bp[i + s - 1] < x) ? s : 0;
    const float2 sg = P.seg[i];
    return fmaf(sg.x, x, sg.y);
}

// 64-bit add into a shared-memory bin with the hardware's 32-bit atomics (a 64-bit shared atomicAdd compiles to a compare-and-swap
// spin loop: 32 lanes on one bin -- iteration 0, every message still 0 -- took ~100 us per iteration).  The low word's returned
// old value tells whether THIS add wrapped it; the high word gets the addend's high word plus that carry, which is 0 for nearly
// every small addend of either sign, so the second atomic is rare.  Exact and order-independent like the 64-bit add it replaces.
__device__ __forceinline__ void fx_add(long long* slot, long long x) {
    if (x == 0) return;
    unsigned int* w = reinterpret_cast<unsigned int*>(slot);
    const unsigned int lo = (unsigned int)x, hi = (unsigned int)((unsigned long long)x >> 32);
    const unsigned int old = atomicAdd(w, lo);
    const unsigned int h = hi + ((old + lo < old) ? 1u : 0u);
    if (h) atomicAdd(w + 1, h);
}
// ---- 1 -> h -> 1 Softplus MLP on a COMPACT domain as a cubic table --------------------------------
// The check-phase MLP of decoder_v2_4 (quantum/decoder_v2_4.py:257, `self.mlp(aggr_out[:, 0])`) is a
// smooth scalar function f(x) = b2 + sum_k w2_k softplus(w1_k x + b1_k) of ONE variable whose argument
// is a sum of tanh values minus one of them: |x| <= (max check degree - 1), a domain known from the
// graph (the read-out MLP's argument m is bounded by T * max|f|).  Each CTA tabulates it once per
// launch: N uniform intervals, per interval the cubic Hermite interpolant through (f, f') at both
// ends -- node values from the packed direct evaluation, node derivatives from 4th-order central
// differences.  The interpolation error is bounded by h^4 / 384 * max|d4f/dx4| <= h^4 / 384 * 0.125 *
// sum_k |w2_k| w1_k^4, evaluated from the weights in the prologue; if the bound exceeds the budget
// (1e-7 check phase, 4e-6 read-out) the kernel keeps the direct evaluation.  One evaluation is then
// ~12 instructions + one 16-byte shared load instead of h x (1.5 MUFU + ~7 FMA).
struct CubicTab {
    const float4* c;   // [N] (a0, a1, a2, a3): f(x_i + t h) ~= a0 + t (a1 + t (a2 + t a3)), t in [0, 1]
    float inv_h, off, umax;
};
__device__ __forceinline__ float cubic_tab_eval(const CubicTab& T, float x) {
    float u = fmaf(x, T.inv_h, T.off);
    u = fminf(fmaxf(u, 0.f), T.umax);
    const float v = (u - 0.5f) + 12582912.0f;                  // round-to-nearest of u - 0.5 == floor(u) (ties land on a node)
    const int i = __float_as_int(v) - 0x4B400000;
    const float t = u - (v - 12582912.0f);
    const float4 c = T.c[i];
    return fmaf(fmaf(fmaf(c.w, t, c.z), t, c.y), t, c.x);
}
// Interpolation-error bound of an n-interval table on [-R, R] from the RAW weights w1[h] | b1[h] | w2[h]
// (identical arithmetic in every thread -> a CTA-uniform decision).
__device__ __forceinline__ float cubic_tab_bound(const float* w, int h, float step) {
    float m4 = 0.f;
    for (int k = 0; k < h; ++k) {
        float a = __ldg(w + k);
        a *= a;
        m4 = fmaf(fabsf(__ldg(w + 2 * h + k)), a * a, m4);
    }
    const float s2 = step * step;
    return s2 * s2 * (0.125f / 384.0f) * m4;
}
// Build the table with the whole CTA (contains __syncthreads()).  W: the MLP staged (pre-scaled) in shared
// memory; F: n + 6 floats of shared scratch.  Returns this thread's max |f| over the nodes it touched.
// TWO_IN: W is a 2 -> h -> 1 MLP and the table is its section f(., x1v) at a fixed second input.
template <bool TWO_IN = false>
__device__ __forceinline__ float cubic_tab_build(const MlpSmem& W, int hp, float Rdom, int n, float4* dst, float* F,
                                                 int tid, int nthr, float x1v = 0.f) {
    const float step = 2.0f * Rdom / (float)n;
    for (int j0 = tid * 2; j0 < n + 5; j0 += nthr * 2) {          // nodes -2 .. n+2, two per thread per pass
        const float xa[2] = {-Rdom + step * (float)(j0 - 2), -Rdom + step * (float)(j0 - 1)};
        const float xb[2] = {x1v, x1v};
        float oa[2];
        if constexpr (TWO_IN) mlp_softplus_x2<2, true, 2>(W, hp, xa, xb, oa);
        else mlp_softplus_x2<2, false, 2>(W, hp, xa, xa, oa);
        F[j0] = oa[0];
        F[j0 + 1] = oa[1];
    }
    __syncthreads();
    float fm = 0.f;
    for (int i = tid; i < n; i += nthr) {
        const float a = F[i], b = F[i + 1], f0 = F[i + 2], f1 = F[i + 3], c = F[i + 4], d = F[i + 5];
        const float d0 = (8.f * (f1 - b) - (c - a)) * (1.f / 12.f);      // h f'(x_i), 4th-order central difference
        const float d1 = (8.f * (c - f0) - (d - b)) * (1.f / 12.f);
        dst[i] = make_float4(f0, d0, 3.f * (f1 - f0) - 2.f * d0 - d1, 2.f * (f0 - f1) + d0 + d1);
        fm = fmaxf(fm, fmaxf(fabsf(f0), fabsf(f1)));
    }
    __syncthreads();
    return fm;
}

// tanh(a/2): one per edge-iteration, so the full-accuracy libm version is affordable.
// (tanh.approx.f32 has ~5e-4 relative error: too coarse for the 1e-4 logit bar, SURVEY 9.)
__device__ __forceinline__ float tanh_half(float a) { return tanhf(0.5f * a); }

// P(flip) = sigmoid(-logit) = 1 / (1 + e^logit)
__device__ __forceinline__ float sigmoid_neg(float logit) { return 1.0f / (1.0f + expf(logit)); }

// tanh(a/2) = 1 - 2 / (1 + e^a) with ex2 + rcp (2 MUFU, 5 instructions): absolute error ~2e-7, used where
// the instruction count matters (streamed kernel); e^a = inf / 0 give exactly +1 / -1.
__device__ __forceinline__ float rcp_fast(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float tanh_half_fast(float a) {
    const float e = ex2_approx(a * kLog2e);
    return fmaf(-2.0f, rcp_fast(1.0f + e), 1.0f);
}

// ---- sum-product (BP) pieces (reference quantum/BP.py:103-117, classical/BP.py:101-116), written so
// that fp32 keeps the accuracy the fp64 reference has in the saturated regime, with MUFU-based
// evaluation (3 MUFU + ~15 FMA-type instructions each instead of four libm calls) ----
// 1 - e^{-u} for u >= 0, p = e^{-u} from ex2.approx: the series u (1 - u/2 + u^2/6 - u^3/24 + u^4/120 - u^5/720) below
// u = 0.25 (truncation <= 5e-8 relative), 1 - p above.  Subtraction turns p's error (up to 2^-22 relative) into a relative
// error of p / (1 - p) 2^-22 in 1 - p: 9.5 2^-22 at u = 0.1, 3.5 2^-22 at 0.25 (tests/test_sum_product_formula.py).
__device__ __forceinline__ float bp_one_minus_exp(float u, float p) {
    float ser = fmaf(u, -1.0f / 720.0f, 1.0f / 120.0f);
    ser = fmaf(-ser, u, 1.0f / 24.0f);
    ser = fmaf(-ser, u, 1.0f / 6.0f);
    ser = fmaf(-ser, u, 0.5f);
    ser = fmaf(-ser, u, 1.0f);
    return u < 0.25f ? u * ser : 1.0f - p;
}
// log|tanh(a/2)| after clamp(a, -10, 10), clamped below at log(eps1).  With q = e^{-|a|}:
//   |a| <  1.4 : ln2 * lg2((1 - q) / (1 + q)), 1 - q from bp_one_minus_exp   (value <= -0.5: lg2.approx is accurate; by
//                subtraction, 1 - q would carry q's absolute error ~2.4e-7, i.e. ~2.4e-7 / |a| in the value)
//   |a| >= 1.4 : -2 atanh(q) = -2 q (1 + q^2/3 + q^4/5 + q^6/7 + q^8/9)   (q <= 0.25; no cancellation
//                near saturation, where log|tanh| ~ -2q is tiny and feeds log(1 - prod) downstream)
// 2 atanh(q) = log((1 + q) / (1 - q)) = 2 q (1 + q^2/3 + q^4/5 + q^6/7 + q^8/9) for 0 <= q <= 0.25 (truncation <= 1e-7 relative)
__device__ __forceinline__ float bp_two_atanh_small(float q) {
    const float q2 = q * q;
    float ser = fmaf(q2, 1.0f / 9.0f, 1.0f / 7.0f);
    ser = fmaf(ser, q2, 0.2f);
    ser = fmaf(ser, q2, 1.0f / 3.0f);
    ser = fmaf(ser, q2, 1.0f);
    return 2.0f * q * ser;
}
template <bool CLAMP_IN = true>   // false: quantum/neural_BP.py:108 takes tanh(m/2) without the +-10 clamp
__device__ __forceinline__ float bp_log_abs_tanh_half(float a, float log_eps1) {
    const float aa = CLAMP_IN ? fminf(fabsf(a), 10.0f) : fabsf(a);
    const float q = ex2_approx(-aa * kLog2e);
    const float far = -bp_two_atanh_small(q);
    const float near = kLn2 * lg2_approx(bp_one_minus_exp(aa, q) * rcp_fast(1.0f + q));     // aa == 0 -> -inf
    return fmaxf(aa < 1.4f ? near : far, log_eps1);
}
// m = log((1+o)/(1-o)), o = sign * exp(ext) clamped to [-1+eps2, 1-eps2]; ext <= 0 (up to rounding).  With p = |o| = e^{-u}:
//   u <= 1.4 : ln2 (lg2(1 + p) - lg2(1 - p)), 1 - p from bp_one_minus_exp   (where the clamp can bind)
//   u >  1.4 : 2 atanh(p) as a series (p < 0.25: the clamp cannot bind; 1 + p and 1 - p would round p away below 2^-24,
//              and m, the next layer's message, would lose its digits)
__device__ __forceinline__ float bp_check_out(float ext, bool odd, float eps2) {
    const float u = fmaxf(-ext, 0.0f);
    const float p = ex2_approx(-u * kLog2e);
    const float one_minus = fmaxf(bp_one_minus_exp(u, p), eps2);
    const float near = kLn2 * (lg2_approx(1.0f + fminf(p, 1.0f - eps2)) - lg2_approx(one_minus));
    const float mag = u > 1.4f ? bp_two_atanh_small(p) : near;
    return odd ? -mag : mag;
}
// Derivatives of the two sum-product pieces above, for neural BP's training backward (gd_backward_nbp.cu).
// dm/dext of bp_check_out: m = log((1+o)/(1-o)), o = ±e^ext -> dm/dext = ±1 / sinh(-ext), with no 1 - o^2 to cancel.  0 where
// the clamp of |o| at 1 - eps2 binds, decided from ext as bp_check_out decides it: in fp32, o rounds to ±1 long before.
__device__ __forceinline__ float bp_dcheck_out(float ext, bool odd, float eps2) {
    const float u = fmaxf(-ext, 0.0f);
    if (bp_one_minus_exp(u, ex2_approx(-u * kLog2e)) < eps2) return 0.0f;
    const float r = 1.0f / sinhf(u);
    return odd ? -r : r;
}
// d/da log|tanh(a/2)| = 1 / sinh(a) (0 past |a| ~ 89, where sinh overflows); 0 where bp_log_abs_tanh_half<false>(a) returned
// its lower clamp log(eps1) (lv: that value)
__device__ __forceinline__ float bp_dlog_abs_tanh_half(float a, float lv, float log_eps1) {
    return lv > log_eps1 ? 1.0f / sinhf(a) : 0.0f;
}

// torch.nn.GRUCell(1, 1) (quantum/QGNNNI_ca.py:188,198; gate order r, z, n):
//   r = s(w_ir x + b_ir + w_hr h + b_hr), z = s(w_iz x + b_iz + w_hz h + b_hz),
//   n = tanh(w_in x + b_in + r (w_hn h + b_hn)),  h' = (1 - z) n + z h
// g = weight_ih[3] | weight_hh[3] | bias_ih[3] | bias_hh[3].  sigmoid / tanh via ex2 + rcp (abs. error ~2e-7).
__device__ __forceinline__ float sigmoid_fast(float a) { return rcp_fast(1.0f + ex2_approx(-a * kLog2e)); }
__device__ __forceinline__ float gru_cell(const float* g, float x, float h) {
    const float r = sigmoid_fast(fmaf(g[0], x, g[6]) + fmaf(g[3], h, g[9]));
    const float z = sigmoid_fast(fmaf(g[1], x, g[7]) + fmaf(g[4], h, g[10]));
    const float n = tanh_half_fast(2.0f * (fmaf(g[2], x, g[8]) + r * fmaf(g[5], h, g[11])));
    return fmaf(z, h - n, n);
}

}  // namespace gd
