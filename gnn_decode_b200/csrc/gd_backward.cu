// Backward of the fused decoder_v2_4 decoder (training, BASELINE config 4): gradient of a loss
// w.r.t. the 10h+3 MLP weights, given dL/dlogit [B, V].  Replaces autograd through the reference's
// T x 2 x ~12 eager ops (quantum/decoder_v2_4.py:280-292, loss.backward() at :335).
//
// Structure per tile of syndromes (edge arrays [E][tile] fp32 in shared memory -- or, for codes whose arrays do not fit
// there, in a per-CTA slab of the caller's workspace: the same kernel body, see WORK_GLOBAL), iterations in reverse,
// activations (m_it, a_it) re-read from the stash the training forward wrote:
//   * "sum over siblings minus self" is self-adjoint, so the gather-of-gradients is the same
//     deterministic segmented sum as the forward reduce;
//   * the per-edge MLP backward is the expensive part and is mapped DIFFERENTLY from the forward:
//     a warp takes one (syndrome, edge) item at a time and its LANES ARE HIDDEN UNITS (4 per
//     lane for h = 128).  Each lane keeps its units' weights and its weight-gradient accumulators
//     in registers for the whole kernel -- no atomics and no per-item cross-lane reduction for the
//     weight gradients; only the scalar input gradient dx needs one 5-step shuffle sum per item;
//   * weight gradients leave the kernel as per-warp partial vectors and are summed by a second
//     kernel in a fixed order in double precision: bit-reproducible ("deterministic two-stage
//     wgrad reduction"), ready for one NCCL all-reduce of 10h+3 floats.
#include "gd_common.cuh"
#include "gd_math.cuh"
#include "gd_options.cuh"
#include "gd_decode.cuh"
#include <stdlib.h>
#include <string.h>

namespace gd {

constexpr int kBwdThreads = 512;
constexpr int kUPL = 4;          // hidden units per lane (h <= 128)
constexpr int kItems = 4;        // items processed together per warp (ILP across the MUFU chains; the dx reduction assumes 4)

struct BwdParams {
    const float* x;           // [B, N]
    const float* stash;       // [(T+1)][2][E][B]
    const float* grad_logit;  // [B, V]
    const float* weights;     // packed raw weights
    const int* run_flag;      // NULL, or: run only if *run_flag != 0 (the stash header's old_count, gd_lean.cuh)
    float* partials;          // [grid * warps][np_pad]
    GraphTables tb;
    long long B;
    int T, V, C, E, N, hid;
    int tile, R, n_tiles, maxvc, np_pad;
    int off_tab, off_x, off_node, off_node2, off_dm, off_a, off_xin, off_x1, off_g, off_dx, off_mb, off_ab;
    // check-phase MLP through its cubic table and the table's ADJOINT (see decode_bwd_kernel)
    int ctab_n, off_ctab, off_w2s, off_bins, off_mbins;
    float ctab_R;
    // variable-phase MLP items are laid out in vlist order (edges of variables with degree >= 2 first); the
    // n_static = E - n_vact edges of degree-1 variables see ext == 0 in every iteration, so their upstream
    // gradients are summed over the iterations (off_gacc) and pushed through the MLP once per tile
    int n_vact, off_gacc;
    // WORK_GLOBAL: the per-tile work arrays (off_x .. off_gacc, byte offsets) live at slab + blockIdx.x * slab_floats
    float* slab;
    long long slab_floats;
};

constexpr int kPairs = kUPL / 2;
typedef unsigned long long u64;

__device__ __forceinline__ u64 mul2(u64 a, u64 b) {
    u64 d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ float rcp_approx(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ void cp_async4(float* dst_smem, const float* src_gmem) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(dst_smem)),
                 "l"(src_gmem)
                 : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ float sign_one(float h) {   // copysign(1, h)
    return __uint_as_float((__float_as_uint(h) & 0x80000000u) | 0x3f800000u);
}

// This lane's kUPL hidden units of one MLP as kPairs packed (f32x2) pairs; w1a/w1b/b1 pre-scaled to
// base 2 like the forward, w2 in natural units.
struct LaneMlp {
    u64 w1a[kPairs], w1b[kPairs], b1[kPairs], w2[kPairs];
};
struct LaneAcc {
    u64 w1a[kPairs], w1b[kPairs], b1[kPairs], w2[kPairs];
    float b2;
};

__device__ __forceinline__ void load_lane_mlp(LaneMlp& L, const float* w, int h, bool two_in, int lane) {
#pragma unroll
    for (int q = 0; q < kPairs; ++q) {
        float a[2], b[2], c[2], d[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int k = lane * kUPL + q * 2 + u;
            const bool in = k < h;
            a[u] = in ? w[two_in ? 2 * k : k] * kLog2e : 0.f;
            d[u] = (in && two_in) ? w[2 * k + 1] * kLog2e : 0.f;
            b[u] = in ? w[(two_in ? 2 : 1) * h + k] * kLog2e : 0.f;
            c[u] = in ? w[(two_in ? 3 : 2) * h + k] : 0.f;
        }
        L.w1a[q] = pack2(a[0], a[1]); L.w1b[q] = pack2(d[0], d[1]);
        L.b1[q] = pack2(b[0], b[1]); L.w2[q] = pack2(c[0], c[1]);
    }
}
__device__ __forceinline__ void zero_acc(LaneAcc& A) {
#pragma unroll
    for (int q = 0; q < kPairs; ++q) A.w1a[q] = A.w1b[q] = A.b1[q] = A.w2[q] = 0ull;
    A.b2 = 0.f;
}

// One MLP backward over all items of the tile.  xin/g/dx are [E][tile] shared arrays (item index
// i = e*tile + s is linear).  For the two-input MLP the second input is prior[var(e)] from the x slab.
// Per hidden unit: h' -> t = 2^-|h'| -> r = 1/(1+t), l = lg2(1+t) (3 MUFU); softplus/ln2 = max(h',0)+l;
// sigmoid(h) = 1/2 + sign(h)(r - 1/2); dh = g w2 sigmoid.  All FMA-type work is packed f32x2 over a
// pair of hidden units (half the issue slots), so the loop is bound by the MUFU pipe.
template <bool TWO_IN>
__device__ __forceinline__ void mlp_backward_items(const LaneMlp& L, LaneAcc& A, const float* xin, const float* xin1,
                                                   const float* g, float* dx, int n_items, int warp, int n_warps,
                                                   int lane) {
    const u64 one2 = pack2(1.0f, 1.0f), half2 = pack2(0.5f, 0.5f), mhalf2 = pack2(-0.5f, -0.5f);
    for (int i0 = warp * kItems; i0 < n_items; i0 += n_warps * kItems) {
        u64 xx[kItems], yy[kItems], gg[kItems], dx2[kItems];
#pragma unroll
        for (int j = 0; j < kItems; ++j) {
            const int i = i0 + j < n_items ? i0 + j : n_items - 1;
            const float x0 = xin[i];
            const float gv = i0 + j < n_items ? g[i] : 0.f;
            const float x1 = TWO_IN ? xin1[i] : 0.f;
            xx[j] = pack2(x0, x0); yy[j] = pack2(x1, x1); gg[j] = pack2(gv, gv);
            dx2[j] = 0ull;
            A.b2 += gv;
        }
#pragma unroll
        for (int q = 0; q < kPairs; ++q) {
#pragma unroll
            for (int j = 0; j < kItems; ++j) {
                u64 h2 = fma2(L.w1a[q], xx[j], L.b1[q]);
                if (TWO_IN) h2 = fma2(L.w1b[q], yy[j], h2);
                float hl, hh;
                unpack2(h2, hl, hh);
                const float tl = ex2_approx(-fabsf(hl)), th = ex2_approx(-fabsf(hh));
                float ol, oh;
                unpack2(add2(pack2(tl, th), one2), ol, oh);
                const u64 r2 = pack2(rcp_approx(ol), rcp_approx(oh));
                const u64 l2 = pack2(lg2_approx(ol), lg2_approx(oh));
                const u64 sp2 = add2(l2, pack2(fmaxf(hl, 0.f), fmaxf(hh, 0.f)));        // softplus / ln2
                const u64 sig2 = fma2(pack2(sign_one(hl), sign_one(hh)), add2(r2, mhalf2), half2);
                const u64 dh2 = mul2(mul2(gg[j], L.w2[q]), sig2);                        // dL/d(pre-activation)
                A.w2[q] = fma2(gg[j], sp2, A.w2[q]);                                     // x ln2 when written out
                A.w1a[q] = fma2(dh2, xx[j], A.w1a[q]);
                if (TWO_IN) A.w1b[q] = fma2(dh2, yy[j], A.w1b[q]);
                A.b1[q] = add2(A.b1[q], dh2);
                dx2[j] = fma2(dh2, L.w1a[q], dx2[j]);                                    // / log2e when written out
            }
        }
        // transposed warp reduction of the kItems (= 4) per-lane partial dx: 6 shuffles instead of 20;
        // lanes 0, 8, 16, 24 end up holding the sums of items 0, 1, 2, 3
        float v[kItems];
#pragma unroll
        for (int j = 0; j < kItems; ++j) {
            float lo, hi;
            unpack2(dx2[j], lo, hi);
            v[j] = lo + hi;
        }
        const bool b4 = lane & 16, b3 = lane & 8;
        const float ra = __shfl_xor_sync(0xffffffffu, b4 ? v[0] : v[2], 16);
        const float rb = __shfl_xor_sync(0xffffffffu, b4 ? v[1] : v[3], 16);
        const float k0 = (b4 ? v[2] : v[0]) + ra, k1 = (b4 ? v[3] : v[1]) + rb;
        const float rc = __shfl_xor_sync(0xffffffffu, b3 ? k0 : k1, 8);
        float k = (b3 ? k1 : k0) + rc;
        k += __shfl_xor_sync(0xffffffffu, k, 4);
        k += __shfl_xor_sync(0xffffffffu, k, 2);
        k += __shfl_xor_sync(0xffffffffu, k, 1);
        const int item = i0 + (b4 ? 2 : 0) + (b3 ? 1 : 0);
        if ((lane & 7) == 0 && item < n_items) dx[item] = k * kLn2;        // 1/log2e == ln2
    }
}

__device__ __forceinline__ void store_acc(float* dst, const LaneAcc& A, int h, bool two_in, int lane) {
    // packed order of one MLP: W1 [h, k_in] row-major | b1 [h] | W2 [h] | b2
#pragma unroll
    for (int q = 0; q < kPairs; ++q) {
        float a[2], d[2], b[2], c[2];
        unpack2(A.w1a[q], a[0], a[1]); unpack2(A.w1b[q], d[0], d[1]);
        unpack2(A.b1[q], b[0], b[1]); unpack2(A.w2[q], c[0], c[1]);
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int k = lane * kUPL + q * 2 + u;
            if (k < h) {
                if (two_in) { dst[2 * k] = a[u]; dst[2 * k + 1] = d[u]; }
                else dst[k] = a[u];
                dst[(two_in ? 2 : 1) * h + k] = b[u];
                dst[(two_in ? 3 : 2) * h + k] = c[u] * kLn2;
            }
        }
    }
    if (lane == 0) dst[(two_in ? 4 : 3) * h] = A.b2;
}

// WORK_GLOBAL = false: every per-tile array in shared memory (tile limited by its size).  WORK_GLOBAL = true: the per-tile work
// arrays (xs .. GA) in this CTA's slab of the workspace, for codes too large for the first form (HGP [[1600,64]]: ~390 KB per
// syndrome); the graph tables, the check table and its adjoint bins stay in shared memory, the bins as 64-bit integers (below).
template <bool WORK_GLOBAL>
__global__ void __launch_bounds__(kBwdThreads, 1) decode_bwd_kernel(const BwdParams p) {
    extern __shared__ __align__(128) unsigned char smem[];
    pdl_enter();
    if (p.run_flag && *p.run_flag == 0) return;               // the table forward wrote this step's stash: gd_lean.cu's backward runs
    const int tile = p.tile, R = p.R, E = p.E, V = p.V, C = p.C, N = p.N, h = p.hid, T = p.T;
    const int tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31, warp = tid >> 5, n_warps = nthr >> 5;
    const int s = tid % tile, r = tid / tile;
    const bool ew = r < R;                      // threads beyond R*tile only take part in the MLP phases
    unsigned char* const wk = WORK_GLOBAL ? reinterpret_cast<unsigned char*>(p.slab + (size_t)blockIdx.x * p.slab_floats) : smem;
    float* xs = reinterpret_cast<float*>(wk + p.off_x);
    float* node = reinterpret_cast<float*>(wk + p.off_node);
    float* DM = reinterpret_cast<float*>(wk + p.off_dm);
    float* A_ = reinterpret_cast<float*>(wk + p.off_a);
    float* XI = reinterpret_cast<float*>(wk + p.off_xin);
    float* X1 = reinterpret_cast<float*>(wk + p.off_x1);
    float* MB = reinterpret_cast<float*>(wk + p.off_mb);
    float* AB = reinterpret_cast<float*>(wk + p.off_ab);
    float* node2 = reinterpret_cast<float*>(wk + p.off_node2);
    float* G_ = reinterpret_cast<float*>(wk + p.off_g);
    float* DX = reinterpret_cast<float*>(wk + p.off_dx);
    uint16_t* tab = reinterpret_cast<uint16_t*>(smem + p.off_tab);
    uint16_t* edge_var = tab;
    uint16_t* edge_chk = edge_var + E;
    uint16_t* var_ptr = edge_chk + E;
    uint16_t* var_edges = var_ptr + (V + 1);
    uint16_t* chk_ptr = var_edges + E;
    uint16_t* chk_edges = chk_ptr + (C + 1);
    uint16_t* vpos = chk_edges + E;                      // position of edge e in vlist order
    for (int i = tid; i < E; i += nthr) vpos[p.tb.vlist[i]] = (uint16_t)i;
    const int n_act = p.n_vact, n_static = E - n_act;
    float* GA = reinterpret_cast<float*>(wk + p.off_gacc);
    for (int i = tid; i < E; i += nthr) {
        edge_var[i] = (uint16_t)p.tb.edge_var[i];
        edge_chk[i] = (uint16_t)p.tb.edge_chk[i];
        var_edges[i] = (uint16_t)p.tb.var_edges[i];
        chk_edges[i] = (uint16_t)p.tb.chk_edges[i];
    }
    for (int i = tid; i <= V; i += nthr) var_ptr[i] = (uint16_t)p.tb.var_ptr[i];
    for (int i = tid; i <= C; i += nthr) chk_ptr[i] = (uint16_t)p.tb.chk_ptr[i];

    LaneAcc acc1, acc2, acc3;
    zero_acc(acc1); zero_acc(acc2); zero_acc(acc3);
    const float* w1p = p.weights;
    const float* w2p = w1p + 4 * h + 1;
    const float* w3p = w2p + 3 * h + 1;
    const int n_items = E * tile;
    const size_t EB_ = (size_t)E * p.B;
    // ---- the 1 -> h -> 1 check-phase MLP (decoder_v2_4.py:257) without per-unit work ----
    // Forward it is a cubic table f on |x| <= d_c - 1 (gd_math.cuh CubicTab, DESIGN.md 4.1).  Backward:
    //   dL/dx      = g f'(x)                      -- the derivative of the table's cubic piece;
    //   dL/dtheta  = sum_i g_i phi_theta(x_i)     -- phi_theta = df/dtheta is again a smooth scalar function of x, so
    //                its Hermite interpolant gives  sum_j [ A_j phi(x_j) + D_j h phi'(x_j) ]  with the ADJOINT bins
    //                A_j = sum_i g_i h00/h01(t_i), D_j = sum_i g_i h10/h11(t_i): four scatter-adds per item now, and one
    //                pass over (nodes x hidden units) at the very end, instead of h x 3 MUFU per item.
    // The bins are accumulated as FIXED-POINT integers (scale from the phase's max |g|: integer adds commute, so shared-memory
    // atomics stay bit-reproducible) and flushed into double master bins after every phase.  The scale keeps
    // n_items * max|g| below 2^30 in 32-bit bins; with WORK_GLOBAL, n_items = E * tile is large (HGP: ~3e5) and 32 bits would
    // leave ~3e3 units for the largest item, so that variant takes 64-bit bins and 2^62: every item keeps the float
    // product's own precision.
    CubicTab ctab{};
    bool use_ctab = false;
    unsigned int* bins = reinterpret_cast<unsigned int*>(smem + p.off_bins);      // [2][n+1]
    unsigned long long* bins64 = reinterpret_cast<unsigned long long*>(smem + p.off_bins);
    double* mbins = reinterpret_cast<double*>(smem + p.off_mbins);                // [2][n+1]
    unsigned int* gmax_bits = WORK_GLOBAL ? reinterpret_cast<unsigned int*>(bins64 + 2 * (p.ctab_n + 1)) : bins + 2 * (p.ctab_n + 1);
    if (p.ctab_n > 0 && E * tile >= p.ctab_n + 8) {
        float* w2s = reinterpret_cast<float*>(smem + p.off_w2s);
        const int hp = (h + 7) / 8 * 8;
        for (int k = tid; k < hp; k += nthr) {
            const bool in = k < h;
            w2s[k] = in ? w2p[k] * kLog2e : 0.f;
            w2s[hp + k] = 0.f;
            w2s[2 * hp + k] = in ? w2p[h + k] * kLog2e : 0.f;
            w2s[3 * hp + k] = in ? w2p[2 * h + k] * kLn2 : 0.f;
        }
        __syncthreads();
        const float step = 2.0f * p.ctab_R / (float)p.ctab_n;
        use_ctab = cubic_tab_bound(w2p, h, step) <= 1e-7f;
        if (use_ctab) {
            const MlpSmem W2s{w2s, w2s + hp, w2s + 2 * hp, w2s + 3 * hp, w2p[3 * h]};
            float4* cdst = reinterpret_cast<float4*>(smem + p.off_ctab);
            cubic_tab_build(W2s, hp, p.ctab_R, p.ctab_n, cdst, DM, tid, nthr);    // DM is idle scratch here
            ctab = CubicTab{cdst, 1.0f / step, p.ctab_R / step, (float)p.ctab_n - 0.001f};
            for (int j = tid; j < 2 * (p.ctab_n + 1); j += nthr) {
                if constexpr (WORK_GLOBAL) bins64[j] = 0ull;
                else bins[j] = 0u;
                mbins[j] = 0.0;
            }
            if (tid == 0) *gmax_bits = 0u;
        }
    }
    __syncthreads();

    auto seg_sum = [&](const uint16_t* ptr, const uint16_t* ids, int n_nodes, const float* src, float* dstn) {
        if (ew)
            for (int n = r; n < n_nodes; n += R) {
                float a = 0.f;
                for (int i = ptr[n]; i < ptr[n + 1]; ++i) a += src[ids[i] * tile + s];
                dstn[n * tile + s] = a;
            }
    };
    // asynchronous prefetch of one iteration's stash (a_it -> AB, m_it -> MB) by the thread that will
    // consume the same elements; latency is hidden behind the MLP phases
    auto prefetch_stash = [&](int it, long long s0, bool valid) {
        if (ew && valid && it >= 0) {
            const float* st_m = p.stash + (size_t)it * 2 * EB_ + s0 + s;
            const float* st_a = st_m + EB_;
            for (int e = r; e < E; e += R) {
                if constexpr (WORK_GLOBAL) {        // (the same thread reads them back, behind the same barriers)
                    MB[e * tile + s] = __ldcs(st_m + (size_t)e * p.B);
                    AB[e * tile + s] = __ldcs(st_a + (size_t)e * p.B);
                } else {
                    cp_async4(MB + e * tile + s, st_m + (size_t)e * p.B);
                    cp_async4(AB + e * tile + s, st_a + (size_t)e * p.B);
                }
            }
        }
        cp_async_commit();
    };

    for (int tix = blockIdx.x; tix < p.n_tiles; tix += gridDim.x) {
        const long long s0 = (long long)tix * tile;
        const int nvalid = (int)min((long long)tile, p.B - s0);
        const bool valid = s < nvalid;
        for (int i = tid; i < tile * N; i += nthr) xs[i] = i < nvalid * N ? __ldg(p.x + s0 * N + i) : 0.f;
        if (ew && !valid)
            for (int e = r; e < E; e += R) MB[e * tile + s] = AB[e * tile + s] = 0.f;   // padded syndromes stay 0
        prefetch_stash(T - 1, s0, valid);
        // ---- read-out backward: logit[v] = sum_{e in v} mlp3(m_T[e]) + prior[v] ----
        if (ew)
            for (int e = r; e < E; e += R) {
                const int at = e * tile + s;
                XI[at] = valid ? __ldg(p.stash + (size_t)T * 2 * EB_ + (size_t)e * p.B + s0 + s) : 0.f;
                G_[at] = valid ? __ldg(p.grad_logit + (s0 + s) * V + edge_var[e]) : 0.f;
            }
        __syncthreads();
        if (ew)
            for (int e = r; e < E; e += R) X1[vpos[e] * tile + s] = xs[s * N + edge_var[e]];   // prior of the edge's variable (vlist order)
        for (int i = tid; i < n_static * tile; i += nthr) GA[i] = 0.f;
        {
            LaneMlp L;
            load_lane_mlp(L, w3p, h, false, lane);
            mlp_backward_items<false>(L, acc3, XI, XI, G_, DM, n_items, warp, n_warps, lane);
        }
        cp_async_wait_all();
        if (ew)
            for (int e = r; e < E; e += R) A_[e * tile + s] = tanh_half(AB[e * tile + s]);   // t of iteration T-1
        __syncthreads();
        for (int it = T - 1; it >= 0; --it) {
            // entry: A_ = t_it = tanh(a_it/2), MB = m_it, DM = dL/dm_{it+1}
            seg_sum(chk_ptr, chk_edges, C, A_, node);             // Sc(t)
            seg_sum(var_ptr, var_edges, V, MB, node2);            // Sv(m_it)
            __syncthreads();
            // m_{it+1} = mlp2(ext_c) * sign + m_it :  dg = dm' * sign, ext_c = Sc[chk] - t
            if (ew)
                for (int e = r; e < E; e += R) {
                    const int at = e * tile + s, c = edge_chk[e];
                    XI[at] = node[c * tile + s] - A_[at];
                    G_[at] = DM[at] * xs[s * N + V + c];
                }
            __syncthreads();
            if (use_ctab) {
                const int nb = p.ctab_n + 1;
                float gm = 0.f;
                for (int i = tid; i < n_items; i += nthr) gm = fmaxf(gm, fabsf(G_[i]));
                for (int o = 16; o > 0; o >>= 1) gm = fmaxf(gm, __shfl_xor_sync(0xffffffffu, gm, o));
                if (lane == 0) atomicMax(gmax_bits, __float_as_uint(gm));
                __syncthreads();
                const float gmax = __uint_as_float(*gmax_bits);
                // |sum over a bin| <= n_items * gmax: keep it below 2^30 (32-bit bins) / 2^62 (64-bit bins)
                const float scale = gmax > 0.f ? (WORK_GLOBAL ? 4611686018427387904.0f : 1073741824.0f) / (gmax * (float)n_items) : 0.f;
                for (int i = tid; i < n_items; i += nthr) {
                    const float xv = XI[i], gv = G_[i];
                    float u = fmaf(xv, ctab.inv_h, ctab.off);
                    u = fminf(fmaxf(u, 0.f), ctab.umax);
                    const float vv = (u - 0.5f) + 12582912.0f;
                    const int j = __float_as_int(vv) - 0x4B400000;
                    const float t = u - (vv - 12582912.0f);
                    const float4 c = ctab.c[j];
                    DX[i] = gv * fmaf(fmaf(3.0f * c.w, t, 2.0f * c.z), t, c.y) * ctab.inv_h;
                    if (gv != 0.f) {
                        const float t2 = t * t, t3 = t2 * t, gs = gv * scale;
                        const float h01 = 3.0f * t2 - 2.0f * t3;
                        if constexpr (WORK_GLOBAL) {
                            atomicAdd(bins64 + j, (unsigned long long)__float2ll_rn(gs * (1.0f - h01)));
                            atomicAdd(bins64 + j + 1, (unsigned long long)__float2ll_rn(gs * h01));
                            atomicAdd(bins64 + nb + j, (unsigned long long)__float2ll_rn(gs * (t3 - 2.0f * t2 + t)));
                            atomicAdd(bins64 + nb + j + 1, (unsigned long long)__float2ll_rn(gs * (t3 - t2)));
                        } else {
                            atomicAdd(bins + j, (unsigned int)__float2int_rn(gs * (1.0f - h01)));
                            atomicAdd(bins + j + 1, (unsigned int)__float2int_rn(gs * h01));
                            atomicAdd(bins + nb + j, (unsigned int)__float2int_rn(gs * (t3 - 2.0f * t2 + t)));
                            atomicAdd(bins + nb + j + 1, (unsigned int)__float2int_rn(gs * (t3 - t2)));
                        }
                    }
                }
                __syncthreads();
                if (scale > 0.f) {
                    const double inv = 1.0 / (double)scale;
                    for (int j = tid; j < 2 * nb; j += nthr) {
                        if constexpr (WORK_GLOBAL) {
                            mbins[j] += (double)(long long)bins64[j] * inv;
                            bins64[j] = 0ull;
                        } else {
                            mbins[j] += (double)(int)bins[j] * inv;
                            bins[j] = 0u;
                        }
                    }
                }
                if (tid == 0) *gmax_bits = 0u;
            } else {
                LaneMlp L;
                load_lane_mlp(L, w2p, h, false, lane);
                mlp_backward_items<false>(L, acc2, XI, XI, G_, DX, n_items, warp, n_warps, lane);
            }
            __syncthreads();
            seg_sum(chk_ptr, chk_edges, C, DX, node);             // gather of gradients over the check
            __syncthreads();
            // dt = S[chk] - dext_c ; da = dt (1 - t^2) / 2 ; ext_v = Sv[var] - m_it
            if (ew)
                for (int e = r; e < E; e += R) {
                    const int at = e * tile + s;
                    const float t = A_[at];
                    const float dt = node[edge_chk[e] * tile + s] - DX[at];
                    const float gq = dt * (1.0f - t * t) * 0.5f;
                    const int pos = vpos[e];
                    if (pos < n_act) {
                        G_[pos * tile + s] = gq;
                        XI[pos * tile + s] = node2[edge_var[e] * tile + s] - MB[at];
                    } else {
                        GA[(pos - n_act) * tile + s] += gq;      // degree-1 variable: ext == 0, same input every iteration
                    }
                }
            prefetch_stash(it - 1, s0, valid);                    // MB / AB are free now
            __syncthreads();
            {
                LaneMlp L;
                load_lane_mlp(L, w1p, h, true, lane);
                mlp_backward_items<true>(L, acc1, XI, X1, G_, DX, n_act * tile, warp, n_warps, lane);
            }
            __syncthreads();
            // gather of gradients over the variable (DX is in vlist order; a degree-1 variable has no sibling: 0)
            if (ew)
                for (int n = r; n < V; n += R) {
                    float a = 0.f;
                    for (int i = var_ptr[n]; i < var_ptr[n + 1]; ++i) {
                        const int pos = vpos[var_edges[i]];
                        a += pos < n_act ? DX[pos * tile + s] : 0.f;
                    }
                    node[n * tile + s] = a;
                }
            __syncthreads();
            cp_async_wait_all();
            if (ew)
                for (int e = r; e < E; e += R) {
                    const int at = e * tile + s, pos = vpos[e];
                    DM[at] += node[edge_var[e] * tile + s] - (pos < n_act ? DX[pos * tile + s] : 0.f);
                    A_[at] = tanh_half(AB[at]);                   // t of the next (earlier) iteration
                }
            __syncthreads();
        }
        if (n_static > 0) {
            // the degree-1 variables' edges: one MLP backward with the iteration-summed gradient, input (0, prior)
            for (int i = tid; i < n_static * tile; i += nthr) XI[i] = 0.f;
            __syncthreads();
            LaneMlp L;
            load_lane_mlp(L, w1p, h, true, lane);
            mlp_backward_items<true>(L, acc1, XI, X1 + n_act * tile, GA, DX, n_static * tile, warp, n_warps, lane);
            __syncthreads();
        }
    }
    // ---- per-warp partial weight gradients, packed order ----
    float* dst = p.partials + ((size_t)blockIdx.x * n_warps + warp) * p.np_pad;
    store_acc(dst, acc1, h, true, lane);
    store_acc(dst + 4 * h + 1, acc2, h, false, lane);
    store_acc(dst + 7 * h + 2, acc3, h, false, lane);
    if (use_ctab) {
        // weight gradients of the check-phase MLP from the adjoint bins: one pass over (nodes x hidden units)
        __syncthreads();
        float* d0 = p.partials + (size_t)blockIdx.x * n_warps * p.np_pad + 4 * h + 1;     // warp 0's row, MLP 2
        const int nb = p.ctab_n + 1;
        const float step = 2.0f * p.ctab_R / (float)p.ctab_n;
        for (int k = tid; k < h; k += nthr) {
            const float w1 = w2p[k], b1 = w2p[h + k], w2 = w2p[2 * h + k];
            double gw1 = 0.0, gb1 = 0.0, gw2 = 0.0;
            for (int j = 0; j < nb; ++j) {
                const float xj = -p.ctab_R + step * (float)j;
                const float z = fmaf(w1, xj, b1);
                const float e = expf(-fabsf(z));
                const float sp = fmaxf(z, 0.f) + log1pf(e);
                const float sg = (z >= 0.f ? 1.0f : e) / (1.0f + e);
                const float dsg = sg * (1.0f - sg);
                const double A = mbins[j], D = mbins[nb + j] * (double)step;
                gw2 += A * (double)sp + D * (double)(sg * w1);
                gb1 += A * (double)(w2 * sg) + D * (double)(w2 * dsg * w1);
                gw1 += A * (double)(w2 * sg * xj) + D * (double)(w2 * (dsg * w1 * xj + sg));
            }
            d0[k] += (float)gw1;
            d0[h + k] += (float)gb1;
            d0[2 * h + k] += (float)gw2;
        }
        if (tid == 0) {
            double gb2 = 0.0;
            for (int j = 0; j < nb; ++j) gb2 += mbins[j];
            d0[3 * h] += (float)gb2;
        }
    }
}

// stage 2: fixed-order sum over the per-warp partials (double accumulation) -> grad[n_params]
__global__ void reduce_partials_kernel(const float* __restrict__ partials, int n_rows, int np_pad, int n_params,
                                       float* __restrict__ grad, int accumulate, const int* run_flag) {
    pdl_enter();
    if (run_flag && *run_flag == 0) return;                   // the table backward (gd_lean.cu) produced this step's gradient
    const int pidx = blockIdx.x * blockDim.x + threadIdx.x;
    if (pidx >= n_params) return;
    double a = 0.0;
    for (int rw = 0; rw < n_rows; ++rw) a += (double)partials[(size_t)rw * np_pad + pidx];
    grad[pidx] = accumulate ? grad[pidx] + (float)a : (float)a;
}

static int align_up_b(int x, int a) { return (x + a - 1) / a * a; }

struct BwdPlan {
    BwdParams p;
    int threads, grid, smem, n_rows;
    bool work_global;        // decode_bwd_kernel<true>: the work arrays in a slab of grid * p.slab_floats workspace floats
};

// The shared-memory form when at least 4 syndromes' work arrays fit there (and GD_FORCE_STREAMED is not set), the
// global-memory form otherwise.
static int plan_bwd(const gd_graph* g, const gd_model* m, int64_t B, BwdPlan* out) {
    BwdParams& p = out->p;
    memset(&p, 0, sizeof(p));
    const int V = g->V, C = g->C, N = g->N, E = (int)g->E;
    const int maxvc = V > C ? V : C;
    p.B = B; p.T = m->iters; p.V = V; p.C = C; p.E = E; p.N = N; p.hid = m->hidden; p.maxvc = maxvc;
    p.tb = g->t;
    p.np_pad = align_up_b((int)gd_weights_size(m), 32);
    if (g->E >= 65536) {
        set_error("gd_decode_bwd: E=%lld edges; the backward's graph tables hold 16-bit edge ids (E < 65536)", (long long)g->E);
        return GD_ERR_UNSUPPORTED;
    }
    const int64_t per_syn = ((int64_t)N + 2LL * maxvc + 8LL * E + (E - (opt_on(OPT_NO_VSKIP) ? E : g->n_vact))) * 4;
    const int tab_bytes = (5 * E + V + C + 2) * 2;
    // the form is decided before the layout: the global-memory form's bins are 64-bit
    int64_t tmax = 0;
    bool work_global = opt_on(OPT_FORCE_STREAMED);
    for (int pass = 0; pass < 2; ++pass) {
        int fixed = align_up_b(tab_bytes, 128);
        p.n_vact = opt_on(OPT_NO_VSKIP) ? E : g->n_vact;
        if (!opt_on(OPT_NO_CTAB)) {
            p.ctab_n = kCtabN;
            p.ctab_R = (float)(g->max_chk_deg > 1 ? g->max_chk_deg - 1 : 1);
            const int hp = (m->hidden + 7) / 8 * 8;
            p.off_ctab = fixed; fixed += p.ctab_n * 16;
            p.off_w2s = fixed; fixed += 4 * hp * 4;
            p.off_mbins = fixed; fixed += 2 * (p.ctab_n + 1) * 8;
            p.off_bins = fixed; fixed += work_global ? 2 * (p.ctab_n + 1) * 8 + 16 : (2 * (p.ctab_n + 1) + 4) * 4;
            fixed = align_up_b(fixed, 128);
        }
        out->smem = fixed;
        tmax = (g->max_smem_optin - fixed) / per_syn;
        if (work_global) break;
        if (tmax >= 4) break;
        work_global = true;
    }
    if (work_global && out->smem > g->max_smem_optin) {
        set_error("gd_decode_bwd: the graph tables (%d bytes) do not fit shared memory", out->smem);
        return GD_ERR_UNSUPPORTED;
    }
    out->work_global = work_global;
    // tile: multiple of 4 dividing the work evenly over the SMs (same criterion as the forward); the global-memory form is not
    // limited by shared memory and takes the larger tile on a tie (longer contiguous rows)
    int tile = 4;
    double best = -1.0;
    for (int t = 4; (work_global || t <= tmax) && t <= 128; t += 4) {
        const int64_t n_t = (B + t - 1) / t;
        const int64_t rounds = (n_t + g->sm_count - 1) / g->sm_count;
        const double eff = (double)B / ((double)rounds * g->sm_count * t);
        if (eff > best + 1e-9 || (work_global && eff > best - 1e-9)) { best = eff; tile = t; }
    }
    p.tile = tile;
    p.R = kBwdThreads / tile;
    if (p.R > E) p.R = E;
    if (p.R < 1) p.R = 1;
    int o = 0;
    p.off_tab = o; o = work_global ? 0 : out->smem;
    p.off_x = o; o += tile * N * 4; o = align_up_b(o, 16);
    p.off_node = o; o += maxvc * tile * 4;
    p.off_node2 = o; o += maxvc * tile * 4;
    p.off_dm = o; o += E * tile * 4;
    p.off_a = o; o += E * tile * 4;
    p.off_xin = o; o += E * tile * 4;
    p.off_x1 = o; o += E * tile * 4;
    p.off_g = o; o += E * tile * 4;
    p.off_dx = o; o += E * tile * 4;
    p.off_mb = o; o += E * tile * 4;
    p.off_ab = o; o += E * tile * 4;
    p.off_gacc = o; o += (E - p.n_vact) * tile * 4;
    if (work_global) p.slab_floats = align_up_b(o, 16) / 4;
    else out->smem = o;
    out->threads = kBwdThreads;
    p.n_tiles = (int)((B + tile - 1) / tile);
    out->grid = p.n_tiles < g->sm_count ? p.n_tiles : g->sm_count;
    out->n_rows = out->grid * (kBwdThreads / 32);
    return GD_OK;
}

// workspace: per-warp partials | the table backward's adjoint bins (gd_lean.cu) | the global-memory form's slab
static int64_t bwd_slab_offset(const gd_graph* g, const gd_model* m, const BwdPlan& pl) {
    return ((int64_t)pl.n_rows * pl.p.np_pad + lean_bwd_bins_floats(g, m) + 4 + 3) & ~(int64_t)3;
}

}  // namespace gd

extern "C" int64_t gd_bwd_workspace_floats(const gd_graph* g, const gd_model* model, int64_t B) {
    if (g && gd_model_valid(model) && model->program == GD_PROG_CGNNI && B > 0) return gd::light_bwd_workspace_floats(g, model, B);
    if (!g || !gd_model_valid(model) || model->program != GD_PROG_V2_4 || model->hidden > 32 * gd::kUPL || B <= 0) {
        gd::set_error("gd_bwd_workspace_floats: unsupported model (need GD_PROG_V2_4 with hidden <= %d, or GD_PROG_CGNNI)",
                      32 * gd::kUPL);
        return -1;
    }
    gd::BwdPlan pl;
    if (gd::plan_bwd(g, model, B, &pl) != GD_OK) return -1;
    // per-warp partial gradient vectors of the edge-owner backward, then the adjoint bins of the table backward (gd_lean.cu),
    // then the per-CTA work slabs of the global-memory form
    if (pl.work_global) return gd::bwd_slab_offset(g, model, pl) + (int64_t)pl.grid * pl.p.slab_floats;
    return (int64_t)pl.n_rows * pl.p.np_pad + gd::lean_bwd_bins_floats(g, model) + 4;
}

extern "C" int gd_decode_bwd(const gd_graph* g, const gd_model* model, const float* weights_dev, const float* x_dev,
                             const float* stash_dev, const float* grad_logit_dev, float* grad_weights_dev,
                             float* workspace_dev, int32_t accumulate, int64_t B, void* stream) {
    GD_CHECK_ARG(g != nullptr, "gd_decode_bwd: graph is NULL");
    GD_CHECK_ARG(gd_model_valid(model) && (model->program == GD_PROG_V2_4 || model->program == GD_PROG_CGNNI),
                 "gd_decode_bwd: only GD_PROG_V2_4 and GD_PROG_CGNNI have a backward kernel");
    GD_CHECK_ARG(model->hidden <= 32 * gd::kUPL, "gd_decode_bwd: hidden=%d > %d unsupported", model->hidden, 32 * gd::kUPL);
    GD_CHECK_ARG(B >= 0, "gd_decode_bwd: negative B");
    GD_CHECK_ARG(grad_weights_dev != nullptr, "gd_decode_bwd: grad_weights is NULL");
    const int n_params = (int)gd_weights_size(model);
    cudaStream_t st = (cudaStream_t)stream;
    if (B == 0) {
        if (!accumulate) GD_CUDA(cudaMemsetAsync(grad_weights_dev, 0, sizeof(float) * n_params, st));
        return GD_OK;
    }
    GD_CHECK_ARG(weights_dev && x_dev && stash_dev && grad_logit_dev && workspace_dev, "gd_decode_bwd: NULL buffer");
    gd::DeviceGuard dg(g->device);
    GD_CUDA(dg.status());
    gd::Route r;
    int rc = gd::route_decode(g, model, B, gd::Use::TrainBwd, &r);
    if (rc != GD_OK) return rc;
    if (r.family == gd::Family::Light)
        return gd::light_backward(g, model, weights_dev, x_dev, stash_dev, grad_logit_dev, grad_weights_dev, workspace_dev,
                                  accumulate, B, st);
    gd::BwdPlan pl;
    rc = gd::plan_bwd(g, model, B, &pl);
    if (rc != GD_OK) return rc;
    pl.p.x = x_dev; pl.p.stash = stash_dev; pl.p.grad_logit = grad_logit_dev; pl.p.weights = weights_dev;
    pl.p.partials = workspace_dev;
    if (pl.work_global) pl.p.slab = workspace_dev + gd::bwd_slab_offset(g, model, pl);
    if (r.family == gd::Family::Lean) {
        // decoder_v2_4 on surface / toric codes: when the table forward wrote the stash (its header says so, on the device), the
        // table backward produces the gradient and the two kernels below return at once; otherwise the other way round
        float* bins = workspace_dev + (((int64_t)pl.n_rows * pl.p.np_pad + 3) & ~(int64_t)3);   // 16-byte aligned (64-bit atomics)
        rc = gd::lean_backward(const_cast<gd_graph*>(g), model, r.lean[0], weights_dev, x_dev, stash_dev, grad_logit_dev,
                               grad_weights_dev, bins, accumulate, B, st);
        if (rc != GD_OK) return rc;
        pl.p.run_flag = &gd::lean_train_hdr(const_cast<float*>(stash_dev), g, model, B)->old_count;
    }
    void (*k)(const gd::BwdParams) = pl.work_global ? gd::decode_bwd_kernel<true> : gd::decode_bwd_kernel<false>;
    GD_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, pl.smem));
    GD_CUDA(gd::pdl_launch(k, dim3(pl.grid), dim3(pl.threads), (size_t)pl.smem, st, pl.p));
    GD_CUDA(gd::pdl_launch(gd::reduce_partials_kernel, dim3((n_params + 127) / 128), dim3(128), 0, st, workspace_dev, pl.n_rows,
                           pl.p.np_pad, n_params, grad_weights_dev, accumulate ? 1 : 0, pl.p.run_flag));
    return GD_OK;
}
