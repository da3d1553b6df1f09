// On-GPU synthetic syndrome sampler: Philox4x32-10, counter = (sample index, block), key = seed.
// Reproduces the LAYOUT and DISTRIBUTION of the reference's gen_syn (quantum/error_generate.py:
// 252-278: p drawn uniformly from the list P per sample, prior = log((1-p)/p) on all V slots,
// independent X and Z flips, x = [prior | (-1)^(H^T e mod 2)], y = e) -- the reference itself
// uses the unseeded Mersenne Twister of Python/NumPy, so only the distribution can match.
// noise == 1 adds the depolarizing channel BASELINE.json names (not present in the reference).
// noise == 2 / 3 is the classical input of classical/CGNNI.py:125-147,159: BPSK of the all-zero (2) or
// all-one (3) codeword over AWGN, sigma = 10^(-SNR/20) with the SNR (dB) drawn from the list per
// sample, x = [2 y / sigma^2 | 0 ... 0]; the "err" output is the transmitted codeword (data.y).
#include "gd_common.cuh"

namespace gd {

constexpr int kMaxP = 64;
struct SampleParams {
    float p[kMaxP];
    float prior[kMaxP];
    int n_p;
    int noise;
    uint32_t seed_lo, seed_hi;
    unsigned long long first;
    float* x;
    uint8_t* err;
    long long B;
    int V, C, N;
    GraphTables tb;
};

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u;
        k.y += 0xBB67AE85u;
    }
    return c;
}
__device__ __forceinline__ float u01(uint32_t w) { return (float)(w >> 8) * (1.0f / 16777216.0f); }

// one warp per sample; lane l draws Philox blocks l, l+32, ... (4 slots / qubits per block)
__global__ void __launch_bounds__(128) sample_kernel(const SampleParams p) {
    extern __shared__ uint8_t esm[];  // [4 warps][Vpad]
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int V = p.V, Vpad = (V + 15) / 16 * 16;
    uint8_t* e = esm + wib * Vpad;
    const uint2 key = make_uint2(p.seed_lo, p.seed_hi);
    for (long long b = blockIdx.x * 4ll + wib; b < p.B; b += gridDim.x * 4ll) {
        const unsigned long long sid = p.first + (unsigned long long)b;
        const uint32_t s_lo = (uint32_t)sid, s_hi = (uint32_t)(sid >> 32);
        const uint4 sel = philox4x32_10(make_uint4(s_lo, s_hi, 0u, 0u), key);   // stream 0: p choice
        const int pi = (int)(sel.x % (uint32_t)p.n_p);
        const float pr = p.p[pi], prior = p.prior[pi];
        if (p.noise >= 2) {
            // AWGN: Box-Muller on the four uniforms of a Philox block -> four N(0,1) draws
            const float sigma = pr, inv_var2 = prior;      // p[] holds sigma, prior[] holds 2 / sigma^2
            const float tx = p.noise == 2 ? 1.0f : -1.0f;
            float* xr = p.x + b * p.N;
            for (int j0 = lane * 4; j0 < V; j0 += 128) {
                const uint4 r = philox4x32_10(make_uint4(s_lo, s_hi, (uint32_t)(j0 >> 2), 1u), key);
                const float u0 = ((float)(r.x >> 8) + 1.0f) * (1.0f / 16777216.0f), u1 = u01(r.y);
                const float u2 = ((float)(r.z >> 8) + 1.0f) * (1.0f / 16777216.0f), u3 = u01(r.w);
                const float r0 = sqrtf(-2.0f * logf(u0)), r1 = sqrtf(-2.0f * logf(u2));
                float s0, c0, s1, c1;
                sincospif(2.0f * u1, &s0, &c0);
                sincospif(2.0f * u3, &s1, &c1);
                const float nz[4] = {r0 * c0, r0 * s0, r1 * c1, r1 * s1};
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    if (j0 + q < V) {
                        xr[j0 + q] = (tx + sigma * nz[q]) * inv_var2;
                        if (p.err) p.err[b * V + j0 + q] = p.noise == 3 ? 1 : 0;
                    }
            }
            for (int c = lane; c < p.C; c += 32) xr[V + c] = 0.0f;
            continue;
        }
        if (p.noise == 0) {
            for (int j0 = lane * 4; j0 < V; j0 += 128) {
                const uint4 r = philox4x32_10(make_uint4(s_lo, s_hi, (uint32_t)(j0 >> 2), 1u), key);
                const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    if (j0 + q < V) e[j0 + q] = u01(w[q]) < pr ? 1 : 0;
            }
        } else {
            const int n = V >> 1;
            const float t1 = pr / 3.0f, t2 = 2.0f * pr / 3.0f;
            for (int j0 = lane * 4; j0 < n; j0 += 128) {
                const uint4 r = philox4x32_10(make_uint4(s_lo, s_hi, (uint32_t)(j0 >> 2), 1u), key);
                const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    if (j0 + q < n) {
                        const float u = u01(w[q]);
                        e[j0 + q] = u < t2 ? 1 : 0;                       // X or Y -> X part
                        e[n + j0 + q] = (u >= t1 && u < pr) ? 1 : 0;      // Y or Z -> Z part
                    }
            }
        }
        __syncwarp();
        float* xr = p.x + b * p.N;
        for (int j = lane; j < V; j += 32) {
            xr[j] = prior;
            if (p.err) p.err[b * V + j] = e[j];
        }
        for (int c = lane; c < p.C; c += 32) {
            int par = 0;
            for (int i = p.tb.chk_ptr[c]; i < p.tb.chk_ptr[c + 1]; ++i) par ^= e[p.tb.edge_var[p.tb.chk_edges[i]]];
            xr[V + c] = par ? -1.0f : 1.0f;
        }
        __syncwarp();
    }
}

}  // namespace gd

extern "C" int gd_sample(const gd_graph* g, int32_t noise, const float* p_list, int32_t n_p, uint64_t seed,
                         uint64_t first_sample, float* x_dev, uint8_t* err_dev, int64_t B, void* stream) {
    GD_CHECK_ARG(g != nullptr, "gd_sample: graph is NULL");
    GD_CHECK_ARG(noise >= 0 && noise <= 3, "gd_sample: noise must be 0 (iid X/Z), 1 (depolarizing), 2/3 (AWGN, codeword 0/1)");
    GD_CHECK_ARG(p_list && n_p >= 1 && n_p <= gd::kMaxP, "gd_sample: need 1..%d error rates", gd::kMaxP);
    GD_CHECK_ARG(noise != 1 || (g->V % 2) == 0, "gd_sample: depolarizing noise needs V = 2n slots");
    GD_CHECK_ARG(B >= 0, "gd_sample: negative B");
    if (B == 0) return GD_OK;
    GD_CHECK_ARG(x_dev != nullptr, "gd_sample: x is NULL");
    gd::SampleParams p;
    for (int i = 0; i < n_p && noise >= 2; ++i) {   // p_list = SNR in dB (CGNNI.py:129: sigma = (1 / 10^(SNR/10))^0.5)
        const double sigma = sqrt(1.0 / pow(10.0, (double)p_list[i] / 10.0));
        p.p[i] = (float)sigma;
        p.prior[i] = (float)(2.0 / (sigma * sigma));
    }
    for (int i = 0; i < n_p && noise < 2; ++i) {
        GD_CHECK_ARG(p_list[i] > 0.f && p_list[i] < 1.f, "gd_sample: error rate %g outside (0,1)", (double)p_list[i]);
        const double pd = (double)p_list[i];
        const double pm = noise == 0 ? pd : 2.0 * pd / 3.0;   // marginal flip probability of one slot
        p.p[i] = p_list[i];
        p.prior[i] = (float)log((1.0 - pm) / pm);
    }
    p.n_p = n_p; p.noise = noise; p.seed_lo = (uint32_t)seed; p.seed_hi = (uint32_t)(seed >> 32);
    p.first = first_sample; p.x = x_dev; p.err = err_dev; p.B = B; p.V = g->V; p.C = g->C; p.N = g->N; p.tb = g->t;
    int64_t blocks = (B + 3) / 4;
    if (blocks > (int64_t)g->sm_count * 16) blocks = (int64_t)g->sm_count * 16;
    const int smem = 4 * ((g->V + 15) / 16 * 16);
    gd::DeviceGuard dg(g->device);
    GD_CUDA(dg.status());
    cudaError_t e = cudaSuccess;
    if (smem > 48 * 1024)
        e = cudaFuncSetAttribute(gd::sample_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e == cudaSuccess) {
        gd::sample_kernel<<<(int)blocks, 128, smem, (cudaStream_t)stream>>>(p);
        e = cudaGetLastError();
    }
    GD_CUDA(e);
    return GD_OK;
}
