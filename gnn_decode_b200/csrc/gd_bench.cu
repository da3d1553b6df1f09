// Pipe-throughput microbenchmarks: the resident decoders are bound by the MUFU (ex2/lg2) or FP32
// issue rate, not by HBM or the tensor pipe (SURVEY.md section 8d), and MEASURED_PEAKS.json has no
// number for those pipes -- so the roofline denominators for them are measured here, live.
#include "gd_common.cuh"
#include "gd_math.cuh"

namespace gd {

template <int KIND>
__global__ void __launch_bounds__(512) ubench_kernel(float* out, int iters) {
    float a[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) a[j] = 0.01f * (threadIdx.x + 1) + j;
    const float b = 0.999f, c = 0.001f;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if (KIND == 0) a[j] = ex2_approx(-fabsf(a[j]));                       // 1 MUFU
            else if (KIND == 1) a[j] = lg2_approx(1.0f + ex2_approx(-fabsf(a[j])));  // 2 MUFU + 1 FADD
            else if (KIND == 2) a[j] = fmaf(a[j], b, c);                          // 1 FFMA
            else if (KIND == 5) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(a[j] + 1.5f)); a[j] = y; }   // 1 MUFU.RCP + FADD
            else if (KIND == 6) {                                               // backward unit: ex2 + rcp + lg2
                const float t = ex2_approx(-fabsf(a[j])), o = 1.0f + t;
                float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(o));
                a[j] = y + lg2_approx(o);
            }
            else if (KIND == 3) {                                                // softplus unit: the v2_4 inner step
                const float z = fmaf(a[j], b, c);
                const float s = fmaxf(z, 0.f) + lg2_approx(1.0f + ex2_approx(-fabsf(z)));
                a[j] = fmaf(c, s, a[j]);
            }
        }
        if (KIND == 4) {                                                         // packed FFMA2: 2 FMA / instr
            unsigned long long* p = reinterpret_cast<unsigned long long*>(a);
            const float2 bb = make_float2(b, b), cc = make_float2(c, c);
#pragma unroll
            for (int j = 0; j < 4; ++j)
                asm volatile("fma.rn.f32x2 %0, %0, %1, %2;"
                             : "+l"(p[j])
                             : "l"(*reinterpret_cast<const unsigned long long*>(&bb)),
                               "l"(*reinterpret_cast<const unsigned long long*>(&cc)));
        }
    }
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) s += a[j];
    if (s == 123.456f) out[0] = s;
}

// Shared-memory data-pipe throughput: conflict-free 128-bit loads (consecutive lanes read consecutive 16-byte words: 4
// wavefronts of 128 B per warp instruction).  This is the resource that binds the table-only decoder (gd_lean.cu).
__global__ void __launch_bounds__(1024) lds_bench_kernel(float* out, int iters) {
    __shared__ float4 tab[2048];
    for (int i = threadIdx.x; i < 2048; i += blockDim.x) tab[i] = make_float4((float)i, 1.f, 2.f, 3.f);
    __syncthreads();
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    unsigned int idx = threadIdx.x;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float4 c = tab[(idx + j * 96u) & 2047u];
            acc.x += c.x; acc.y += c.y; acc.z += c.z; acc.w += c.w;
        }
        idx += 32u + (unsigned int)(acc.x == 12345.678f);       // keeps the loads inside the loop
    }
    if (acc.x + acc.y + acc.z + acc.w == 123.456f) out[0] = acc.x;
}

}  // namespace gd

// kind: 0 ex2, 1 ex2+lg2(+add), 2 FFMA, 3 softplus unit (2 FFMA 2 FADD 1 FMNMX 2 MUFU), 4 FFMA2.
// result[0] = "units" per second (kind 0/2: instructions x lanes; kind 1/3: units; kind 4: FMAs),
// result[1] = milliseconds of the timed launch.
extern "C" int gd_microbench(int32_t kind, int32_t iters, int device, double* result) {
    GD_CHECK_ARG(result && kind >= 0 && kind <= 7 && iters > 0, "gd_microbench: bad argument");
    gd::DeviceGuard dg(device);
    GD_CUDA(dg.status());
    cudaDeviceProp prop;
    GD_CUDA(cudaGetDeviceProperties(&prop, device));
    gd::DeviceBuffer<float> out;
    GD_CUDA(gd::device_alloc(out, 4));
    const int grid = kind == 7 ? prop.multiProcessorCount : prop.multiProcessorCount * 4, threads = kind == 7 ? 1024 : 512;
    gd::Event e0, e1;
    GD_CUDA(gd::create(e0, cudaEventCreateWithFlags, cudaEventDefault));
    GD_CUDA(gd::create(e1, cudaEventCreateWithFlags, cudaEventDefault));
    float ms = 0.f;
    for (int rep = 0; rep < 3; ++rep) {   // first two are warm-up
        cudaEventRecord(e0.get());
        switch (kind) {
            case 0: gd::ubench_kernel<0><<<grid, threads>>>(out.get(), iters); break;
            case 1: gd::ubench_kernel<1><<<grid, threads>>>(out.get(), iters); break;
            case 2: gd::ubench_kernel<2><<<grid, threads>>>(out.get(), iters); break;
            case 3: gd::ubench_kernel<3><<<grid, threads>>>(out.get(), iters); break;
            case 4: gd::ubench_kernel<4><<<grid, threads>>>(out.get(), iters); break;
            case 5: gd::ubench_kernel<5><<<grid, threads>>>(out.get(), iters); break;
            case 7: gd::lds_bench_kernel<<<grid, threads>>>(out.get(), iters); break;
            default: gd::ubench_kernel<6><<<grid, threads>>>(out.get(), iters); break;
        }
        cudaEventRecord(e1.get());
        cudaEventSynchronize(e1.get());
        cudaEventElapsedTime(&ms, e0.get(), e1.get());
    }
    cudaError_t e = cudaGetLastError();
    GD_CUDA(e);
    // kind 7: units = 128-byte shared-memory wavefronts (a warp-wide 128-bit load is 4 of them)
    const double units = (double)grid * threads * (double)iters * 8.0 * (kind == 7 ? 4.0 / 32.0 : 1.0);
    result[0] = units / (ms * 1e-3);
    result[1] = ms;
    return GD_OK;
}
