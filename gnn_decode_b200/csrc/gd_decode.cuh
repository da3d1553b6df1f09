// Internal interface between the resident (gd_decode.cu) and streamed (gd_streamed.cu) decoders.
#pragma once
#include "gd_common.cuh"

namespace gd {

int streamed_launch_info(const gd_graph* g, const gd_model* model, int64_t B, gd_launch_info* out);
int streamed_decode(gd_graph* g, const gd_model* model, const float* weights_dev, const float* x_dev,
                    float* prob_dev, float* logit_dev, uint8_t* hard_dev, int64_t B, cudaStream_t st);

bool streamed_tma_launch_info(const gd_graph* g, const gd_model* model, int64_t B, gd_launch_info* out);
int streamed_tma_decode(gd_graph* g, const gd_model* model, const float* weights_dev, const float* x_dev,
                        float* prob_dev, float* logit_dev, uint8_t* hard_dev, int64_t B, cudaStream_t st);

// Gated whole-batch launch for gd_decode_host (gd_host.cu): ONE persistent launch over the full batch whose tiles wait for
// the host->device copy of their chunk (in_flags[k] >= epoch, raised by a stream memory operation behind the copy) and
// count completed tiles per chunk (out_counts[k]) so the device->host copy of a chunk can start as soon as its last tile is
// out.  Only the edge-owner resident kernel supports it.
struct Gate {
    const unsigned int* in_flags;
    unsigned int* out_counts;
    int* err;                    // host-mapped: set to 1 if a chunk never arrived (bounded spin)
    unsigned int epoch;
    int chunk_tiles;             // tiles per chunk: chunk of tile t = t / chunk_tiles
};
#ifdef __CUDACC__
// wait until the chunk's host->device copy has landed (flag raised in stream order behind the copy); bounded
__device__ __forceinline__ void gate_wait(const unsigned int* flag, unsigned int epoch, int* err) {
    long long spins = 0;
    while (true) {
        unsigned int v;
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
        if ((int)(v - epoch) >= 0) break;
        if (++spins > (1ll << 22)) { *err = 1; break; }   // seconds: the copy never came; do not hang the GPU
        __nanosleep(100);
    }
}
#endif

bool light_launch_info(const gd_graph* g, const gd_model* model, int64_t B, gd_launch_info* out);
int light_decode(const gd_graph* g, const gd_model* model, const float* weights_dev, const float* x_dev,
                 float* prob_dev, float* logit_dev, uint8_t* hard_dev, int64_t B, cudaStream_t st, const Gate* gate = nullptr,
                 float* stash_dev = nullptr);

bool gated_plan(const gd_graph* g, const gd_model* model, int64_t B, int* tile, int* n_tiles);
int decode_fwd_gated(const gd_graph* g, const gd_model* model, const float* weights_dev, const float* x_dev, float* prob_dev,
                     uint8_t* hard_dev, int64_t B, cudaStream_t st, const Gate& gate);

}  // namespace gd
