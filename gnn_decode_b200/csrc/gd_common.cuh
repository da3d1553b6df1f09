// Shared internals of libgnn_decode_b200.so (not part of the ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <string.h>
#include <vector>
#include <mutex>

#include "../../include/gnn_decode.h"

namespace gd {

void set_error(const char* fmt, ...);

#define GD_CHECK_ARG(cond, ...)                 \
    do {                                        \
        if (!(cond)) {                          \
            gd::set_error(__VA_ARGS__);         \
            return GD_ERR_INVALID;              \
        }                                       \
    } while (0)

#define GD_CUDA(call)                                                                        \
    do {                                                                                     \
        cudaError_t e__ = (call);                                                            \
        if (e__ != cudaSuccess) {                                                            \
            gd::set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #call,                 \
                          cudaGetErrorString(e__));                                          \
            return GD_ERR_CUDA;                                                              \
        }                                                                                    \
    } while (0)

// Makes `device` current for the guard's scope and gives the caller's device back when the scope ends, on every return
// path.  The library's entry points switch only through this guard.
class DeviceGuard {
public:
    explicit DeviceGuard(int device) {
        err_ = cudaGetDevice(&prev_);
        if (err_ == cudaSuccess && prev_ != device) {
            err_ = cudaSetDevice(device);
            switched_ = err_ == cudaSuccess;
        }
    }
    ~DeviceGuard() {
        if (switched_) cudaSetDevice(prev_);
    }
    DeviceGuard(const DeviceGuard&) = delete;
    DeviceGuard& operator=(const DeviceGuard&) = delete;
    cudaError_t status() const { return err_; }   // of the switch: check it with GD_CUDA before using the device

private:
    int prev_ = 0;
    bool switched_ = false;
    cudaError_t err_ = cudaSuccess;
};

// Device blob layout (int32 words): all tables of one Tanner graph, uploaded once.
struct GraphTables {
    const int32_t* edge_var;   // [E]   variable endpoint of edge e
    const int32_t* edge_chk;   // [E]   check endpoint of edge e (un-offset)
    const int32_t* var_ptr;    // [V+1] CSR row pointers
    const int32_t* var_edges;  // [E]   edge ids of each variable, ascending
    const int32_t* chk_ptr;    // [C+1]
    const int32_t* chk_edges;  // [E]
    const int32_t* vlist;      // [E]   edge ids: first the n_vact edges whose variable has degree >= 2, then the rest
};

// Programmatic dependent launch.  Kernels that follow one another on a stream (the passes of a decode call, the launches of a
// training step) are launched with programmatic stream serialisation and begin with pdl_enter(): the next kernel's CTAs are
// scheduled while this one drains, and nothing of this kernel runs before its predecessor has completed and its writes are visible.
// In a launch without the attribute both instructions are no-ops.
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_enter() {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
}
template <typename... KArgs, typename... Args>
static inline cudaError_t pdl_launch(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}
#endif

}  // namespace gd

struct gd_graph {
    int32_t V, C, N;
    int64_t E;
    int32_t max_var_deg, max_chk_deg;
    int32_t n_vact;             // edges on variables of degree >= 2 (a degree-1 variable's message never changes)
    int device;
    int sm_count;
    int max_smem_optin;
    int max_smem_sm;
    int32_t* blob_dev;          // single allocation holding all tables
    gd::GraphTables t;          // device pointers into blob_dev
    std::vector<int32_t> h_edge_var, h_edge_chk, h_var_ptr, h_var_edges, h_chk_ptr, h_chk_edges, h_vlist;
    // lazily grown scratch (guarded by mu): global edge-state workspace for codes too large
    // for shared memory, and gd_decode_host's internal pipeline.
    std::mutex mu;
    float* gstate;
    size_t gstate_bytes;
    void* host_ctx;             // gd_decode_host pipeline state (see gd_host.cu)
    void* lean_ctx;             // check-owner table kernel: per-(R) metadata, workspace pool (see gd_lean.cu)
    // geometries measured by gd_decode_autotune (guarded by mu): key = {program, hidden, iters, flags, B}
    struct TunedGeom { int32_t program, hidden, iters, flags; int64_t B; int32_t tile, R, eb; };
    std::vector<TunedGeom> tuned;
};

static inline bool gd_model_valid(const gd_model* m) {
    if (!m) return false;
    if (m->iters < 0) return false;
    if (m->flags != 0 && !(m->flags == GD_FLAG_ALL_ITERS && (m->program == GD_PROG_GRU_CA || m->program == GD_PROG_V1_2_2))) return false;
    switch (m->program) {
        case GD_PROG_GRU_CA:
        case GD_PROG_V3_0:
        case GD_PROG_V1_2_2:
        case GD_PROG_V2_4_1:
            return m->hidden >= 1 && m->hidden <= 256;
        case GD_PROG_NEURAL_BP:
            return m->hidden >= 1;          // = E, checked against the graph at launch
        case GD_PROG_CGNNI:
        case GD_PROG_QGNNI:
        case GD_PROG_V2_4:
            return m->hidden >= 1 && m->hidden <= 256;
        case GD_PROG_BP_QUANTUM:
        case GD_PROG_BP_CLASSICAL:
            return true;
        default:
            return false;
    }
}
