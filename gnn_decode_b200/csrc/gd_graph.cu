// Graph preprocessing: per-graph COO edge list -> destination-sorted CSR (by variable) and CSC
// (by check) segment tables, so every aggregation is an atomic-free, fixed-order segmented sum.
// Replaces H.to_sparse()._indices() + PyG collate + the int64 gathers/scatters of
// MessagePassing.propagate (reference quantum/decoder_v2_4.py:136-144,164-165,205-206,277).
#include "gd_common.cuh"
#include <string.h>
#include <new>

namespace gd {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

}  // namespace gd

extern "C" const char* gd_last_error(void) { return gd::g_err; }
extern "C" int gd_abi_version(void) { return GD_ABI_VERSION; }

extern "C" int64_t gd_weights_size(const gd_model* m) {
    if (!gd_model_valid(m)) {
        gd::set_error("gd_weights_size: invalid model");
        return -1;
    }
    const int64_t h = m->hidden;
    switch (m->program) {
        case GD_PROG_V2_4: return 10 * h + 3;
        case GD_PROG_CGNNI:
        case GD_PROG_QGNNI: return 6 * h + 2;
        case GD_PROG_NEURAL_BP: return (2 * (int64_t)m->iters + 2) * h + 1;
        case GD_PROG_GRU_CA: return 9 * h + 27;
        case GD_PROG_V3_0: return 11 * h + 27;
        case GD_PROG_V1_2_2: return 8 * h + 2;
        case GD_PROG_V2_4_1: return (int64_t)m->iters * (6 * h + 18) + 3 * h + 19;
        default: return 0;
    }
}

// Stable counting sort of edge ids by key -> (ptr, ids); ids ascending inside each segment.
static void build_segments(const std::vector<int32_t>& key, int32_t n_seg, std::vector<int32_t>& ptr,
                           std::vector<int32_t>& ids, int32_t& max_deg) {
    const size_t E = key.size();
    ptr.assign((size_t)n_seg + 1, 0);
    for (size_t e = 0; e < E; ++e) ptr[(size_t)key[e] + 1]++;
    max_deg = 0;
    for (int32_t s = 0; s < n_seg; ++s) {
        if (ptr[(size_t)s + 1] > max_deg) max_deg = ptr[(size_t)s + 1];
        ptr[(size_t)s + 1] += ptr[s];
    }
    ids.resize(E);
    std::vector<int32_t> cur(ptr.begin(), ptr.end() - 1);
    for (size_t e = 0; e < E; ++e) ids[(size_t)cur[key[e]]++] = (int32_t)e;
}

extern "C" int gd_graph_create(const int64_t* ei, int64_t E, int32_t V, int32_t C, int device,
                               gd_graph** out) {
    GD_CHECK_ARG(out != nullptr, "gd_graph_create: out is NULL");
    *out = nullptr;
    GD_CHECK_ARG(ei != nullptr, "gd_graph_create: edge_index is NULL");
    GD_CHECK_ARG(V > 0 && C > 0, "gd_graph_create: V=%d, C=%d must be positive", V, C);
    GD_CHECK_ARG(E > 0 && E < (int64_t)1 << 30, "gd_graph_create: E=%lld out of range", (long long)E);
    for (int64_t e = 0; e < E; ++e) {
        GD_CHECK_ARG(ei[e] >= 0 && ei[e] < V, "gd_graph_create: edge %lld has variable id %lld outside [0,%d)",
                     (long long)e, (long long)ei[e], V);
        GD_CHECK_ARG(ei[E + e] >= 0 && ei[E + e] < C,
                     "gd_graph_create: edge %lld has check id %lld outside [0,%d) (pass un-offset check ids)",
                     (long long)e, (long long)ei[E + e], C);
    }
    int n_dev = 0;
    GD_CUDA(cudaGetDeviceCount(&n_dev));
    GD_CHECK_ARG(device >= 0 && device < n_dev, "gd_graph_create: device %d not in [0,%d)", device, n_dev);

    gd_graph* g = new (std::nothrow) gd_graph();
    GD_CHECK_ARG(g != nullptr, "gd_graph_create: out of host memory");
    g->V = V; g->C = C; g->N = V + C; g->E = E; g->device = device;
    g->gstate = nullptr; g->gstate_bytes = 0; g->host_ctx = nullptr; g->lean_ctx = nullptr; g->blob_dev = nullptr;
    g->h_edge_var.resize((size_t)E);
    g->h_edge_chk.resize((size_t)E);
    for (int64_t e = 0; e < E; ++e) {
        g->h_edge_var[(size_t)e] = (int32_t)ei[e];
        g->h_edge_chk[(size_t)e] = (int32_t)ei[E + e];
    }
    build_segments(g->h_edge_var, V, g->h_var_ptr, g->h_var_edges, g->max_var_deg);
    build_segments(g->h_edge_chk, C, g->h_chk_ptr, g->h_chk_edges, g->max_chk_deg);

    // edges of variables with degree >= 2 first: only their variable-phase message depends on the iteration
    g->h_vlist.clear();
    for (int pass = 0; pass < 2; ++pass)
        for (int64_t e = 0; e < E; ++e) {
            const int32_t v = g->h_edge_var[(size_t)e];
            const bool act = g->h_var_ptr[(size_t)v + 1] - g->h_var_ptr[(size_t)v] >= 2;
            if (act == (pass == 0)) g->h_vlist.push_back((int32_t)e);
        }
    g->n_vact = 0;
    for (int32_t v = 0; v < V; ++v) {
        const int32_t d = g->h_var_ptr[(size_t)v + 1] - g->h_var_ptr[(size_t)v];
        if (d >= 2) g->n_vact += d;
    }
    // one blob: edge_var | edge_chk | var_ptr | var_edges | chk_ptr | chk_edges | vlist
    const size_t words = (size_t)E * 5 + (size_t)V + 1 + (size_t)C + 1;
    std::vector<int32_t> blob(words);
    size_t o = 0, o_ev, o_ec, o_vp, o_ve, o_cp, o_ce, o_vl;
    auto put = [&](const std::vector<int32_t>& v, size_t& where) {
        where = o;
        memcpy(blob.data() + o, v.data(), v.size() * sizeof(int32_t));
        o += v.size();
    };
    put(g->h_edge_var, o_ev); put(g->h_edge_chk, o_ec); put(g->h_var_ptr, o_vp);
    put(g->h_var_edges, o_ve); put(g->h_chk_ptr, o_cp); put(g->h_chk_edges, o_ce); put(g->h_vlist, o_vl);

    cudaError_t e;
    cudaDeviceProp prop;
    {
        gd::DeviceGuard dg(device);
        e = dg.status();
        if (e == cudaSuccess) e = cudaMalloc((void**)&g->blob_dev, words * sizeof(int32_t));
        if (e == cudaSuccess) e = cudaMemcpy(g->blob_dev, blob.data(), words * sizeof(int32_t), cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = cudaGetDeviceProperties(&prop, device);
    }
    if (e != cudaSuccess) {
        gd::set_error("gd_graph_create: CUDA failure: %s", cudaGetErrorString(e));
        if (g->blob_dev) cudaFree(g->blob_dev);
        delete g;
        return GD_ERR_CUDA;
    }
    g->sm_count = prop.multiProcessorCount;
    g->max_smem_optin = (int)prop.sharedMemPerBlockOptin;
    g->max_smem_sm = (int)prop.sharedMemPerMultiprocessor;
    g->t.edge_var = g->blob_dev + o_ev;
    g->t.edge_chk = g->blob_dev + o_ec;
    g->t.var_ptr = g->blob_dev + o_vp;
    g->t.var_edges = g->blob_dev + o_ve;
    g->t.chk_ptr = g->blob_dev + o_cp;
    g->t.chk_edges = g->blob_dev + o_ce;
    g->t.vlist = g->blob_dev + o_vl;
    *out = g;
    return GD_OK;
}

void gd_host_ctx_destroy(gd_graph* g);  // gd_host.cu
void gd_lean_ctx_destroy(gd_graph* g);  // gd_lean.cu

extern "C" void gd_graph_destroy(gd_graph* g) {
    if (!g) return;
    {
        gd::DeviceGuard dg(g->device);
        gd_host_ctx_destroy(g);
        gd_lean_ctx_destroy(g);
        if (g->gstate) cudaFree(g->gstate);
        if (g->blob_dev) cudaFree(g->blob_dev);
    }
    delete g;
}

extern "C" int gd_graph_dims(const gd_graph* g, int32_t* V, int32_t* C, int64_t* E, int32_t* max_var_deg,
                             int32_t* max_chk_deg) {
    GD_CHECK_ARG(g != nullptr, "gd_graph_dims: graph is NULL");
    if (V) *V = g->V;
    if (C) *C = g->C;
    if (E) *E = g->E;
    if (max_var_deg) *max_var_deg = g->max_var_deg;
    if (max_chk_deg) *max_chk_deg = g->max_chk_deg;
    return GD_OK;
}

extern "C" int gd_graph_tables(const gd_graph* g, int32_t* var_ptr, int32_t* var_edges, int32_t* chk_ptr,
                               int32_t* chk_edges, int32_t* edge_var, int32_t* edge_chk) {
    GD_CHECK_ARG(g != nullptr, "gd_graph_tables: graph is NULL");
    // read back from the DEVICE copy so tests pin what the kernels actually index with
    const size_t E = (size_t)g->E;
    gd::DeviceGuard dg(g->device);
    GD_CUDA(dg.status());
    auto get = [&](int32_t* dst, const int32_t* src, size_t n) -> cudaError_t {
        return dst ? cudaMemcpy(dst, src, n * sizeof(int32_t), cudaMemcpyDeviceToHost) : cudaSuccess;
    };
    cudaError_t e = get(var_ptr, g->t.var_ptr, (size_t)g->V + 1);
    if (e == cudaSuccess) e = get(var_edges, g->t.var_edges, E);
    if (e == cudaSuccess) e = get(chk_ptr, g->t.chk_ptr, (size_t)g->C + 1);
    if (e == cudaSuccess) e = get(chk_edges, g->t.chk_edges, E);
    if (e == cudaSuccess) e = get(edge_var, g->t.edge_var, E);
    if (e == cudaSuccess) e = get(edge_chk, g->t.edge_chk, E);
    GD_CUDA(e);
    return GD_OK;
}

// ---- device-side verification of a PyG-batched edge_index ----
__global__ void check_batched_kernel(const int64_t* __restrict__ ei, const int32_t* __restrict__ edge_var,
                                     const int32_t* __restrict__ edge_chk, int64_t E, int64_t B, int32_t N,
                                     int32_t chk_offset, unsigned long long* __restrict__ bad) {
    const int64_t total = E * B;
    unsigned long long local = 0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t gph = i / E;
        const int64_t e = i - gph * E;
        const int64_t off = gph * N;
        local += (ei[i] != (int64_t)edge_var[e] + off);
        local += (ei[total + i] != (int64_t)edge_chk[e] + off + chk_offset);
    }
    // warp reduce then one atomic per warp
    for (int o = 16; o > 0; o >>= 1) local += __shfl_xor_sync(0xffffffffu, local, o);
    if ((threadIdx.x & 31) == 0 && local) atomicAdd(bad, local);
}

extern "C" int gd_graph_check_batched(const gd_graph* g, const int64_t* ei_dev, int64_t B, int32_t chk_offset,
                                      void* stream, int64_t* mismatches_host) {
    GD_CHECK_ARG(g && ei_dev && mismatches_host, "gd_graph_check_batched: NULL argument");
    GD_CHECK_ARG(B > 0, "gd_graph_check_batched: B must be positive");
    cudaStream_t st = (cudaStream_t)stream;
    gd::DeviceGuard dg(g->device);
    GD_CUDA(dg.status());
    unsigned long long* bad = nullptr;
    cudaError_t e = cudaMalloc((void**)&bad, sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMemsetAsync(bad, 0, sizeof(unsigned long long), st);
    if (e == cudaSuccess) {
        const int64_t total = g->E * B;
        int blocks = (int)((total + 255) / 256);
        if (blocks > g->sm_count * 8) blocks = g->sm_count * 8;
        check_batched_kernel<<<blocks, 256, 0, st>>>(ei_dev, g->t.edge_var, g->t.edge_chk, g->E, B, g->N,
                                                     chk_offset, bad);
        e = cudaGetLastError();
    }
    unsigned long long h = 0;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&h, bad, sizeof(h), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (bad) cudaFree(bad);
    GD_CUDA(e);
    *mismatches_host = (int64_t)h;
    return GD_OK;
}
