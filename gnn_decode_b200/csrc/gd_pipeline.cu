// gd_pipeline: the end-to-end decode with HOST buffers as an asynchronous pipeline.  Replaces the reference's
// `datas = datas.to(device); pred = decoder(datas)` (quantum/decoder_v2_4.py:332-334) plus the read-back of the prediction,
// for callers that stream batches: batch k+1 is copied in while batch k decodes and batch k-1 is copied out.
//
// Three streams -- copy-in, compute, copy-out -- chained per batch by events; `depth` slots of device buffers.  All decode
// kernels run on ONE stream (a decode fills the GPU; running two concurrently only thrashes shared memory), so the table
// cache of the check-owner kernel (gd_lean.cu) is built once and reused by every batch.  submit() never blocks unless all
// slots are in flight (then it waits for the oldest); wait() blocks until a batch's outputs are complete in host memory.
// Inputs come either as x [B, V+C] fp32 (the reference's layout) or packed (one prior float + C check-sign bits per
// syndrome, V hard-decision bits back: what x actually carries -- gen_syn, quantum/error_generate.py:258, 270-276).
#include "gd_common.cuh"
#include <vector>

struct gd_pipeline {
    const gd_graph* g = nullptr;
    gd_model model{};
    int64_t max_B = 0;
    int depth = 0;
    int nw = 0, vw = 0;
    cudaStream_t s_in = nullptr, s_comp = nullptr, s_out = nullptr;
    float* w_dev = nullptr;
    struct Slot {
        float* x = nullptr;          // [max_B, N]   (unpacked submissions)
        float* prior = nullptr;      // [max_B]
        uint32_t* synd = nullptr;    // [max_B, nw]
        float* prob = nullptr;       // [max_B, V]
        uint8_t* hard = nullptr;     // [max_B, V]
        uint32_t* bits = nullptr;    // [max_B, vw]
        cudaEvent_t ev_in = nullptr, ev_comp = nullptr, ev_out = nullptr;
        bool in_flight = false;
        int rc = GD_OK;
    };
    std::vector<Slot> slots;
    long long submitted = 0;         // tickets handed out so far; ticket t lives in slot t % depth
    std::mutex mu;
};

namespace {

void pipeline_free(gd_pipeline* p) {
    if (!p) return;
    gd::DeviceGuard dg(p->g->device);
    for (auto& s : p->slots) {
        if (s.ev_out && s.in_flight) cudaEventSynchronize(s.ev_out);
        cudaFree(s.x); cudaFree(s.prior); cudaFree(s.synd); cudaFree(s.prob); cudaFree(s.hard); cudaFree(s.bits);
        if (s.ev_in) cudaEventDestroy(s.ev_in);
        if (s.ev_comp) cudaEventDestroy(s.ev_comp);
        if (s.ev_out) cudaEventDestroy(s.ev_out);
    }
    if (p->s_in) cudaStreamDestroy(p->s_in);
    if (p->s_comp) cudaStreamDestroy(p->s_comp);
    if (p->s_out) cudaStreamDestroy(p->s_out);
    cudaFree(p->w_dev);
    delete p;
}

// make slot `i` reusable: its previous batch must have left the device
int slot_acquire(gd_pipeline* p, int i) {
    gd_pipeline::Slot& s = p->slots[i];
    if (s.in_flight) {
        GD_CUDA(cudaEventSynchronize(s.ev_out));
        s.in_flight = false;
    }
    return GD_OK;
}

}  // namespace

extern "C" int gd_pipeline_create(const gd_graph* g, const gd_model* model, const float* weights_host, int64_t max_B,
                                  int32_t depth, gd_pipeline** out) {
    GD_CHECK_ARG(out != nullptr, "gd_pipeline_create: out is NULL");
    *out = nullptr;
    GD_CHECK_ARG(g != nullptr && gd_model_valid(model), "gd_pipeline_create: invalid graph / model");
    GD_CHECK_ARG(model->flags == 0, "gd_pipeline_create: per-iteration outputs (GD_FLAG_ALL_ITERS) are device-path only");
    GD_CHECK_ARG(max_B > 0 && max_B < ((int64_t)1 << 31), "gd_pipeline_create: max_B out of range");
    GD_CHECK_ARG(depth >= 1 && depth <= 8, "gd_pipeline_create: depth must be 1..8");
    const int64_t n_w = gd_weights_size(model);
    GD_CHECK_ARG(n_w == 0 || weights_host, "gd_pipeline_create: weights is NULL");
    gd::DeviceGuard dg(g->device);
    GD_CUDA(dg.status());
    gd_pipeline* p = new gd_pipeline();
    p->g = g; p->model = *model; p->max_B = max_B; p->depth = depth;
    p->nw = (g->C + 31) / 32; p->vw = (g->V + 31) / 32;
    p->slots.resize(depth);
    cudaError_t e = cudaStreamCreateWithFlags(&p->s_in, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&p->s_comp, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&p->s_out, cudaStreamNonBlocking);
    if (e == cudaSuccess && n_w) e = cudaMalloc((void**)&p->w_dev, (size_t)n_w * sizeof(float));
    if (e == cudaSuccess && n_w) e = cudaMemcpy(p->w_dev, weights_host, (size_t)n_w * sizeof(float), cudaMemcpyHostToDevice);
    for (auto& s : p->slots) {
        if (e == cudaSuccess) e = cudaMalloc((void**)&s.prior, (size_t)max_B * sizeof(float));
        if (e == cudaSuccess) e = cudaMalloc((void**)&s.synd, (size_t)max_B * p->nw * sizeof(uint32_t));
        if (e == cudaSuccess) e = cudaMalloc((void**)&s.bits, (size_t)max_B * p->vw * sizeof(uint32_t));
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s.ev_in, cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s.ev_comp, cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s.ev_out, cudaEventDisableTiming);
    }
    if (e != cudaSuccess) {
        gd::set_error("gd_pipeline_create: %s", cudaGetErrorString(e));
        pipeline_free(p);
        return GD_ERR_CUDA;
    }
    *out = p;
    return GD_OK;
}

extern "C" void gd_pipeline_destroy(gd_pipeline* p) { pipeline_free(p); }

extern "C" int gd_pipeline_set_weights(gd_pipeline* p, const float* weights_host) {
    GD_CHECK_ARG(p != nullptr, "gd_pipeline_set_weights: pipeline is NULL");
    const int64_t n_w = gd_weights_size(&p->model);
    if (n_w == 0) return GD_OK;
    GD_CHECK_ARG(weights_host != nullptr, "gd_pipeline_set_weights: weights is NULL");
    std::lock_guard<std::mutex> lk(p->mu);
    gd::DeviceGuard dg(p->g->device);
    GD_CUDA(dg.status());
    // in compute-stream order: batches already submitted keep the old weights (pageable source: staged before the call returns)
    cudaError_t e = cudaMemcpyAsync(p->w_dev, weights_host, (size_t)n_w * sizeof(float), cudaMemcpyHostToDevice, p->s_comp);
    GD_CUDA(e);
    return GD_OK;
}

// shared tail of the two submit forms: the compute + copy-out legs and the ticket
static int pipeline_finish(gd_pipeline* p, gd_pipeline::Slot& s, int rc, cudaError_t e, int32_t* ticket) {
    s.rc = rc;
    if (rc != GD_OK) return rc;
    GD_CUDA(e);
    s.in_flight = true;
    if (ticket) *ticket = (int32_t)(p->submitted & 0x7fffffff);
    ++p->submitted;
    return GD_OK;
}

extern "C" int gd_pipeline_submit_packed(gd_pipeline* p, const float* prior_host, const uint32_t* synd_host, float* prob_host,
                                         uint32_t* hard_bits_host, int64_t B, int32_t* ticket) {
    GD_CHECK_ARG(p != nullptr, "gd_pipeline_submit_packed: pipeline is NULL");
    GD_CHECK_ARG(B > 0 && B <= p->max_B, "gd_pipeline_submit_packed: B=%lld outside (0, max_B=%lld]", (long long)B, (long long)p->max_B);
    GD_CHECK_ARG(prior_host && synd_host, "gd_pipeline_submit_packed: inputs are NULL");
    GD_CHECK_ARG(prob_host || hard_bits_host, "gd_pipeline_submit_packed: no output requested");
    std::lock_guard<std::mutex> lk(p->mu);
    const gd_graph* g = p->g;
    gd::DeviceGuard dg(g->device);
    GD_CUDA(dg.status());
    const int i = (int)(p->submitted % p->depth);
    gd_pipeline::Slot& s = p->slots[i];
    int rc = slot_acquire(p, i);
    cudaError_t e = cudaSuccess;
    if (rc == GD_OK && prob_host && !s.prob) e = cudaMalloc((void**)&s.prob, (size_t)p->max_B * g->V * sizeof(float));
    if (rc == GD_OK && e == cudaSuccess) {
        e = cudaMemcpyAsync(s.prior, prior_host, (size_t)B * sizeof(float), cudaMemcpyHostToDevice, p->s_in);
        if (e == cudaSuccess) e = cudaMemcpyAsync(s.synd, synd_host, (size_t)B * p->nw * sizeof(uint32_t), cudaMemcpyHostToDevice, p->s_in);
        if (e == cudaSuccess) e = cudaEventRecord(s.ev_in, p->s_in);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(p->s_comp, s.ev_in, 0);
        if (e == cudaSuccess)
            rc = gd_decode_packed_fwd(g, &p->model, p->w_dev, s.prior, s.synd, prob_host ? s.prob : nullptr,
                                      hard_bits_host ? s.bits : nullptr, B, (void*)p->s_comp);
        if (rc == GD_OK && e == cudaSuccess) e = cudaEventRecord(s.ev_comp, p->s_comp);
        if (rc == GD_OK && e == cudaSuccess) e = cudaStreamWaitEvent(p->s_out, s.ev_comp, 0);
        if (rc == GD_OK && e == cudaSuccess && hard_bits_host)
            e = cudaMemcpyAsync(hard_bits_host, s.bits, (size_t)B * p->vw * sizeof(uint32_t), cudaMemcpyDeviceToHost, p->s_out);
        if (rc == GD_OK && e == cudaSuccess && prob_host)
            e = cudaMemcpyAsync(prob_host, s.prob, (size_t)B * g->V * sizeof(float), cudaMemcpyDeviceToHost, p->s_out);
        if (rc == GD_OK && e == cudaSuccess) e = cudaEventRecord(s.ev_out, p->s_out);
    }
    return pipeline_finish(p, s, rc, e, ticket);
}

extern "C" int gd_pipeline_submit(gd_pipeline* p, const float* x_host, float* prob_host, uint8_t* hard_host, int64_t B,
                                  int32_t* ticket) {
    GD_CHECK_ARG(p != nullptr, "gd_pipeline_submit: pipeline is NULL");
    GD_CHECK_ARG(B > 0 && B <= p->max_B, "gd_pipeline_submit: B=%lld outside (0, max_B=%lld]", (long long)B, (long long)p->max_B);
    GD_CHECK_ARG(x_host != nullptr, "gd_pipeline_submit: x is NULL");
    GD_CHECK_ARG(prob_host || hard_host, "gd_pipeline_submit: no output requested");
    std::lock_guard<std::mutex> lk(p->mu);
    const gd_graph* g = p->g;
    gd::DeviceGuard dg(g->device);
    GD_CUDA(dg.status());
    const int i = (int)(p->submitted % p->depth);
    gd_pipeline::Slot& s = p->slots[i];
    int rc = slot_acquire(p, i);
    cudaError_t e = cudaSuccess;
    if (rc == GD_OK && !s.x) e = cudaMalloc((void**)&s.x, (size_t)p->max_B * g->N * sizeof(float));
    if (rc == GD_OK && e == cudaSuccess && prob_host && !s.prob) e = cudaMalloc((void**)&s.prob, (size_t)p->max_B * g->V * sizeof(float));
    if (rc == GD_OK && e == cudaSuccess && hard_host && !s.hard) e = cudaMalloc((void**)&s.hard, (size_t)p->max_B * g->V);
    if (rc == GD_OK && e == cudaSuccess) {
        e = cudaMemcpyAsync(s.x, x_host, (size_t)B * g->N * sizeof(float), cudaMemcpyHostToDevice, p->s_in);
        if (e == cudaSuccess) e = cudaEventRecord(s.ev_in, p->s_in);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(p->s_comp, s.ev_in, 0);
        if (e == cudaSuccess)
            rc = gd_decode_fwd(g, &p->model, p->w_dev, s.x, prob_host ? s.prob : nullptr, nullptr, hard_host ? s.hard : nullptr, B,
                               (void*)p->s_comp);
        if (rc == GD_OK && e == cudaSuccess) e = cudaEventRecord(s.ev_comp, p->s_comp);
        if (rc == GD_OK && e == cudaSuccess) e = cudaStreamWaitEvent(p->s_out, s.ev_comp, 0);
        if (rc == GD_OK && e == cudaSuccess && prob_host)
            e = cudaMemcpyAsync(prob_host, s.prob, (size_t)B * g->V * sizeof(float), cudaMemcpyDeviceToHost, p->s_out);
        if (rc == GD_OK && e == cudaSuccess && hard_host)
            e = cudaMemcpyAsync(hard_host, s.hard, (size_t)B * g->V, cudaMemcpyDeviceToHost, p->s_out);
        if (rc == GD_OK && e == cudaSuccess) e = cudaEventRecord(s.ev_out, p->s_out);
    }
    return pipeline_finish(p, s, rc, e, ticket);
}

extern "C" int gd_pipeline_wait(gd_pipeline* p, int32_t ticket) {
    GD_CHECK_ARG(p != nullptr, "gd_pipeline_wait: pipeline is NULL");
    cudaEvent_t ev = nullptr;
    {
        std::lock_guard<std::mutex> lk(p->mu);
        const long long newest = p->submitted - 1;
        long long t = (newest & ~0x7fffffffll) | (long long)(uint32_t)ticket;
        if (t > newest) t -= 0x80000000ll;
        GD_CHECK_ARG(ticket >= 0 && t >= 0 && t <= newest, "gd_pipeline_wait: unknown ticket %d", ticket);
        if (newest - t >= p->depth) return GD_OK;                 // its slot was reused since: submit() already waited for it
        gd_pipeline::Slot& s = p->slots[(int)(t % p->depth)];
        if (!s.in_flight) return GD_OK;
        ev = s.ev_out;
    }
    GD_CUDA(cudaEventSynchronize(ev));                            // outside the lock: other threads may keep submitting
    return GD_OK;
}

extern "C" int gd_pipeline_drain(gd_pipeline* p) {
    GD_CHECK_ARG(p != nullptr, "gd_pipeline_drain: pipeline is NULL");
    std::lock_guard<std::mutex> lk(p->mu);
    for (auto& s : p->slots)
        if (s.in_flight) {
            GD_CUDA(cudaEventSynchronize(s.ev_out));
            s.in_flight = false;
        }
    return GD_OK;
}
