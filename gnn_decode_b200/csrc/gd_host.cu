// gd_decode_host: the end-to-end call with HOST buffers.  Replaces the reference's
// `datas = datas.to(device); pred = decoder(datas)` (quantum/decoder_v2_4.py:332-334) plus the
// read-back of the prediction.  The batch is cut into chunks that are submitted to one internal gd_pipeline per graph
// (gd_pipeline.cu), so one chunk's copies overlap the decode of its neighbours; the call then waits for all of them.
#include "gd_decode.cuh"
#include <algorithm>

namespace gd {

struct HostCtx {
    std::mutex call_mu;              // one gd_decode_host call at a time per graph: the pipeline is shared state
    gd_pipeline* pipe = nullptr;
    gd_model model{};                // the pipeline was created for this model ...
    int64_t max_B = 0;               // ... and chunks of up to max_B syndromes
    ~HostCtx() { gd_pipeline_destroy(pipe); }
};
template struct Delete<HostCtx>;

}  // namespace gd

extern "C" int gd_decode_host(const gd_graph* gc, const gd_model* model, const float* weights_host,
                              const float* x_host, float* prob_host, uint8_t* hard_host, int64_t B) {
    gd_graph* g = const_cast<gd_graph*>(gc);
    GD_CHECK_ARG(g != nullptr, "gd_decode_host: graph is NULL");
    GD_CHECK_ARG(gd_model_valid(model), "gd_decode_host: invalid model");
    GD_CHECK_ARG(B >= 0 && B < ((int64_t)1 << 31), "gd_decode_host: B out of range");
    GD_CHECK_ARG(model->flags == 0, "gd_decode_host: per-iteration outputs (GD_FLAG_ALL_ITERS) are device-path only");
    if (B == 0) return GD_OK;
    GD_CHECK_ARG(x_host != nullptr, "gd_decode_host: x is NULL");
    GD_CHECK_ARG(prob_host || hard_host, "gd_decode_host: no output requested");
    const int64_t n_w = gd_weights_size(model);
    GD_CHECK_ARG(n_w == 0 || weights_host, "gd_decode_host: weights is NULL");

    gd::DeviceGuard dg(g->device);
    GD_CUDA(dg.status());
    gd::Route r;
    int rc = gd::route_decode(g, model, B, gd::Use::Infer, &r);
    if (rc != GD_OK) return rc;
    // chunks: multiples of 8 syndromes (output alignment); >= 4096 syndromes each, at most 4; the streamed kernels take the
    // batch in one piece.  GNNI.autotune (message_passing.py) tunes the launch geometry for these chunk sizes: keep the two
    // in step.
    int n_chunks = (int)std::min<int64_t>(4, std::max<int64_t>(1, B / 8192));
    if (r.family == gd::Family::StreamedTma || r.family == gd::Family::Streamed) n_chunks = 1;
    const int64_t per = ((B + n_chunks - 1) / n_chunks + 7) / 8 * 8;

    std::unique_lock<std::mutex> lk(g->mu);
    if (!g->host_ctx) g->host_ctx.reset(new gd::HostCtx());
    gd::HostCtx* c = g->host_ctx.get();
    lk.unlock();  // gd_decode_fwd takes the same mutex for the streamed workspace
    std::lock_guard<std::mutex> call_lk(c->call_mu);
    const bool same_model = c->model.program == model->program && c->model.hidden == model->hidden &&
                            c->model.iters == model->iters && c->model.flags == model->flags;
    if (!c->pipe || per > c->max_B || !same_model) {
        gd_pipeline_destroy(c->pipe);
        rc = gd_pipeline_create(g, model, weights_host, per, 4, &c->pipe);
        if (rc != GD_OK) return rc;
        c->model = *model;
        c->max_B = per;
    }
    rc = gd_pipeline_set_weights(c->pipe, weights_host);
    for (int64_t b0 = 0; b0 < B && rc == GD_OK; b0 += per) {
        const int64_t nb = std::min<int64_t>(per, B - b0);
        rc = gd_pipeline_submit(c->pipe, x_host + b0 * g->N, prob_host ? prob_host + b0 * g->V : nullptr,
                                hard_host ? hard_host + b0 * g->V : nullptr, nb, nullptr);
    }
    // drain even after an error: chunks already submitted are still writing into the caller's buffers
    const int rc_drain = gd_pipeline_drain(c->pipe);
    return rc != GD_OK ? rc : rc_drain;
}
