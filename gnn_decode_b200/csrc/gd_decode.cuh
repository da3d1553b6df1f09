// Internal interface of the decode kernel families and of the routing that picks one per call (DESIGN.md §4):
// the check-owner table kernel (gd_lean.cu), the node-owner kernel (gd_decode_light.cu), the edge-owner resident kernel
// (gd_decode.cu), and the TMA-staged (gd_streamed_tma.cu) and register-batched (gd_streamed.cu) streamed kernels.
#pragma once
#include "gd_common.cuh"
#include "gd_lean.cuh"
#include "gd_light.cuh"

namespace gd {

// ---- edge-owner resident kernel (gd_decode.cu) ----
struct DecodeParams {
    const float* x;
    float* prob;
    float* logit;
    uint8_t* hard;
    const float* weights;
    float* stash;           // training only: [(T+1)][2][E][B] = per-iteration (m_it, a_it), final m in slot T
    GraphTables tb;
    long long B;
    int T, V, C, E, N;
    int tile, R, hid, hp, n_tiles, maxvc, all_iters, wslot;
    int n_vact;             // edges on variables of degree >= 2 (GraphTables::vlist)
    int vdirect, cdirect;   // V2_4: max variable degree <= 2 / max check degree <= 4 -> sibling messages are read directly
    int scratch_bytes;      // bytes of shared memory from off_x to the end (prologue scratch)
    int rtab_n, off_rtab;   // V2_4: intervals of the read-out MLP's cubic table (0 = direct) and its smem offset
    int ctab_n, off_ctab;   // V2_4: intervals of the check-phase cubic table (0 = direct evaluation) and its smem offset
    float ctab_R;           // half-width of its domain: max check degree - 1
    // V2_4: cubic tables of the variable-phase MLP's sections f(ext, prior = const), one per distinct prior value a CTA
    // meets (inputs made like the reference's gen_syn carry one prior per syndrome, drawn from a short list)
    int vtab_n, vtab_k, off_vtab, off_vmeta;
    int off_w, off_tab, off_x, off_node, off_m, off_t;
    // deferred pass behind the check-owner table kernel (gd_lean.cu): decode only the listed syndromes (*defer_count > 0),
    // the whole batch (-1) or nothing (0); all NULL otherwise
    const int* defer_count;
    const int* defer_idx;
    uint32_t* hard_bits;    // optional packed hard decisions [B][ceil(V/32)]
    float* aux_prob; float* aux_logit;   // GD_PROG_V3_0: the check-node read-out [B][C]
};

struct DecodePlan {
    DecodeParams p;
    int threads, grid, smem, resident, eb, npad;
};

// Intervals of decoder_v2_4's cubic tables in the edge-owner kernel: check phase, read-out, variable phase.  The edge-owner
// backward builds its adjoint check table with kCtabN too: it differentiates the function the forward evaluated.
constexpr int kCtabN = 512, kRtabN = 2048, kVtabN = 512;

// ---- streamed kernels: the edge state lives in a per-CTA slab in global memory ----
struct StreamParams {
    const float* x;
    float* prob;
    float* logit;
    uint8_t* hard;
    const float* weights;
    GraphTables tb;
    float* slab;
    long long B;
    long long slab_floats;   // per CTA
    int T, V, C, E, N;
    int tile, R, hid, hp, n_tiles;
    int ctab_n, rtab_n;      // V2_4: intervals of the check-phase / read-out cubic tables (0 = direct evaluation)
    float ctab_R;
};

struct StreamPlan {
    StreamParams p;
    int threads, grid, smem;
};

struct StreamTmaParams {
    const float* x;
    float* prob;
    float* logit;
    uint8_t* hard;
    const float* weights;
    GraphTables tb;
    float* slab;
    long long B;
    long long slab_floats;   // per CTA
    int T, V, C, E, N;
    int tile, lanes, W, hid, hp, n_tiles;
    int stage_rows;          // rows of tile floats per pipeline stage
    int S;                   // pipeline stages per warp (2..4): S - 1 nodes are in flight while one is evaluated
    int vchunk;              // variables per variable-phase item
    int vrows;               // row index of the first prior row inside a variable-phase stage
    int off_w, off_stage;    // shared-memory byte offsets (mbarriers sit at 0)
    int off_ctab, off_rtab, ctab_n, rtab_n;   // decoder_v2_4: cubic tables of the check-phase and read-out MLPs (0: none)
    float ctab_R;
    float* stash;            // training (decoder_v2_4): [(T+1)][2][E][B], the edge-owner kernel's layout (gnn_decode.h)
};

struct StreamTmaPlan {
    StreamTmaParams p;
    int threads, grid, smem, npad;
    bool ok;                 // false: the register-batched kernel takes the call (plan_streamed_tma says why)
    const char* why;         // the reason when !ok
};

int plan_streamed(const gd_graph* g, const gd_model* m, int64_t B, StreamPlan* out);
// train: decoder_v2_4's training forward (the kernel also writes the stash); no batch-size gate, training has no other
// streamed kernel
void plan_streamed_tma(const gd_graph* g, const gd_model* m, int64_t B, StreamTmaPlan* out, bool train = false);

// ---- routing ----
// The buffers of one decode call; NULL where the call does not ask for them.
struct DecodeIO {
    const float* weights;
    const float* x;                              // [B][V+C], or NULL with the packed inputs below
    const float* prior; const uint32_t* synd;    // packed inputs (gd_decode_packed_fwd)
    float* prob; float* logit; uint8_t* hard; uint32_t* hard_bits;
    float* stash;                                // training forward
    float* aux_prob; float* aux_logit;           // GD_PROG_V3_0: the check-node read-out
};

enum class Family { Lean, Light, EdgeOwner, StreamedTma, Streamed };

enum class Use {
    Infer,      // gd_decode_fwd(_aux), gd_decode_host, the launch / table queries, the autotuner
    Packed,     // gd_decode_packed_fwd: decoder_v2_4 on the resident kernels only
    Train,      // gd_decode_fwd_train
    TrainBwd,   // gd_decode_bwd: the same family as Train; the backward kernels lay out their own shared memory
};

struct Route {
    Family family = Family::EdgeOwner;
    std::vector<LeanPlan> lean;  // Lean: one plan per launch (the whole graph, or each of its connected components)
    LightPlan light;             // Light
    DecodePlan edge;             // EdgeOwner; Lean: its deferred pass (Train / Infer / Packed)
    StreamTmaPlan tma;           // StreamedTma
    StreamPlan streamed;         // Streamed
};

// Decides which family serves (graph, model, B) for `use` and plans it; a gd_status (argument errors and the refusals of
// programs or codes no kernel serves).  Runs on the graph's device: the table kernel's planning uploads metadata.
int route_decode(const gd_graph* g, const gd_model* model, int64_t B, Use use, Route* out);
gd_launch_info route_launch_info(const Route& r);
// Launches the routed family on the current device (the graph's).
int decode_routed(gd_graph* g, const gd_model* model, const Route& r, const DecodeIO& io, int64_t B, cudaStream_t st);

// ---- the families' launchers: plan + buffers -> gd_status ----
int edge_decode(const gd_graph* g, const gd_model* model, DecodePlan pl, const DecodeIO& io, cudaStream_t st,
                const DeferList* dl = nullptr);
// *no_resources: the table kernel could not get its memory pool or a table set, and enqueued nothing that decodes
int lean_decode(gd_graph* g, const gd_model* model, const std::vector<LeanPlan>& pls, const DecodePlan& deferred,
                const DecodeIO& io, int64_t B, cudaStream_t st, bool* no_resources);
int light_decode(const LightPlan& pl, const gd_model* model, const DecodeIO& io, cudaStream_t st);
int streamed_decode(gd_graph* g, const StreamPlan& pl, const gd_model* model, const DecodeIO& io, cudaStream_t st);
int streamed_tma_decode(gd_graph* g, const StreamTmaPlan& pl, const gd_model* model, const DecodeIO& io, cudaStream_t st);

}  // namespace gd
