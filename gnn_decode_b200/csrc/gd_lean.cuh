// Internal interface of the check-owner table kernel for decoder_v2_4 on surface / toric codes (gd_lean.cu).
#pragma once
#include "gd_common.cuh"

namespace gd {

constexpr int kLeanMaxSlots = 64;   // distinct priors a table set can hold (one 8 KB variable-phase table each, in global memory)

// per call: two of them live in the header and alternate, so that call n's decode kernel can clear the one call n + 1 will
// use (nobody else touches it in between: its last reader, the deferred pass of call n - 1, is long done) -- no memset launch
struct LeanCall {
    int overflow;                // more distinct priors than table slots: the whole batch takes the edge-owner kernel
    int defer_count;             // syndromes listed in defer_idx; -1 = all of them, in batch order
    int count[kLeanMaxSlots];    // syndromes of this batch that carry the prior of slot k
    unsigned int fmax_new;       // max |mlp2| over the check table's nodes, gathered by the prep kernel when the weights changed
    unsigned int d2_new;         // ... max |mlp2'| there, and max |mlp3'| on a coarse grid over the widest domain the tables can take:
    unsigned int d3_new;         //   the amplification estimate the table kernel sizes the variable-phase tables with
    int pad[1];
};

// Device-side state of one table set (lives in a cache entry of the graph, persists across calls): the tables are rebuilt
// only when the content hash of (weights, T, table sizes) changes, variable-phase tables are added as new priors show up.
struct LeanHeader {
    unsigned long long hash;     // what the tables were built from
    unsigned long long built_mask;   // slots whose variable-phase table is complete
    unsigned long long pending_hash; // hash of this call's weights; becomes `hash` once the table kernel has rebuilt
    int rebuild;                 // this call found other weights: every table is rebuilt
    int n_slots;                 // distinct priors in the list
    int vt_n_eff;                // pieces of the variable-phase tables: base * 2^k, finer for wider message domains
    int vt_mult;                 // ... at least base * vt_mult: raised by the decode kernel when a table set missed its budget (0 = 1)
    int forced;                  // the decode kernel asked for the rebuild (hash cleared): keep vt_mult
    int pad0;
    unsigned int fmax_bits;      // max |mlp2| over the check table's nodes (float bits, rounded up)
    unsigned int f3max_bits;     // max |mlp3| over the read-out table's nodes
    unsigned int err_c_bits;     // a-posteriori interpolation error of the check table (sampled interval midpoints)
    unsigned int err_r_bits;     // ... of the read-out table
    unsigned int d2max_bits;     // max |mlp2'| and max |mlp3'| over the nodes: how much a table error is amplified on its way
    unsigned int d3max_bits;     //   to the logits (the variable-phase tables' budget shrinks with their product)
    unsigned int err_v_bits[kLeanMaxSlots];  // ... of each variable-phase table (in units of tanh output)
    unsigned int slot_bits[kLeanMaxSlots];   // prior value (float bits) of table slot k; 0xFFFFFFFF = free
    LeanCall calls[2];
};

// Training (decoder_v2_4): the header at the END of the stash buffer (gd_stash_floats() reserves kLeanTrainTailFloats + B floats
// behind the edge-owner kernel's [(T+1)][2][E][B] layout).  It says which forward wrote the stash, so the matching backward runs:
// both forwards / both backwards are launched every step and the one whose turn it is not returns at once -- the choice is made
// on the device, no host synchronisation.
constexpr int kLeanTrainTailFloats = 512;
struct LeanTrainHdr {
    int status;                  // 1: the table kernel wrote an m-only stash [T][E][B] (sorted positions) for ALL rows; 0: edge-owner layout
    int old_count;               // DeferList count of the edge-owner forward / backward: 0 when status == 1, -1 (all rows) otherwise
    int n_slots;
    int pad;
    unsigned int fmax_bits;      // max |mlp2| the tables' domains were built from
    int vt_n_eff;                // pieces of the variable-phase tables
    unsigned int pad1[2];
    int count[kLeanMaxSlots];
    unsigned int slot_bits[kLeanMaxSlots];
    // followed (at float offset kLeanTrainTailFloats) by idx[B]: the prior-sorted syndrome list
};
static_assert(sizeof(LeanTrainHdr) <= kLeanTrainTailFloats * 4, "training header");

// Edge-owner kernel pass over the syndromes the lean kernel deferred (gd_decode.cu).
struct DeferList {
    const int* count;            // &LeanCall::defer_count
    const int* idx;              // [B] syndrome indices (valid when *count > 0)
};

struct LeanParams {
    // packed inputs, sorted by prior
    const int* idx;              // [B] syndrome ids: first the call->count[0] ones that carry the prior of slot 0, then slot 1's, ...
    const uint32_t* sgn;         // [B][nw] bit c = check c's input is -1
    float* prob; float* logit; uint8_t* hard; uint32_t* hard_bits;
    LeanHeader* hdr;
    LeanCall* call;              // this call's state
    LeanCall* next_call;         // the next call's: cleared here
    float* stash;                // training: m after every iteration, [T][E][B] by sorted position (NULL otherwise)
    LeanTrainHdr* train;         // training: the header at the end of the stash buffer
    const int* idx_src;          // training: the prior-sorted list, copied behind the header
    const float4* ctab; const float4* rtab; const float4* vtab;   // global tables: (n + 2) pieces each, piece 0 = interval -1
    const uint32_t* meta;        // device metadata blob of this (graph, R)
    long long B;
    int T, V, C, E, nw, vw, P;   // P = odd pitch of the staged logits; E = edges of THIS launch's part of the graph
    int v_lo, nv, part;          // the part's variables [v_lo, v_lo + nv); part = 1: one of several launches (connected components)
    int R, G, NCH;               // owners per group, groups per CTA, checks per owner (padded)
    int ct_n, rt_n, vt_n;        // vt_n: BASE piece count of the variable-phase tables (the header holds the one in use)
    int train_vt_max;            // training: most pieces the backward kernel can seat
    int off_me, off_ms, off_mi, off_var, off_ct, off_rt, off_vt, off_state;   // shared-memory byte offsets
};

struct LeanMeta;
// One launch of the table kernel: the whole graph, or one of its connected components.
struct LeanPlan {
    LeanParams p;
    int threads, grid, smem, n_tiles;
    const LeanMeta* meta;
    int n_parts = 1;                       // launches this plan is one of
};

// Plans the table kernel for (graph, model, B); false when it does not serve them.  whole_only: training (the stash is laid
// out by global edge id), and the forward and the backward of a step plan alike.
bool lean_plan(gd_graph* g, const gd_model* m, int64_t B, std::vector<LeanPlan>* out, bool whole_only = false);
// training: the table backward of the forward `fwd` planned.  It runs only if the stash header says the table forward wrote
// the stash; when it has no room at all it launches nothing (the forward saw the same and left the stash to the edge-owner
// kernel).  grad_weights_dev receives (or accumulates) the 10h+3 gradients; bins_dev: lean_bwd_bins_floats() floats.
int lean_backward(gd_graph* g, const gd_model* model, const LeanPlan& fwd, const float* weights_dev, const float* x_dev,
                  const float* stash_dev, const float* grad_logit_dev, float* grad_weights_dev, float* bins_dev, int accumulate,
                  int64_t B, cudaStream_t st);
int64_t lean_bwd_bins_floats(const gd_graph* g, const gd_model* model);
inline LeanTrainHdr* lean_train_hdr(float* stash, const gd_graph* g, const gd_model* m, int64_t B) {
    return reinterpret_cast<LeanTrainHdr*>(stash + (int64_t)(m->iters + 1) * 2 * g->E * B);
}
int packed_via_unpack(gd_graph* g, const float* prior_dev, const uint32_t* synd_dev, int64_t B, cudaStream_t st,
                      int (*run)(void* ctx, const float* x_dev), void* ctx);

}  // namespace gd
