/*
 * gnn_decode.h -- C ABI of the B200-native message-passing decoder (libgnn_decode_b200.so).
 *
 * This is the drop-in boundary for the hot path of ironmanaudi/GNN-decode: the forked PyG
 * MessagePassing.propagate() -> scatter "sum over siblings minus self" -> per-edge update(),
 * iterated Nc times by GNNI.forward over a PyG-batched (block-diagonal) Tanner graph.
 * The reference has no FFI (pure Python); each entry point cites the reference interface it
 * replaces.  Paths are relative to the reference tree (GNN-decode/).
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types cross this boundary;
 *   - every function returns an int status (GD_OK == 0); gd_last_error() gives the thread-local
 *     message of the last failure; no C++ exception crosses the boundary;
 *   - "dev" pointers are CUDA device pointers on the graph's device, "host" pointers are host;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); all device
 *     entry points are asynchronous on that stream and allocate nothing on the hot path
 *     (exception: the global-state workspace of very large codes is grown lazily, once);
 *   - tensors are fp32, row-major, BATCH-MAJOR exactly like the reference's flattened tensors:
 *       x      [B, V+C]   == data.x [B*(V+C), 1]   (prior LLR of the V variable nodes, then the
 *                                                   C check-node inputs: (-1)^syndrome, or 0)
 *       m      [B, E]     == edge-resident messages [B*E, 1], edges in the order of the
 *                            per-graph edge_index (H.to_sparse()._indices(): by variable, then check)
 *       prob   [B, V]     == GNNI.forward output [B*V, 1] = P(bit/qubit flipped)
 */
#ifndef GNN_DECODE_H_
#define GNN_DECODE_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GD_ABI_VERSION 2

enum gd_status {
    GD_OK = 0,
    GD_ERR_INVALID = 1,      /* bad argument (the Python layer raises ValueError)          */
    GD_ERR_CUDA = 2,         /* CUDA runtime failure (RuntimeError)                         */
    GD_ERR_UNSUPPORTED = 3   /* valid request this build has no kernel for (RuntimeError)   */
};

/* The five phase programs on the hot path (SURVEY.md section 9.1). */
enum gd_program {
    GD_PROG_CGNNI = 0,        /* classical/CGNNI.py:212-284      hidden 10 ReLU              */
    GD_PROG_QGNNI = 1,        /* quantum/QGNNI.py:186-252        hidden 10 ReLU, x syndrome  */
    GD_PROG_V2_4 = 2,         /* quantum/decoder_v2_4.py:230-294 hidden 128 Softplus         */
    GD_PROG_BP_QUANTUM = 3,   /* quantum/BP.py:101-124,191-219   sum-product, syndrome sign  */
    GD_PROG_BP_CLASSICAL = 4, /* classical/BP.py:99-123,231-259  sum-product                 */
    /* the "next" update programs (SURVEY.md 8(f)-3).  GD_PROG_NEURAL_BP also decodes codes whose edge state does not fit
       shared memory (the TMA-staged streamed kernel; edges in the canonical variable-sorted order there, GD_ERR_UNSUPPORTED
       otherwise); programs 6-9 have a resident kernel only: */
    GD_PROG_NEURAL_BP = 5,    /* quantum/neural_BP.py:236-314    sum-product + per-edge learned weights,
                                 2*Nc un-tied layers, gated residual alpha * m_p, weighted read-out */
    GD_PROG_GRU_CA = 6,       /* quantum/QGNNNI_ca.py:177-251    hidden 20 ReLU MLPs + GRUCell(1,1) updates,
                                 sign-multiplied check phase, one read-out per iteration              */
    GD_PROG_V3_0 = 7,         /* quantum/decoder_v3_0.py:199-290 hidden 10 ReLU MLPs of [sum, node input] + GRUCell(1,1)
                                 per phase, no tanh; a SECOND read-out at the check nodes (gd_decode_fwd_aux) */
    GD_PROG_V1_2_2 = 8,       /* quantum/decoder_v1_2_2.py:212-278 hidden 256 Tanh MLP of [sum, prior] (variable phase),
                                 sum-product check phase + residual, Tanh-MLP read-out of EVERY iteration */
    GD_PROG_V2_4_1 = 9        /* quantum/decoder_v2_4_1.py:255-349 decoder_v2_4 with 2*Nc UN-TIED layers (hidden 128 Softplus),
                                 per-edge-type weights (8 types, derived from the graph: every check must have 4 edges) and a
                                 gated residual sigmoid(alpha) / sigmoid(beta) */
};

/* gd_model.flags */
#define GD_FLAG_ALL_ITERS 1   /* GD_PROG_GRU_CA / GD_PROG_V1_2_2: the reference returns a LIST of Nc predictions
                                 (deep supervision, QGNNNI_ca.py:239-249, decoder_v1_2_2.py:267-278); prob / logit /
                                 hard are then [iters, B, V] instead of [B, V] (the last iteration otherwise) */

/* flow of one propagate(): which node type the reduce runs over. */
enum gd_phase {
    GD_PHASE_VAR = 0,  /* flow='source_to_target': reduce over edge_index[0] (variable nodes) */
    GD_PHASE_CHK = 1   /* flow='target_to_source': reduce over edge_index[1] (check nodes)    */
};

/* Opaque, immutable, device-resident Tanner-graph tables (destination-sorted CSR by variable
 * and CSC by check, per-edge endpoints).  Replaces the per-batch int64 edge_index gathers /
 * scatters of MessagePassing.propagate (decoder_v2_4.py:136-144). */
typedef struct gd_graph gd_graph;

/* Model description for the fused decoder.  `weights` buffers are packed fp32 in state_dict
 * order of the tensors the reference's forward actually uses:
 *   V2_4       : ggc1.mlp.{0.weight[h,2],0.bias[h],2.weight[1,h],2.bias[1]},
 *                ggc2.mlp.{0.weight[h,1],0.bias[h],2.weight[1,h],2.bias[1]}, mlp.{same}   (10h+3)
 *   CGNNI      : ggc2.mlp2.{...}, mlp.{...}                                                (6h+2)
 *   QGNNI      : ggc2.mlp.{...},  mlp.{...}                                                (6h+2)
 *   BP_*       : none (weights may be NULL)
 *   NEURAL_BP  : for l in 0..iters-1: layers.{2l}.W[E], layers.{2l}.W_p[E]; then W[E], W_p[E], alpha
 *                ((2 iters + 2) E + 1 floats; `hidden` carries E, checked against the graph)
 *   GRU_CA     : ggc1.mlp1{0.weight[h,1],0.bias[h],2.weight[1,h],2.bias[1]}, ggc1.rnn{weight_ih[3],
 *                weight_hh[3],bias_ih[3],bias_hh[3]}, ggc2.mlp2{...}, ggc2.rnn{...}, mlp{...}   (9h+27)
 *   V3_0       : ggc1.mlp1{0.weight[h,2],0.bias[h],2.weight[1,h],2.bias[1]}, ggc1.rnn1{weight_ih[3],weight_hh[3],
 *                bias_ih[3],bias_hh[3]}, ggc2.mlp2{0.weight[h,2],...}, ggc2.rnn2{...}, mlp{0.weight[h,1],...}   (11h+27)
 *                (the state_dict's ggc1.mlp2 / ggc1.rnn2 / ggc2.mlp1 / ggc2.rnn1 are never used by the forward)
 *   V1_2_2     : ggc1.mlp{0.weight[h,2],0.bias[h],2.weight[1,h],2.bias[1]}, mlp{0.weight[h,2],...}              (8h+2)
 *   V2_4_1     : for l in 0..iters-1: layers.{2l}.mlp1{0.weight[h,1],0.bias[h],2.weight[1,h],2.bias[1]}, layers.{2l}.W[8],
 *                layers.{2l}.W_p[8], layers.{2l+1}.mlp{...}; then mlp{...}, W[8], W_p[8], alpha, beta
 *                (iters (6h+18) + 3h+19; the W / W_p of the target_to_source layers are never used by the forward)
 */
typedef struct gd_model {
    int32_t program;   /* enum gd_program                                   */
    int32_t hidden;    /* h: 128 for V2_4, 10 for CGNNI/QGNNI, 0 for BP, 20 for GRU_CA; E for NEURAL_BP */
    int32_t iters;     /* Nc (T) message-passing iterations                  */
    int32_t flags;     /* 0, or GD_FLAG_ALL_ITERS (GRU_CA, V1_2_2)           */
} gd_model;

const char* gd_last_error(void);
int gd_abi_version(void);

/* Number of floats in the packed weight buffer of `model` (0 for BP); <0 on invalid model. */
int64_t gd_weights_size(const gd_model* model);

/* ---- graph preprocessing (replaces CustomDataset.__init__ `H.to_sparse()._indices()` +
 *      PyG DataLoader collate + the `+rows` offset: decoder_v2_4.py:164-165,205-206,277) ---- */

/* edge_index_host: [2, E] int64 row-major, row 0 = variable id in [0,V), row 1 = check id in
 * [0,C) (un-offset, as in data.edge_index of ONE graph).  device: CUDA ordinal. */
int gd_graph_create(const int64_t* edge_index_host, int64_t E, int32_t V, int32_t C, int device,
                    gd_graph** out);
void gd_graph_destroy(gd_graph* g);
int gd_graph_dims(const gd_graph* g, int32_t* V, int32_t* C, int64_t* E, int32_t* max_var_deg,
                  int32_t* max_chk_deg);
/* Copy the tables back to host int32 arrays (any pointer may be NULL):
 *   var_ptr[V+1], var_edges[E] : CSR, edges of each variable in ascending edge id
 *   chk_ptr[C+1], chk_edges[E] : CSC, edges of each check in ascending edge id
 *   edge_var[E], edge_chk[E]   : endpoints of each edge                                  */
int gd_graph_tables(const gd_graph* g, int32_t* var_ptr, int32_t* var_edges, int32_t* chk_ptr,
                    int32_t* chk_edges, int32_t* edge_var, int32_t* edge_chk);
/* Verify on the device that a PyG-batched edge_index_dev [2, B*E] int64 is the block-diagonal
 * replication of the graph: ei[0][g*E+e] == var[e] + g*(V+C), ei[1][g*E+e] == chk[e] + g*(V+C)
 * + chk_offset (chk_offset = V after GNNI.forward's `.add(rows)`, 0 for raw data.edge_index).
 * Writes the number of mismatching entries to *mismatches_host (synchronises the stream). */
int gd_graph_check_batched(const gd_graph* g, const int64_t* edge_index_dev, int64_t B,
                           int32_t chk_offset, void* stream, int64_t* mismatches_host);

/* ---- one propagate() (decoder_v2_4.py:85-148, CGNNI.py:52-112, QGNNI.py:54-116,
 *      quantum/BP.py:54-124, classical/BP.py:52-123) fused with GraphConv.update
 *      (decoder_v2_4.py:253-257, CGNNI.py:238-242, QGNNI.py:207-214) ----
 * m_dev [B,E] in, out_dev [B,E] out.  weights_dev is the packed k->h->1 MLP of THIS GraphConv
 * only ({0.weight, 0.bias, 2.weight, 2.bias}; NULL where the phase has no MLP).
 * x_dev [B,V+C] may be NULL only where the reference
 * passes post=None (CGNNI check phase).  With fuse_update == 0 the kernel stops before
 * update() and writes the tensor the reference hands to self.update(): out_dev is [B,E,F]
 * with F = gd_propagate_features(program, phase) (2 where the reference `cat`s extra). */
int gd_propagate_features(int32_t program, int32_t phase);
int gd_propagate_fwd(const gd_graph* g, const gd_model* model, int32_t phase, int32_t fuse_update,
                     const float* m_dev, const float* x_dev, const float* weights_dev,
                     float* out_dev, int64_t B, void* stream);

/* ---- the fused decoder: GNNI.forward (decoder_v2_4.py:272-294, CGNNI.py:259-284,
 *      QGNNI.py:228-252, quantum/BP.py:199-219, classical/BP.py:239-259) ----
 * One persistent kernel keeps a tile of syndromes' edge state on chip for all `iters`
 * iterations.  Outputs (any may be NULL): prob_dev [B,V] fp32 = sigmoid(-logit) (clamped to
 * [1e-7,1-1e-7] for the classical programs as the reference does), logit_dev [B,V] fp32,
 * hard_dev [B,V] uint8 = (prob > 0.5) (neural_BP.py:338 semantics).
 * Arithmetic: fp32.  The scalar 1 -> h -> 1 MLPs are evaluated as tables built per launch from the weights
 * (ReLU: exact piecewise-linear segments; Softplus: cubic Hermite on the compact argument domain, used only
 * when an error bound computed from the weights is below 1e-7 / 4e-6, else the direct sum) -- logits stay
 * within 1e-4 relative of the fp64 reference (tests/test_parity_gpu.py).  Results are deterministic and do
 * not depend on how the batch is tiled or sharded.
 * GD_PROG_V2_4 on graphs with variable degree <= 2 and check degree <= 4 (every surface / toric code) and iters <= 32 takes
 * the check-owner table kernel (csrc/gd_lean.cu): all three MLPs and the tanh as cubic tables built in double precision
 * once per weight set and kept in a per-(stream, weights pointer) cache on the device that a content hash validates on every
 * call -- editing the weights in place is fine.  Rows the tables cannot serve (priors that differ inside a row, check
 * inputs other than +-1, non-finite priors) are decoded by the direct evaluation, per row; a batch with more than 64
 * distinct priors, or weights whose tables miss their error budget, as a whole.  gd_decode_launch_info() tells which
 * kernel a call takes; GD_NO_LEAN=1 (gd_set_option) keeps to the edge-owner kernel.
 * Codes whose edge state does not fit shared memory run the streamed global-memory kernel, whose
 * per-graph state slab is allocated lazily and is NOT re-entrant: serialise streamed decodes of
 * one gd_graph across streams (gd_decode_launch_info().resident == 0 tells which path is taken). */
int gd_decode_fwd(const gd_graph* g, const gd_model* model, const float* weights_dev,
                  const float* x_dev, float* prob_dev, float* logit_dev, uint8_t* hard_dev,
                  int64_t B, void* stream);

/* gd_decode_fwd plus the SECOND read-out of the programs that have one (any output may be NULL):
 *   GD_PROG_V3_0: aux_prob_dev / aux_logit_dev [B, C] = the check-node prediction res_p = mlp(sum over the check's edges of
 *   the messages after the LAST variable phase) (decoder_v3_0.py:267-268, 276); prob = sigmoid(-logit).
 * The reference returns both read-outs over all V+C nodes; the remaining rows are constants of the inputs (res at a check
 * row = mlp(0) + its syndrome input, res_p at a variable row = mlp(0)) that the caller's drop-in class fills in.
 * Other programs: GD_ERR_UNSUPPORTED when an aux pointer is given. */
int gd_decode_fwd_aux(const gd_graph* g, const gd_model* model, const float* weights_dev,
                      const float* x_dev, float* prob_dev, float* logit_dev, uint8_t* hard_dev,
                      float* aux_prob_dev, float* aux_logit_dev, int64_t B, void* stream);

/* The same decode with PACKED inputs and outputs.  What the reference's x carries per syndrome (gen_syn,
 * quantum/error_generate.py:258, 270-276) is ONE prior value log((1-p)/p), repeated on all V variables, and C check signs:
 *   prior_dev     [B] fp32            the prior LLR of the syndrome's variables
 *   synd_dev      [B, ceil(C/32)] u32 bit c (of word c / 32) set = check c fired, i.e. its input is -1
 *   prob_dev      [B, V] fp32         optional, as gd_decode_fwd
 *   hard_bits_dev [B, ceil(V/32)] u32 optional, bit v set = (prob > 0.5): the hard decision of variable v
 * 8 + 8 bytes per syndrome instead of 296 + 250 at rotated d = 5.  Results are bit-identical to gd_decode_fwd on the
 * expanded x.  GD_PROG_V2_4, resident codes only (GD_ERR_UNSUPPORTED otherwise). */
int gd_decode_packed_fwd(const gd_graph* g, const gd_model* model, const float* weights_dev, const float* prior_dev,
                         const uint32_t* synd_dev, float* prob_dev, uint32_t* hard_bits_dev, int64_t B, void* stream);

/* Same computation with HOST buffers: host->device copy of x, the kernel, device->host copy of
 * the requested outputs.  The batch is cut into up to 4 chunks that run through an internal gd_pipeline (below) kept
 * per graph; returns when the outputs are complete.  Calls on one graph are serialised internally (they share that
 * pipeline); use one gd_pipeline per caller for concurrency.  Replaces `datas.to(device); pred = decoder(datas)`
 * (decoder_v2_4.py:332-334) followed by reading the prediction back. weights_host is the packed buffer on the host. */
int gd_decode_host(const gd_graph* g, const gd_model* model, const float* weights_host,
                   const float* x_host, float* prob_host, uint8_t* hard_host, int64_t B);

/* ---- the same end-to-end call as an ASYNCHRONOUS PIPELINE for callers that stream batches: batch k+1 is copied in
 *      while batch k decodes and batch k-1 is copied out (three internal streams chained by events, `depth` slots of
 *      device buffers, all decode kernels on one stream so the decoder's tables are built once).  The weights are
 *      copied at creation (gd_pipeline_set_weights replaces them in stream order).  submit returns at once unless all
 *      `depth` slots are in flight (then it waits for the oldest batch); gd_pipeline_wait(ticket) returns when that
 *      batch's outputs are complete in host memory; host buffers must stay valid until then and should be pinned
 *      (pageable memory works, the copies then stage synchronously).  One pipeline may be driven from several host
 *      threads (calls are serialised).
 *      gd_pipeline_submit        x_host [B, V+C] fp32 -> prob_host [B, V] fp32 and / or hard_host [B, V] uint8
 *      gd_pipeline_submit_packed prior_host [B] fp32 + synd_host [B, ceil(C/32)] u32 -> hard_bits_host [B, ceil(V/32)] u32
 *                                and / or prob_host (the layouts of gd_decode_packed_fwd): 16 bytes per syndrome over
 *                                PCIe instead of 546 at rotated d = 5.  GD_PROG_V2_4 only. ---- */
typedef struct gd_pipeline gd_pipeline;
int gd_pipeline_create(const gd_graph* g, const gd_model* model, const float* weights_host, int64_t max_B, int32_t depth,
                       gd_pipeline** out);
void gd_pipeline_destroy(gd_pipeline* p);
int gd_pipeline_set_weights(gd_pipeline* p, const float* weights_host);
int gd_pipeline_submit(gd_pipeline* p, const float* x_host, float* prob_host, uint8_t* hard_host, int64_t B, int32_t* ticket);
int gd_pipeline_submit_packed(gd_pipeline* p, const float* prior_host, const uint32_t* synd_host, float* prob_host,
                              uint32_t* hard_bits_host, int64_t B, int32_t* ticket);
int gd_pipeline_wait(gd_pipeline* p, int32_t ticket);
int gd_pipeline_drain(gd_pipeline* p);   /* wait for every batch submitted so far */

/* ---- training (BASELINE config 4): forward that also stashes the per-iteration activations, and
 *      the hand-written backward (replaces autograd through the loop, decoder_v2_4.py:334-340,
 *      CGNNI.py:314-329).  Programs: GD_PROG_V2_4, GD_PROG_CGNNI and GD_PROG_NEURAL_BP.  stash_dev holds
 *      gd_stash_floats() floats:
 *        GD_PROG_V2_4     : [(iters+1)][2][E][B] (+ a header of the table kernel, gd_lean.cuh);
 *        GD_PROG_CGNNI    : [iters][E][B], m after every iteration (the backward recomputes the rest);
 *        GD_PROG_NEURAL_BP: [iters][E][B], m^1 .. m^iters (m^0 = 0 is not stored; the backward recomputes the rest).
 *      GD_PROG_V2_4 trains on any code the library decodes: where the edge state does not fit shared memory
 *      (or under GD_FORCE_STREAMED) the forward is the TMA-staged streamed kernel writing the same stash
 *      layout, and where the backward's per-tile arrays do not fit shared memory its work arrays go to the
 *      workspace; the two choices are independent.  There, graphs in another edge order than the canonical
 *      variable-sorted one, and graphs with E >= 65536, return GD_ERR_UNSUPPORTED.
 *      GD_PROG_CGNNI trains on the node-owner kernel only: graphs in another edge order than the canonical
 *      variable-sorted one, and codes whose edge state does not fit shared memory, return GD_ERR_UNSUPPORTED.
 *      GD_PROG_NEURAL_BP (model.hidden == E, else GD_ERR_INVALID) trains on every code on the TMA-staged streamed
 *      forward and its own backward; graphs in another edge order than the canonical variable-sorted one return
 *      GD_ERR_UNSUPPORTED before anything is launched.
 *      gd_decode_bwd takes dL/dlogit [B,V], the gradient w.r.t. the logit BEFORE the clamp the classical
 *      programs apply (prob = sigmoid(-logit), so dL/dlogit = -dL/dprob * prob * (1 - prob); for CGNNI with
 *      prob = clamp(s, 1e-7, 1-1e-7), s = sigmoid(-logit): -dL/dprob * s * (1 - s) where 1e-7 <= s <= 1-1e-7,
 *      else 0) and writes (accumulate == 0) or adds (accumulate != 0) dL/dweights in the packed order of
 *      gd_model.  workspace_dev: gd_bwd_workspace_floats() floats (8-byte aligned) of per-warp partial sums
 *      (GD_PROG_V2_4; where the backward does not fit shared memory also one work slab per CTA, about
 *      390 KB per syndrome of the CTA's tile at HGP [[1600,64]]), per-CTA fixed-point bins
 *      (GD_PROG_CGNNI), or (GD_PROG_NEURAL_BP, 16-byte aligned) one record of (2 iters + 2) E partial gradients
 *      and one slab of (N + V + 4 E) rows of the CTA's tile per CTA -- 960 MB at HGP [[1600,64]], iters = 15,
 *      B = 4096 (86 CTAs of 48 syndromes) -- reduced in a fixed order ->
 *      bit-reproducible gradients; gd_bwd_workspace_floats returns -1 for other programs. ---- */
int64_t gd_stash_floats(const gd_graph* g, const gd_model* model, int64_t B);
int gd_decode_fwd_train(const gd_graph* g, const gd_model* model, const float* weights_dev,
                        const float* x_dev, float* prob_dev, float* logit_dev, float* stash_dev,
                        int64_t B, void* stream);
int64_t gd_bwd_workspace_floats(const gd_graph* g, const gd_model* model, int64_t B);
int gd_decode_bwd(const gd_graph* g, const gd_model* model, const float* weights_dev,
                  const float* x_dev, const float* stash_dev, const float* grad_logit_dev,
                  float* grad_weights_dev, float* workspace_dev, int32_t accumulate, int64_t B,
                  void* stream);

/* ---- training loss, fused with its gradient (replaces LossFunc.forward(train=1) + the autograd of it,
 *      quantum/decoder_v2_4.py:304-317; sparse check lists instead of the dense H^T matmul and the O(B)
 *      cat loops):  z = y + prob;  loss_b = sum_c |sin(pi/2 sum_{v in c} z_v)| + sum_k |sin(pi/2 logical_k . z)|.
 *      prob_dev [B,V] fp32, y_dev [B,V] uint8 (the sampled error, data.y), logical_dev [K,V] uint8.
 *      Outputs: loss_per_syndrome_dev [B] (the caller sums it: a fixed order, deterministic),
 *      grad_prob_dev [B,V] = dL/dprob and grad_logit_dev [B,V] = -dL/dprob * prob * (1 - prob), the
 *      tensor gd_decode_bwd takes (either gradient pointer may be NULL). ---- */
int gd_loss_v2_4(const gd_graph* g, const uint8_t* logical_dev, int32_t K, const float* prob_dev,
                 const uint8_t* y_dev, float* loss_per_syndrome_dev, float* grad_prob_dev,
                 float* grad_logit_dev, int64_t B, void* stream);

/* ---- data-parallel training: one-shot all-reduce of the flat gradient (10h+3 floats) over NVLink / NVSwitch peer
 *      memory in ONE kernel (replaces nothing in the reference, which is single-GPU; BASELINE config 4).
 *      Every rank owns a symmetric buffer of gd_p2p_buffer_floats(n) floats (zero-initialised once) that all ranks
 *      have mapped; peer_ptrs_host[r] is rank r's buffer as seen from THIS process.  The kernel publishes src in the
 *      caller's buffer, raises its epoch flag, waits (bounded) for the peers and writes dst[i] = scale * sum over ranks
 *      in rank order -- bit-identical on every rank.  epoch must be 1, 2, 3, ... on successive calls, the same on all
 *      ranks; if a peer never arrives (bounded wait, tens of seconds) *err_dev is set to 1 and NOTHING is written: dst and,
 *      for gd_p2p_allreduce_adam, the weights and moments keep their values -- check err_dev before trusting a step. ---- */
int64_t gd_p2p_buffer_floats(int32_t n);
int gd_p2p_allreduce(const uint64_t* peer_ptrs_host, int32_t world, int32_t rank, const float* src_dev,
                     float* dst_dev, int32_t n, uint32_t epoch, float scale, int32_t* err_dev, void* stream);

/* ---- optimizer step (replaces torch.optim.Adam(decoder.parameters(), lr=3e-4, weight_decay=1e-9).step(),
 *      quantum/decoder_v2_4.py:323, 338) on the FLAT fp32 master weight vector (the `weights_dev` layout of
 *      gd_decode_fwd) in one launch.  Arithmetic of torch.optim.Adam's default path: g += weight_decay * w;
 *      m += (1-beta1)(g-m); v = beta2 v + (1-beta2) g^2; w -= lr/(1-beta1^step) * m / (sqrt(v)/sqrt(1-beta2^step) + eps).
 *      step = 1, 2, 3, ... is the step being taken; the gradient is read as grad_scale * grad_dev[i].
 *      gd_p2p_allreduce_adam = gd_p2p_allreduce with this update applied to the reduced gradient in the same kernel
 *      (dst_dev may be NULL when the reduced gradient itself is not needed): the exchange step of data-parallel
 *      training and the optimizer are ONE launch, and every rank applies a bit-identical update. ---- */
typedef struct gd_adam {
    double lr, beta1, beta2, eps, weight_decay;   /* doubles, as Python passes them: 1 - beta is formed before rounding to fp32 */
    int32_t step;
} gd_adam;
int gd_adam_step(const gd_adam* opt, float* weights_dev, const float* grad_dev, float* exp_avg_dev,
                 float* exp_avg_sq_dev, int64_t n, float grad_scale, void* stream);
int gd_p2p_allreduce_adam(const uint64_t* peer_ptrs_host, int32_t world, int32_t rank, const float* src_dev,
                          float* dst_dev, int32_t n, uint32_t epoch, float scale, int32_t* err_dev,
                          const gd_adam* opt, float* weights_dev, float* exp_avg_dev, float* exp_avg_sq_dev,
                          void* stream);

/* Launch geometry the library picked for (graph, model, B): for benchmarks / roofline. */
typedef struct gd_launch_info {
    int32_t tile;            /* syndromes per CTA tile                          */
    int32_t threads;         /* threads per CTA                                 */
    int32_t grid;            /* CTAs                                            */
    int32_t smem_bytes;      /* dynamic shared memory per CTA                   */
    int32_t resident;        /* 1 = edge state in shared memory, 0 = in global  */
    int32_t n_tiles;
} gd_launch_info;
int gd_decode_launch_info(const gd_graph* g, const gd_model* model, int64_t B, gd_launch_info* out);
/* Cubic tables the resident GD_PROG_V2_4 kernel plans for (graph, model, B): out4 = {check-phase intervals, read-out
 * intervals, variable-phase intervals per table, variable-phase table slots}; 0 = that MLP is evaluated directly (the
 * kernel additionally checks an interpolation-error bound from the weights at launch and falls back if it fails). */
int gd_decode_tables_info(const gd_graph* g, const gd_model* model, int64_t B, int32_t* out4);
/* Optional one-time geometry autotuning for (graph, model, B): times the best `max_candidates` (0 = 24) geometries of the
 * planner's model with the caller's own weights and batch (outputs go to a scratch buffer) and remembers the fastest;
 * later gd_decode_fwd / gd_decode_host calls with the same (model, B) use it.  Synchronises the stream.  Only the
 * edge-owner resident kernel is tuned; other paths return immediately.  *chosen (may be NULL) receives the result. */
int gd_decode_autotune(const gd_graph* g, const gd_model* model, const float* weights_dev, const float* x_dev,
                       int64_t B, int32_t max_candidates, void* stream, gd_launch_info* chosen);

/* ---- synthetic input: on-GPU Philox4x32-10 sampler with the layout and distribution of
 *      gen_syn (error_generate.py:252-278): per sample s, p = p_list[philox(seed, s) % n_p];
 *      x = [log((1-p)/p)]*V | (-1)^(H^T e mod 2);  y = e.
 *      noise: 0 = reference iid X/Z flips (each of the V slots flips w.p. p);
 *             1 = depolarizing on V/2 qubits (X,Y,Z each p/3; slot j = X part, j+V/2 = Z part,
 *                 prior = log((1-2p/3)/(2p/3)));
 *             2 / 3 = the classical input of Gen_Data.AWGN + CustomDataset (classical/CGNNI.py:
 *                 125-147,159): BPSK of the all-zero (2) / all-one (3) codeword over AWGN,
 *                 p_list = SNR in dB (one drawn per sample), sigma = 10^(-SNR/20),
 *                 x = [2 y / sigma^2]*V | 0*C (Box-Muller on the Philox words); err = the codeword. */
int gd_sample(const gd_graph* g, int32_t noise, const float* p_list_host, int32_t n_p,
              uint64_t seed, uint64_t first_sample, float* x_dev, uint8_t* err_dev, int64_t B,
              void* stream);

/* ---- evaluation (neural_BP.py:338-348 semantics): counts, over B samples, how many decodes
 *      leave a non-zero residual syndrome (H^T (e xor ehat) != 0) and how many flip a logical
 *      (logical_dev [K, V] uint8 row-major ON THE DEVICE, may be NULL with K = 0; rows are applied
 *      to (e xor ehat) directly, exactly as `logical` from H_Prep.get_logical is used).  counts_dev[0] = residual
 *      syndrome failures, counts_dev[1] = logical failures among syndrome-satisfying decodes,
 *      counts_dev[2] = total failures (either). counts are ADDED to (uint64). */
int gd_eval_failures(const gd_graph* g, const uint8_t* logical_dev, int32_t K,
                     const uint8_t* err_dev, const uint8_t* hard_dev, int64_t B,
                     unsigned long long* counts_dev, void* stream);

/* ---- measurement support: throughput of the pipes that bound the resident decoders
 *      (kind 0 MUFU ex2, 1 ex2+lg2, 2 FFMA, 3 one Softplus hidden unit, 4 packed FFMA2, 5 rcp, 6 ex2+rcp+lg2,
 *      7 shared-memory wavefronts: conflict-free 128-bit loads, units = 128-byte wavefronts -- the pipe that binds the
 *      table-only decoder of surface / toric codes).
 *      result[0] = units / s over the whole GPU, result[1] = ms of the timed launch. ---- */
int gd_microbench(int32_t kind, int32_t iters, int device, double* result);

/* ---- library tunables.  Every planner switch (GD_NO_LEAN, GD_FORCE_STREAMED, GD_LEAN_R, ... -- the list is in
 *      gnn_decode_b200/csrc/gd_options.cuh) lives in one table that is filled from the environment ONCE, at first use;
 *      nothing on the launch path reads the environment.  gd_set_option changes an entry at run time (unset != 0:
 *      back to "not given").  Returns GD_ERR_INVALID for an unknown name. ---- */
int gd_set_option(const char* name, int64_t value, int32_t unset);

#ifdef __cplusplus
}
#endif
#endif /* GNN_DECODE_H_ */
