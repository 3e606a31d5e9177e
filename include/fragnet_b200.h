/*
 * fragnet_b200 -- C ABI of the B200 (sm_100a) kernels behind FragNet's GAT2 hot path.
 *
 * The reference (pnnl/FragNet) is pure Python; on this path it calls three third-party
 * native ops through their Python bindings:
 *     torch_scatter.scatter_add / scatter_softmax    fragnet/model/gat/gat2.py:153-165,210-219,
 *                                                    234,257-268,303-312,820-821
 *     torch_geometric.utils.add_self_loops           fragnet/model/gat/gat2.py:179
 *     torch.index_select / nn.Linear (ATen)          fragnet/model/gat/gat2.py:139-147,189-201,...
 * The entry points below are what a binding for that boundary links against.  Conventions:
 *   - every pointer is a DEVICE pointer owned by the caller (PyTorch tensors); the library never
 *     allocates, frees or synchronises; outputs and workspaces are caller-allocated;
 *   - the last argument is the cudaStream_t to launch on (passed as void*);
 *   - return value: 0 = ok, negative = argument validation error (see fnb_error_string),
 *     positive = cudaError_t of a failed launch;
 *   - the kernel-level entry points are re-entrant; the program-level ones (fnb_encoder_*, fnb_pretrain_heads_*,
 *     fnb_pretrain_step) fork onto three lazily created, library-owned auxiliary streams (+ events) per device and join
 *     back before they return, so one host thread per device should drive them (the reference's loops are single
 *     threaded).  FNB_STREAMS=1 in the environment keeps every launch on the caller's stream, FNB_PDL=0 turns
 *     programmatic dependent launch off.
 *     Process-wide state otherwise: a diagnostic launch counter;
 *   - all feature matrices are row-major fp32 with D = 128
 *     columns, H = 4 heads of d = 32 (the only geometry FragNet's gat2 uses with emb_dim 128);
 *   - graph indices handed in are int64 (as produced by the reference's collate_fn,
 *     fragnet/dataset/data.py:931-948); the CSR arrays produced and consumed are int32.
 */
#ifndef FRAGNET_B200_H
#define FRAGNET_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FNB_D 128 /* embedding width  */
#define FNB_H 4   /* attention heads  */
#define FNB_ABI_VERSION 13

/* arithmetic of the dense projections */
#define FNB_PRECISION_FP32 0 /* FP32 FFMA: bit-for-bit comparable with the reference within 1e-5            */
#define FNB_PRECISION_TF32 1 /* tcgen05 tensor cores, TF32 operands, FP32 accumulate (stated tolerance 2e-3) */
#define FNB_PRECISION_TF32X3 2 /* tcgen05 tensor cores, 3xTF32 error-compensated split (hi*hi + hi*lo + lo*hi),
                                  FP32 accumulate: FP32-grade results, within 1e-5 of the reference             */

/* edge-term modes of the fused attention kernels (SURVEY.md App. A.5) */
#define FNB_EDGE_NONE 0   /* no edge term                                              */
#define FNB_EDGE_AFFINE1 1 /* bond graph: S_e[h] = attr[slot]*coef[h] + coef[4+h]       */
#define FNB_EDGE_AFFINE6 2 /* fragment-connection graph: attr[slot,0:6] . coef[h,0:6] + coef[24+h] */
#define FNB_EDGE_TABLE 3  /* atom / fragment graph: S_e = table[eid[slot], 0:4]; eid >= n_real -> 0 (self loop) */

int fnb_version(void);
const char *fnb_error_string(int code);
/* Diagnostic: number of kernels this library has launched in this process (monotonic). */
uint64_t fnb_launch_count(void);

/* Scratch bytes every backward / reduction entry point may use (constant, independent of sizes). */
size_t fnb_scratch_bytes(void);

/* ---- (a) on-device collate: destination-sorted CSR + reverse (source-sorted) CSR ------------
 * Replaces the implicit grouping done by scatter_softmax/scatter_add (gat2.py:153-165 etc.) and
 * add_self_loops (gat2.py:179).  Edges are (dst[e], src[e]), e < n_edges; with
 * append_self_loops != 0, n_nodes extra edges (i,i) with ids n_edges+i follow them.
 * Slots of one destination are ordered by edge id (== stable sort by destination):
 *   rowptr[n_nodes+1], col[slot] = source node, row[slot] = destination node (may be NULL),
 *   eid[slot] = edge id, slot_of_eid[e] = slot
 * Reverse CSR groups the same edges by source, again ordered by edge id:
 *   rrowptr[n_nodes+1], rslot[r] = forward slot of that edge, rdst[r] = its destination node.
 * With rrowptr != NULL and at least one edge, rslot, rdst and slot_of_eid are required.
 * src == NULL means src[e] = e (membership lists such as atom_to_frag_ids, gat2.py:234).
 * status[0] is set non-zero on the device if an index is out of [0, n_nodes); it is not zeroed here (may be NULL).
 * This is the counting sort of fnb_batch_plan_build run over one graph.  Its kernels index with int32 and stride by
 * up to 148*16*256 = 606208 threads, so n_nodes and the edge count (with self loops) must each be at most
 * 2^31 - 1 - 606208 (FNB_ERR_SIZE otherwise).
 */
size_t fnb_csr_workspace_bytes(int64_t n_nodes, int64_t n_edges_total);
int fnb_csr_build(const int64_t *dst, const int64_t *src, int64_t n_edges, int64_t n_nodes,
                  int append_self_loops, int32_t *rowptr, int32_t *col, int32_t *row, int32_t *eid,
                  int32_t *slot_of_eid, int32_t *rrowptr, int32_t *rslot, int32_t *rdst,
                  void *workspace, size_t workspace_bytes, int32_t *status, void *stream);

/* out[r, 0:width] = in[index[r], 0:width]  -- puts per-edge attributes into CSR slot order. */
int fnb_gather_rows(const float *in, const int32_t *index, int64_t n_rows, int width, float *out,
                    void *stream);

/* offsets[g] = first position i with sorted_ids[i] >= g, g = 0..n_segments (molecule boundaries
 * of the sorted `batch` / `frag_batch` vectors, data.py:896-901). */
int fnb_segment_offsets(const int64_t *sorted_ids, int64_t n, int64_t n_segments, int32_t *offsets,
                        void *stream);

/* int64 -> int32 narrowing of an index vector (atom_to_frag_ids, batch). */
int fnb_narrow_index(const int64_t *in, int64_t n, int32_t *out, void *stream);

/* ---- dense projection with the per-node logit scalars fused into the epilogue ---------------
 * h[n,:] = x[n,:] @ W^T + b          (nn.Linear; projection_{a,b,fb}, gat2.py:142,189,247)
 * S[n,h]   = <h[n,h,:], alpha[h, off_t : off_t+32]>    (target half of the head vector)
 * S[n,4+h] = <h[n,h,:], alpha[h, off_s : off_s+32]>    (source half)
 * x [n_rows,K], W [128,K], b [128], alpha [4,alpha_stride].  S may be NULL.
 */
int fnb_proj_fwd(const float *x, const float *W, const float *b, int64_t n_rows, int K,
                 const float *alpha, int alpha_stride, int off_t, int off_s, float *h, float *S,
                 int precision, void *stream);
/* dx = dh @ W (dx may be NULL); dW = dh^T @ x; db = column sums of dh (may be NULL: fnb_gat_bwd_tiled can emit
 * it for free as d_bias).  scratch: fnb_scratch_bytes(). */
int fnb_proj_bwd(const float *x, const float *W, const float *dh, int64_t n_rows, int K, float *dx,
                 float *dW, float *db, int precision, void *scratch, void *stream);
/* S for features that are not projected (fragment graph: hf = pooled atoms, gat2.py:285). */
int fnb_node_scalars(const float *h, int64_t n_rows, const float *alpha, int alpha_stride,
                     int off_t, int off_s, float *S, void *stream);

/* w[n,h] = sum of p over the edges whose SOURCE is n (gat2.py:165,219,268,312), atomics-free over
 * the reverse CSR.  rslot and p_saved may be NULL for a graph without edges. */
int fnb_attn_by_source(const int32_t *rrowptr, const int32_t *rslot, const float *p_saved,
                       int64_t n_nodes, float *w, void *stream);

/* ---- fused attention block (gat_tiled.cu) --------------------------------------------------------------
 * Forward, gather -> edge logit -> LeakyReLU(0.2) -> segment softmax -> aggregate in one launch
 * (gat2.py:146-169, 196-224, 250-272, 286-316):
 *   z[e,h] = S[t,h] + S_e[e,h] + S[s,4+h];  p = softmax over the slots of t;  out[t] = sum p*h[s]
 * with t, s the destination and source of slot e and S_e the edge term of edge_mode (FNB_EDGE_*).  The affine modes
 * compute their constants from the tiny edge-attribute embedding (App. A.5) in the kernel's prologue:
 *   coef[h*in + k] = sum_j We[j,k] alpha_e[h,j],  coef[4*in + h] = <be, alpha_e[h,:]>   (in = 1 or 6).
 * p_saved [n_edges,4] (slot order; the sign bit carries z>0 for the LeakyReLU derivative) may be NULL for inference.
 * Rows [mask_lo, mask_hi) of out and y are zeroed (bond / frag-bond / atom masks, gat2.py:173-176,227-231,275-278);
 * pass mask_lo = mask_hi = -1 for none.  If next_alpha_e != NULL, also emits
 * next_Se[t,h] = <out[t,:], next_alpha_e[h, 0:128]>, the edge term of the graph whose edges are this graph's nodes
 * (bond -> atom, fbond -> fragment).
 *
 * Backward, destination pass then source pass, both atomics-free.  The destination pass (CSR) writes dz[slot,h], the
 * gradient of the pre-LeakyReLU logit z, and dSt[t,h] = sum of dz over the slots of t (the gradient of S[t,h]).  The
 * source pass (reverse CSR) writes
 *   dh[s] = sum p*dout[t] + dSt[s]*alpha_t + dSs[s]*alpha_s,   dSs[s,h] = sum of dz over the edges leaving s,
 * with alpha_t = alpha[h, off_t:+32], alpha_s = alpha[h, off_s:+32], and the head-vector gradients
 * d_alpha[h, off_t:+32] and d_alpha[h, off_s:+32] (written, not accumulated); the affine modes also write
 * d_alpha[h, off_e:+32], dWe and dbe.  d_bias[128] = column sums of dh (the bias gradient of the projection that
 * produced h), or NULL to skip.  The 128-wide edge slice of TABLE mode is fnb_edge_table_bwd_fused's.
 *
 * Layout (DESIGN.md section 3): a CTA owns up to 64 consecutive destination nodes, logits are computed one thread per
 * edge slot, the softmax one thread per (node, head) in shared memory, the row aggregation one warp per node.
 * Also folded in: the inter-layer ReLU(Dropout(.)) of gat2.py:414-418 (forward epilogue / edge-table backward) and
 * the cross-CTA reduction of every parameter gradient (last CTA to finish; deterministic, no atomics on floats, no
 * second launch).
 * scratch: fnb_scratch_bytes() bytes whose first 256 bytes are ZERO before the first call and are left zero by
 * every call (arrival counters). */
typedef struct fnb_graph {
  int64_t n_nodes, n_edges, n_real_edges; /* n_edges includes appended self loops */
  const int32_t *rowptr, *col, *row, *eid, *slot_of_eid; /* destination-sorted CSR (fnb_csr_build) */
  const int32_t *rrowptr, *rslot, *rdst;                 /* reverse (source-sorted) CSR             */
  const float *edge_attr; /* slot-ordered attributes: [E] (bond graph), [E,6] (fragment-connection graph), else NULL;
                           * like every slot-ordered buffer, may be NULL when E = 0 */
} fnb_graph;

typedef struct fnb_post_act { /* y = ReLU(Dropout_p(out)); RNG counter of element i is offset + i/4 */
  float p;
  int training, relu;
  uint64_t seed, offset;
} fnb_post_act;

typedef struct fnb_gat_fwd_args {
  const float *h, *S;      /* [N,128] projected features, [N,8] logit scalars */
  int edge_mode;           /* FNB_EDGE_* */
  const float *edge_table; /* TABLE: [n_real_edges,4] (may be NULL when n_real_edges = 0) */
  const float *We, *be;    /* AFFINE1/6: edge_attr_{bond,fbond}_embed weight [32,in] and bias [32] (gat2.py:91-92) */
  const float *alpha_e;    /* AFFINE1/6: head vector at its edge slice, rows alpha_stride apart */
  int alpha_stride;
  float *out;              /* [N,128] pre-activation output, may be NULL when only y is wanted */
  float *y;                /* [N,128] ReLU(Dropout(out)) or NULL */
  fnb_post_act post;
  float *p_saved;          /* [E,4] or NULL (inference) */
  int64_t mask_lo, mask_hi;
  const float *next_alpha_e; /* consumer graph's edge slice [4, next_alpha_stride] or NULL */
  int next_alpha_stride;
  float *next_Se;          /* [N,4] */
} fnb_gat_fwd_args;

typedef struct fnb_gat_bwd_args {
  const float *h, *dout, *p_saved;
  int edge_mode;
  const float *We, *be;    /* AFFINE1/6 */
  const float *alpha;      /* full head vector [4, alpha_stride] */
  int alpha_stride, off_t, off_e, off_s;
  float *dz, *dSt;         /* [E,4], [N,4]: outputs of the destination pass, inputs of the source pass */
  float *dh;               /* [N,128] */
  float *d_alpha;          /* [4, alpha_stride]: slices off_t, off_s (and off_e for AFFINE modes) are written */
  float *d_bias;           /* [128] column sums of dh, or NULL */
  float *dWe, *dbe;        /* AFFINE1/6 */
  void *scratch;
} fnb_gat_bwd_args;

int fnb_gat_fwd_tiled(const fnb_graph *g, const fnb_gat_fwd_args *args, void *stream);
/* destination pass then source pass (two launches) */
int fnb_gat_bwd_tiled(const fnb_graph *g, const fnb_gat_bwd_args *args, void *stream);
/* Same two launches with `between_passes` (a cudaEvent_t of the caller, may be NULL) recorded on `stream` after the
 * destination pass: lets a caller time the two passes separately (bench.py's roofline.kernels). */
int fnb_gat_bwd_tiled_marked(const fnb_graph *g, const fnb_gat_bwd_args *args, void *between_passes, void *stream);
/* g_feat[e,:] = g_base[e,:] (if given) + dy[e,:]*(y[e,:]>0)*post_scale (if given) + sum_h dz[slot_of_eid[e],h]*alpha_e[h,:];
 * d_alpha[h, off_e:off_e+128] = sum_e dz[slot_of_eid[e],h] * feat[e,:] */
int fnb_edge_table_bwd_fused(const fnb_graph *g, const float *dz, const float *feat, const float *alpha,
                             int alpha_stride, int off_e, const float *g_base, const float *dy, const float *y,
                             float post_scale, float *g_feat, float *d_alpha, void *scratch, void *stream);

/* ---- whole-encoder programs (encoder.cu) -------------------------------------------------------
 * FragNet.forward (gat2.py:381-442) = n_layers x FragNetLayerA.forward (gat2.py:121-330) with ReLU(Dropout(.)) on the
 * four outputs of every layer, sequenced on the host side of the library so that a forward (backward) pass is ONE
 * call issuing ~7 (~20) launches per layer back to back.  Activations that the backward needs live in a caller
 * allocated workspace whose layout is a pure function of (plan sizes, options).
 *
 * Modes.  post_act = 1: outputs are y = ReLU(Dropout_p(.)) of the last layer (FragNet.forward); the fragment-graph
 * block runs only where run_frag_block says so (its output is dead in all but the last layer, gat2.py:234).
 * post_act = 0 with n_layers = 1: the bare FragNetLayerA.forward -- outputs are the pre-activation tensors.
 */
typedef struct fnb_layer_params {
  const float *Wb, *bb;       /* projection_b  [128,K_bond], [128]   gat2.py:88  */
  const float *Wfb, *bfb;     /* projection_fb [128,K_fbond]         gat2.py:89  */
  const float *We_b, *be_b;   /* edge_attr_bond_embed  [32,1], [32]  gat2.py:91  */
  const float *We_fb, *be_fb; /* edge_attr_fbond_embed [32,6], [32]  gat2.py:92  */
  const float *Wa, *ba;       /* projection_a  [128,K_atom]          gat2.py:95  */
  const float *a_b, *a, *f, *f_a_b; /* head vectors [4,96] [4,192] [4,192] [4,96]  gat2.py:98-107 */
  int K_atom, K_bond, K_fbond;
  /* per-layer switches */
  int run_frag_block;                 /* fragment-graph block (gat2.py:283-316) */
  int want_attention;                 /* emit the four by-source attention sums of this layer */
  int64_t bond_mask, frag_bond_mask;  /* -1 = none; rows [m,m+2) / [2k,2k+2) zeroed (gat2.py:173-176, 275-278) */
  int64_t atom_mask;                  /* -1 = none; row zeroed (gat2.py:227-231) */
  const int32_t *atom_mask_list;      /* optional device list of rows to zero, n_atom_mask entries */
  int64_t n_atom_mask;
  /* list forms of bond_mask / frag_bond_mask: device lists of ROWS of new_bond_features / new_fbond_features to
   * zero (a masked bond m contributes rows m and m+1, a masked fragment link k rows 2k and 2k+1); used by the
   * batched mask attribution, where every replica of a molecule carries its own mask (viz.py:960-984, 1026-1050,
   * 1145-1169 run one batch-1 forward per mask instead) */
  const int32_t *bond_mask_rows;
  int64_t n_bond_mask_rows;
  const int32_t *fbond_mask_rows;
  int64_t n_fbond_mask_rows;
} fnb_layer_params;

typedef struct fnb_layer_grads { /* same shapes as the parameters; every tensor is written (not accumulated) */
  float *Wb, *bb, *Wfb, *bfb, *We_b, *be_b, *We_fb, *be_fb, *Wa, *ba, *a_b, *a, *f, *f_a_b;
} fnb_layer_grads;

typedef struct fnb_batch_plan {
  fnb_graph bond, atom, fbond, frag;
  const int32_t *pool_rowptr, *pool_col; /* fragment -> member atoms (membership CSR of atom_to_frag_ids) */
  const int32_t *a2f;                    /* int32 atom_to_frag_ids */
  int64_t n_atoms, n_frags;
  /* readout (gat2.py:820-821): molecule boundaries of the sorted batch / frag_batch vectors, or NULL */
  const int32_t *mol_atom_ptr, *mol_frag_ptr; /* [n_graphs + 1] */
  const int32_t *batch32, *frag_batch32;      /* int32 copies of batch [Na], frag_batch [Nf] */
  int64_t n_graphs;
  const int32_t *status; /* device word, non-zero if any index was out of range */
} fnb_batch_plan;

/* The batch dict of the reference's collate_fn (fragnet/dataset/data.py:931-948), device pointers.  Edge lists are
 * contiguous int64 [2, E]: row 0 at the pointer, row 1 at pointer + E. */
typedef struct fnb_batch_inputs {
  const int64_t *edge_index;             /* [2, n_bonds]        atom graph: row 0 = source, row 1 = target (gat2.py:187) */
  const int64_t *frag_index;             /* [2, n_fbond_nodes]  fragment graph: row 0 = source, row 1 = target (:283)   */
  const int64_t *atom_to_frag_ids;       /* [n_atoms]                                                              */
  const int64_t *edge_index_bonds_graph; /* [2, n_bond_edges]   bond graph: row 0 = target, row 1 = source (:138)       */
  const int64_t *edge_index_fbonds;      /* [2, n_fbond_edges]  fragment-connection graph: row 0 = target (:239)        */
  const int64_t *batch, *frag_batch;     /* sorted molecule ids of atoms / fragments, or both NULL                     */
  const float *edge_attr_bonds;          /* [n_bond_edges]      cos(theta)                                             */
  const float *edge_attr_fbonds;         /* [n_fbond_edges, 6]                                                         */
  int64_t n_atoms, n_frags, n_bonds, n_bond_edges, n_fbond_nodes, n_fbond_edges, n_graphs;
} fnb_batch_inputs;

/* One call builds everything index-shaped a batch needs (9 launches): the four CSR + reverse CSR plans, the
 * membership CSR, slot-ordered edge attributes, int32 copies and readout offsets.  arena: caller-allocated,
 * 256-byte aligned, fnb_batch_plan_bytes() bytes; the pointers written to *out point into it. */
size_t fnb_batch_plan_bytes(const fnb_batch_inputs *in);
int fnb_batch_plan_build(const fnb_batch_inputs *in, void *arena, size_t arena_bytes, fnb_batch_plan *out,
                         void *stream);

typedef struct fnb_encoder_opts {
  int n_layers;
  int post_act;          /* 1: ReLU(Dropout) between layers and on the outputs; 0: bare layer (n_layers must be 1) */
  float drop_p;
  int training;
  uint64_t seed, offset; /* RNG key / first counter; the call consumes fnb_encoder_rng_span() counters */
  int precision;         /* FNB_PRECISION_* for the dense projections */
  int save_for_backward; /* keep what fnb_encoder_backward needs */
  int need_dx_atoms, need_dx_bond, need_dx_fbond; /* backward: gradients of the layer-0 inputs.  In the forward,
                                                     need_dx_atoms only selects where input dropout runs (its own
                                                     kernel instead of the padding kernel); the backward is right
                                                     whichever values the forward call had */
  int first_trained_layer; /* 0 .. n_layers: layers below it are frozen (finetuning a pretrained encoder).  The
                              forward saves nothing of theirs for the backward (smaller workspaces); the backward
                              does not visit them, and layer first_trained_layer writes its parameter gradients but
                              no input gradient, so dx_* are written only when it is 0 (see need_dx_*).  Dropout
                              counters are the same whatever its value.  0 = train every layer. */
  int pool_frags;          /* gat2_lite (gat2_lite.py:140): no layer runs the fragment block; the last layer writes
                              out_frags = ReLU(Dropout(pool(pre-activation atoms))) at its fragment dropout site, and the
                              backward passes the gradient of out_frags back through the atom graph's pooling.  Needs
                              post_act = 1 and out_frags.  0 = off. */
  int skip_fbond;          /* skip the fragment-connection chain (projection_fb and its attention block) in the forward
                              and the backward: its outputs and parameter gradients are not written, x_fbond is not
                              read.  For variants without that graph (gat2_edge with frag_table, gat2_lite); a layer that
                              runs the fragment block then needs frag_table.  Its dropout counters stay reserved. */
} fnb_encoder_opts;

typedef struct fnb_encoder_io {
  const float *x_atoms, *x_bond, *x_fbond; /* layer-0 inputs [Na,K_atom] [Nb,K_bond] [Nfb,K_fbond] */
  float *out_atoms, *out_frags, *out_bond, *out_fbond; /* [.,128] outputs of the last layer (out_frags may be NULL
                                                          when no layer runs the fragment block) */
  float *attn_atoms, *attn_frags, *attn_bonds, *attn_fbonds; /* [N,4] of the layer with want_attention, or NULL */
  /* backward only */
  const float *g_atoms, *g_frags, *g_bond, *g_fbond; /* gradients of the four outputs; NULL = zero */
  float *dx_atoms, *dx_bond, *dx_fbond;              /* gradients of the layer-0 inputs (see need_dx_*) */
  /* gat2_edge (fragnet/model/gat/gat2_edge.py:139-160): the fragment graph's edge term comes from the connection
   * attributes, <cnx_attr_transform(cnx_attr[e]), f_e[h]>, not from fragment-connection features.  frag_table: that
   * term per real edge, [Ef,4] in edge-id order, read by the layer that runs the fragment block instead of the table
   * the fragment-connection block would emit (NULL = gat2 behaviour); d_frag_table (backward): its gradient. */
  const float *frag_table;
  float *d_frag_table;
} fnb_encoder_io;

size_t fnb_encoder_workspace_bytes(const fnb_batch_plan *plan, const fnb_encoder_opts *opts,
                                   const fnb_layer_params *layers);
size_t fnb_encoder_bwd_workspace_bytes(const fnb_batch_plan *plan, const fnb_encoder_opts *opts,
                                       const fnb_layer_params *layers);
uint64_t fnb_encoder_rng_span(const fnb_batch_plan *plan, const fnb_encoder_opts *opts,
                                 const fnb_layer_params *layers);
int fnb_encoder_forward(const fnb_batch_plan *plan, const fnb_encoder_opts *opts, const fnb_layer_params *layers,
                        const fnb_encoder_io *io, void *workspace, size_t workspace_bytes, void *scratch,
                        void *stream);
/* workspace = the forward call's workspace (unchanged since), bwd_workspace = fnb_encoder_bwd_workspace_bytes().
 * grads: one entry per layer; the entries of layers below first_trained_layer are not read (may be all NULL). */
int fnb_encoder_backward(const fnb_batch_plan *plan, const fnb_encoder_opts *opts, const fnb_layer_params *layers,
                         const fnb_layer_grads *grads, const fnb_encoder_io *io, void *workspace,
                         size_t workspace_bytes, void *bwd_workspace, size_t bwd_workspace_bytes, void *scratch,
                         void *stream);

/* ---- (d) segment-sum pooling ----------------------------------------------------------------
 * out[seg,:] = sum over members (gat2.py:234 atom->fragment via a membership CSR; gat2.py:820-821
 * readout via contiguous offsets: pass col == NULL).  out rows have stride out_stride floats so
 * the readout can write both halves of the [G,256] concatenation in place.  Optional fused S. */
int fnb_segment_sum(const int32_t *rowptr, const int32_t *col, int64_t n_segments, const float *x,
                    float *out, int64_t out_stride, const float *alpha, int alpha_stride, int off_t,
                    int off_s, float *S, void *stream);
/* dx[i,:] = base[i,:] + g[seg_of[i], 0:128] with g row stride g_stride (base NULL = 0; may alias dx). */
int fnb_segment_gather(const float *g, int64_t g_stride, const int32_t *seg_of, int64_t n_rows,
                       const float *base, float *dx, void *stream);

/* ---- fused ReLU(Dropout(x)) (gat2.py:414-418,436-440) ----------------------------------------
 * y = relu(keep(i) ? x/(1-p) : 0), keep from the counter hash of common.cuh (seed, offset + i/4).  p = 0 or
 * training == 0 gives plain ReLU.  relu == 0 gives plain dropout (input features, gat2.py:396). */
int fnb_dropout_relu_fwd(const float *x, float *y, int64_t n, float p, int training, int relu,
                         uint64_t seed, uint64_t offset, void *stream);
/* dx = dy * (y > 0) / (1-p)   (valid for the fused ReLU form; y is the forward output) */
int fnb_dropout_relu_bwd(const float *dy, const float *y, float *dx, int64_t n, float p,
                         int training, void *stream);

/* ---- compact wire format of a batch dict (host -> device staging, dataset/prefetch.py) ----------------------------
 * collate_fn (fragnet/dataset/data.py:877-948) emits one-hot / small-integer feature matrices as fp32 and every index
 * as int64: 32 MB per 1 024-molecule batch on the wire for 11 MB of information.  The compact format ships those
 * matrices as uint8 and the indices as int32; one launch widens every tensor of a batch into the dtypes the reference
 * produces (exact: the host side verifies the round trip before it narrows). */
#define FNB_WIDEN_U8_F32 0  /* uint8 -> float32 */
#define FNB_WIDEN_I32_I64 1 /* int32 -> int64   */
#define FNB_WIDEN_MAX_JOBS 16
typedef struct fnb_widen_job {
  const void *src; /* n elements, 16-byte aligned */
  void *dst;       /* n elements of the wide type, 16-byte aligned */
  int64_t n;
  int mode;        /* FNB_WIDEN_* */
} fnb_widen_job;
int fnb_widen_batch(const fnb_widen_job *jobs, int n_jobs, void *stream);

/* ---- optimizer step over one flat parameter buffer (the trainer's torch.optim.Adam, pretrain_gat2.py:165) -------
 * torch.optim.Adam's update (no amsgrad) on n contiguous fp32 elements in ONE launch; step counts from 1. */
int fnb_adam_step(float *param, const float *grad, float *exp_avg, float *exp_avg_sq, int64_t n, float lr, float beta1,
                  float beta2, float eps, float weight_decay, int64_t step, void *stream);

/* ---- data-parallel step: gradient exchange fused with the optimizer (dist.cu) ---------------------------------------
 * Replaces ncclAllReduce(grad) + grad *= 1/W + Adam (Fabric DDP semantics, finetune_gat2_pl.py:230) by ONE kernel that
 * reads every rank's gradient buffer through NVLink peer mappings, averages in rank order (bitwise identical parameters
 * on every rank, run-to-run deterministic) and updates the local parameters.  grads[r] / flags[r]: rank r's gradient
 * buffer (n floats) and flag row (2*world uint32, zero before first use) as mapped in THIS process (symmetric memory);
 * epoch: a counter that grows by one per call, the same on every rank; done_counter: one device-local uint32, zero
 * before first use.  Every rank must call it once per step. */
#define FNB_MAX_PEERS 8
typedef struct fnb_peer_set {
  const void *grads[FNB_MAX_PEERS];
  void *flags[FNB_MAX_PEERS];
  int world, rank;
} fnb_peer_set;
int fnb_allreduce_adam_step(const fnb_peer_set *peers, float *param, float *exp_avg, float *exp_avg_sq, int64_t n,
                            float lr, float beta1, float beta2, float eps, float weight_decay, int64_t step,
                            uint32_t epoch, void *done_counter, void *stream);
/* The same exchange and update with per-run Adam step counts: runs[0 .. n_runs) tile [0, n) in ascending order
 * (runs[0].first == 0, runs[r].first == runs[r-1].end, the last end == n), and the elements of run r take the bias
 * corrections of runs[r].step.  This is torch.optim.Adam over parameters whose step counts differ (a resumed run whose
 * lower layers were frozen before).  One launch per optimizer step, as fnb_allreduce_adam_step; with one run its result
 * is bitwise that of fnb_allreduce_adam_step.  Returns FNB_ERR_NULL for runs == NULL, FNB_ERR_ALIGN for a run boundary
 * that is not a multiple of 4, FNB_ERR_SIZE for more than FNB_MAX_ADAM_RUNS runs, an empty, overlapping, gapped or
 * short run table or a step < 1; the other arguments as fnb_allreduce_adam_step.  Nothing is launched on an error. */
#define FNB_MAX_ADAM_RUNS 16
typedef struct fnb_adam_run {
  int64_t first, end; /* floats of the flat buffer, multiples of 4 */
  int64_t step;       /* Adam step count of this run's parameters, from 1 */
} fnb_adam_run;
int fnb_allreduce_adam_runs(const fnb_peer_set *peers, float *param, float *exp_avg, float *exp_avg_sq, int64_t n,
                            const fnb_adam_run *runs, int n_runs, float lr, float beta1, float beta2, float eps,
                            float weight_decay, uint32_t epoch, void *done_counter, void *stream);

/* ---- pretraining heads + loss (heads.cu) -------------------------------------------------------------------------
 * PretrainTask.forward (fragnet/model/gat/pretrain_heads.py:64-102) behind one call per direction: bond-length,
 * bond-angle, dihedral heads (Linear 128-64, ReLU, 64-32, ReLU, 32-1; the bond-length head first reduces
 * cat(x_atoms[ei0], x_atoms[ei1], edge_feat) with Linear(384,128) and applies ReLU in FRONT of every linear,
 * pretrain_heads.py:66-74) and the energy head on the graph readout cat(scatter_add(x_atoms, batch),
 * scatter_add(x_frags, frag_batch)) (Linear 256-128, ReLU, 128-64, ReLU, 64-1; pretrain_heads.py:93-100).
 * The wide first layers run on the projection kernels (precision = FNB_PRECISION_*), the narrow tails in FP32. */
typedef struct fnb_mlp3_params { /* nn.Linear weights [out,in] and biases of one three-linear stack */
  const float *W0, *b0, *W1, *b1, *W2, *b2;
} fnb_mlp3_params;
typedef struct fnb_mlp3_grads {
  float *W0, *b0, *W1, *b1, *W2, *b2;
} fnb_mlp3_grads;
typedef struct fnb_pretrain_head_params {
  const float *Wr, *br;        /* bl_reduce_layer [128,384], [128]                         pretrain_heads.py:26 */
  fnb_mlp3_params bl, ba, da;  /* bl_layers / ba_layers / da_layers: [64,128] [32,64] [1,32]   :27-47 */
  fnb_mlp3_params fc;          /* FC_layers: [128,256] [64,128] [1,64]                         :50-55 */
} fnb_pretrain_head_params;
typedef struct fnb_pretrain_head_grads { /* every tensor of ba, da, fc is written; the bond-length head has no
                                            backward here (the reference's loss never uses it: pretrain_utils.py:24
                                            overwrites loss_lngth), Wr / br / bl are ignored */
  float *Wr, *br;
  fnb_mlp3_grads bl, ba, da, fc;
} fnb_pretrain_head_grads;
typedef struct fnb_pretrain_head_io {
  const float *x_atoms, *x_frags, *edge_feat; /* encoder outputs [Na,128] [Nf,128] [Ea,128] */
  const int64_t *edge_index;                  /* [2,Ea] int64 (batch["edge_index"]) */
  const int32_t *mol_atom_ptr, *mol_frag_ptr; /* [G+1] molecule boundaries (fnb_batch_plan) */
  const int32_t *batch32, *frag_batch32;      /* [Na], [Nf] molecule of every atom / fragment (backward only) */
  int64_t n_atoms, n_frags, n_edges, n_graphs;
  float *bond_length, *bond_angle, *dihedral, *energy; /* [Ea] [Na] [Ea] [G]; bond_length == NULL skips that head */
  /* backward */
  const float *g_bond_angle, *g_dihedral, *g_energy; /* gradients of the three trained outputs */
  float *g_atoms, *g_frags, *g_edge;                 /* [Na,128] [Nf,128] [Ea,128], written */
} fnb_pretrain_head_io;

size_t fnb_pretrain_heads_workspace_bytes(int64_t n_atoms, int64_t n_edges, int64_t n_graphs);
size_t fnb_pretrain_heads_bwd_workspace_bytes(int64_t n_atoms, int64_t n_edges, int64_t n_graphs);
int fnb_pretrain_heads_forward(const fnb_pretrain_head_params *params, const fnb_pretrain_head_io *io, int precision,
                               void *workspace, size_t workspace_bytes, void *scratch, void *stream);
/* workspace = the forward call's workspace (unchanged since). */
int fnb_pretrain_heads_backward(const fnb_pretrain_head_params *params, const fnb_pretrain_head_grads *grads,
                                const fnb_pretrain_head_io *io, int precision, void *workspace, size_t workspace_bytes,
                                void *bwd_workspace, size_t bwd_workspace_bytes, void *scratch, void *stream);

/* loss[0] = sum_t weight_t * mean((pred_t - target_t)^2) over up to 4 terms, and (grad != NULL) its gradient
 * grad_t[i] = 2 weight_t / n_t * (pred_t[i] - target_t[i]), in one launch.  The pretraining loop's loss
 * (fragnet/train/pretrain/pretrain_utils.py:22-26) is dihedral x 2, bond angle x 1, energy x 1. */
typedef struct fnb_mse_term {
  const float *pred, *target;
  int64_t n;
  float weight;
  float *grad;
} fnb_mse_term;
int fnb_mse_sum_loss(const fnb_mse_term *terms, int n_terms, float *loss, void *scratch, void *stream);

/* ---- one pretraining step (step.cu) ------------------------------------------------------------------------------
 * The body of Trainer.train (fragnet/train/pretrain/pretrain_utils.py:12-30) for one batch as ONE call: on-device
 * collate of the batch dict, FragNet.forward, PretrainTask.forward, the loss 2*MSE(dihedral) + MSE(bond angle) +
 * MSE(energy) and, with backward != 0, every parameter gradient (written, not accumulated).  The optimizer update is
 * fnb_adam_step on the caller's flat buffers (a gradient all-reduce can sit in between). */
typedef struct fnb_pretrain_step_args {
  fnb_batch_inputs batch;                         /* index tensors and sizes; n_graphs = molecules = len(y);
                                                     batch / frag_batch are required */
  const float *x_atoms, *x_bond, *x_fbond;        /* [Na,K_atom] [Nb,K_bond] [Nfb,K_fbond] raw features */
  const float *t_bond_angle, *t_dihedral, *t_energy; /* targets bnd_angl [Na], dh_angl [Nb], y [G] */
  int n_layers;
  const fnb_layer_params *layers;                 /* run_frag_block: 1 for the last layer only (gat2.py:234) */
  const fnb_layer_grads *layer_grads;             /* f may be NULL where the fragment block does not run */
  const fnb_pretrain_head_params *heads;
  const fnb_pretrain_head_grads *head_grads;
  float drop_p;
  int training;
  uint64_t seed, offset;                          /* dropout RNG key / first counter (fnb_pretrain_step_rng_span) */
  int precision;
  int backward;                                   /* 0: forward + loss only (validation) */
  float *loss;                                    /* device scalar */
  float *bond_length, *bond_angle, *dihedral, *energy; /* optional prediction outputs; bond_length NULL = head skipped */
  const void *plan_arena;                         /* NULL, or the arena fnb_pretrain_plan_prefetch() filled for exactly this
                                                     `batch` (same pointers and sizes): the step skips its own collate */
} fnb_pretrain_step_args;
size_t fnb_pretrain_step_workspace_bytes(const fnb_pretrain_step_args *args);
uint64_t fnb_pretrain_step_rng_span(const fnb_pretrain_step_args *args);
/* workspace: 256-byte aligned, fnb_pretrain_step_workspace_bytes() bytes. */
int fnb_pretrain_step(const fnb_pretrain_step_args *args, void *workspace, size_t workspace_bytes, void *scratch,
                      void *stream);
/* On-device collate of the NEXT batch ahead of its step, on a library stream, underneath the step that is running: a
 * training loop knows its next batch (DataLoader prefetch), and the plan depends on nothing but the batch's index
 * tensors.  arena: fnb_batch_plan_bytes(next) bytes, 256-byte aligned, not the arena of the plan the running step uses
 * (alternate between two).  batch_ready: a cudaEvent_t after which the tensors of `next` are complete, or NULL if they
 * already are.  The build starts once the encoder forward of the step launched last is complete (underneath its heads
 * and backward), i.e. after the last user of this arena when two arenas alternate.  The next fnb_pretrain_step takes the
 * result through args->plan_arena.  Returns FNB_ERR_MODE
 * when the library runs single-stream (FNB_STREAMS=1): nothing was queued, build inside the step as usual. */
int fnb_pretrain_plan_prefetch(const fnb_batch_inputs *next, void *arena, size_t arena_bytes, void *batch_ready);

/* ---- one finetuning step (finetune.cu, step.cu) -------------------------------------------------------------------
 * The body of TrainerFineTune.train_regr / train_clsf_bce (fragnet/train/utils.py:330-385, :406-470) for a
 * FragNetFineTune model (gat2.py:758-826) as ONE call: on-device collate, FragNet.forward, the graph readout
 * cat(sum atoms, sum fragments), the FTHead, the loss and, with backward != 0, every parameter gradient (written, not
 * accumulated).  The optimizer update is fnb_adam_step on the caller's flat buffers.
 *
 * The head is a list of linear layers, each  y = act(drop_out(drop_in(x) W^T + b)), in exact FP32 in every precision
 * mode.  drop_in covers FTHead1 / FTHead4 (dropout in front of a linear, gat2.py:580-588, :669-675), drop_out FTHead2 /
 * FTHead3 (dropout between a linear and its activation, :719-725, :745-751).  The last layer is a bare linear
 * (act = FNB_ACT_NONE, p_out = 0); its out_dim is the number of classes. */
#define FNB_ACT_NONE 0
#define FNB_ACT_RELU 1
#define FNB_ACT_CELU 2      /* alpha = 1 */
#define FNB_ACT_SILU 3
#define FNB_ACT_GELU 4      /* exact (erf) form */
#define FNB_ACT_SELU 5
#define FNB_ACT_RELU6 6
#define FNB_ACT_LEAKYRELU 7 /* negative slope 0.01 */
#define FNB_MLP_MAX_LAYERS 8
typedef struct fnb_mlp_layer {
  const float *W, *b;  /* nn.Linear weight [out,in] and bias [out] */
  float *dW, *db;      /* their gradients (backward only; written).  Both NULL: the layer is frozen -- no weight
                          gradient is formed, and its input gradient only where a trained layer lies below it or the
                          encoder trains */
  int in_dim, out_dim; /* any positive widths; in_dim of layer 0 = 2 * FNB_D (the readout), of layer l = out_dim of l-1 */
  float p_in, p_out;   /* dropout probability on the layer's input / on its pre-activation output; 0 = none */
  int act;             /* FNB_ACT_* */
} fnb_mlp_layer;

#define FNB_LOSS_MSE 0        /* nn.MSELoss over the flattened predictions (train_regr)                        */
#define FNB_LOSS_BCE_MASKED 1 /* BCE-with-logits over the labels > -0.5, divided by their count (train_clsf_bce) */

/* Dropout counters: the encoder's sites as fnb_encoder_rng_span lays them out from `offset`, then the head's, in layer
 * order (a layer's input site, then its output site; a site exists where its p is non-zero), each a contiguous block
 * of ceil(G * width / 4) counters over the row-major [G, width] tensor.
 *
 * Model versions (`variant`).  The step builds the batch plan from `batch` with the graphs the variant lacks emptied,
 * and the encoder sites follow from those sizes (input; then per layer bond, atom, fragment-connection, fragment):
 *   FNB_VARIANT_GAT2  gat2.  Sites over (Na, Nb, n_fbond_nodes, Nf) rows.
 *   FNB_VARIANT_LITE  gat2_lite (bond graph, atom graph, pooling).  No fragment-connection graph (n_fbond_nodes and
 *                     n_fbond_edges are taken as 0, so the fragment graph has no edges) and no fragment block: the
 *                     last layer's fragment site covers ReLU(Dropout(pool(atoms))).  Sites over (Na, Nb, 0, Nf) rows.
 *                     (The autograd gat2_lite path draws its last layer's three sites in separate blocks.)
 *   FNB_VARIANT_EDGE  gat2_edge.  The fragment graph's edge term is <cnx_attr_transform(cnx_attr[e]), f_e[h]> of the
 *                     last layer (formed on the device); the fragment-connection graph keeps its n_fbond_nodes nodes
 *                     (one per fragment edge) but has no edges (n_fbond_edges is taken as 0) and its chain is skipped;
 *                     its sites stay reserved, exactly as in the autograd gat2_edge call.  Sites over (Na, Nb,
 *                     n_fbond_nodes, Nf) rows.
 * In every variant the layers' fragment-connection tensors (Wfb, bfb, We_fb, be_fb, f_a_b) are read only by GAT2, and
 * x_fbond may be NULL for LITE and EDGE. */
#define FNB_VARIANT_GAT2 0
#define FNB_VARIANT_LITE 1
#define FNB_VARIANT_EDGE 2
typedef struct fnb_finetune_step_args {
  fnb_batch_inputs batch;                   /* as fnb_pretrain_step_args.batch; n_graphs = G molecules */
  const float *x_atoms, *x_bond, *x_fbond;  /* [Na,K_atom] [Nb,K_bond] [Nfb,K_fbond] raw features */
  const float *target;                      /* y: [G * n_classes] (labels < -0.5 are missing with FNB_LOSS_BCE_MASKED) */
  int n_layers;
  const fnb_layer_params *layers;           /* run_frag_block: 1 for the last layer only */
  const fnb_layer_grads *layer_grads;
  int n_head_layers;                        /* 1 .. FNB_MLP_MAX_LAYERS */
  const fnb_mlp_layer *head;
  int loss_kind;                            /* FNB_LOSS_* */
  float drop_p;                             /* the encoder's dropout (the head layers carry their own) */
  int training;
  uint64_t seed, offset;                    /* dropout RNG key / first counter (fnb_finetune_step_rng_span) */
  int precision;                            /* FNB_PRECISION_* of the encoder; the head is FP32 in every mode */
  int backward;                             /* 0: forward + loss only */
  float *loss;                              /* device scalar */
  float *predictions;                       /* optional [G, n_classes] output */
  const void *plan_arena;                   /* NULL, or an arena fnb_pretrain_plan_prefetch() filled for `batch` */
  int first_trained_layer;                  /* 0 .. n_layers (else FNB_ERR_SIZE): encoder layers below it are frozen,
                                               as fnb_encoder_opts.first_trained_layer; their layer_grads entries may
                                               be NULL.  n_layers freezes the encoder: no encoder backward, no readout
                                               backward, layer_grads may be NULL.  A backward that trains nothing
                                               (this at n_layers and every head layer frozen) is FNB_ERR_MODE. */
  /* zero = gat2, exactly as without these fields */
  int variant;                              /* FNB_VARIANT_* (else FNB_ERR_MODE); run_frag_block: 0 in every layer for
                                               LITE, the last layer only otherwise */
  const float *cnx_attr;                    /* EDGE: [n_fbond_nodes, 8] connection attributes, frag_index edge order */
  const float *W_cnx, *b_cnx;               /* EDGE: cnx_attr_transform of the LAST layer, [128, 8], [128] */
  float *dW_cnx, *db_cnx;                   /* EDGE: their gradients (written, with the edge slice f[:, 32:160] of the
                                               last layer's f gradient); NULL when the last encoder layer is frozen */
} fnb_finetune_step_args;
size_t fnb_finetune_step_workspace_bytes(const fnb_finetune_step_args *args);
uint64_t fnb_finetune_step_rng_span(const fnb_finetune_step_args *args);
/* workspace: 256-byte aligned, fnb_finetune_step_workspace_bytes() bytes; scratch: fnb_scratch_bytes(). */
int fnb_finetune_step(const fnb_finetune_step_args *args, void *workspace, size_t workspace_bytes, void *scratch,
                      void *stream);

/* ---- device-side batch assembly from a packed dataset arena (arena.cu) ---------------------------
 * Replaces, for a dataset resident in device memory, collate_fn / collate_fn_pt (fragnet/dataset/data.py:877-948,
 * :951-1032), the node-count offsets of get_incr_* (data.py:11-113) and the per-tensor batch[k].to(device) of the
 * training loops (train/pretrain/pretrain_utils.py:13-14, train/utils.py:335-336): the only per-step host -> device
 * traffic is the list of molecule ids.
 *
 * The arena stores every batch tensor as the concatenation over ALL molecules of the dataset (4-byte elements; index
 * tensors molecule-local int32, one flat array per index row).  A kind is a row-count space: counts[mol] rows per
 * molecule and prefix[mol] = exclusive prefix sum of counts over the dataset (both device arrays of n_mols entries).
 * A job emits one output tensor (or one row of a [2,E] index tensor) for the molecules mol_ids[0..n_batch):
 *   FNB_ARENA_COPY32  dst[rows, width] 4-byte elements copied from src
 *   FNB_ARENA_INDEX   dst[rows] int64 = src[rows] int32 (molecule-local) + number of `offset_kind` rows of the
 *                     molecules before it in this batch (integer arithmetic: no 2^24 ceiling, cf. data.py:883)
 *   FNB_ARENA_FILL    dst[rows] int64 = position of the molecule in the batch (`batch`, `frag_batch`)
 * The caller sizes dst from host copies of the counts; a molecule id outside [0, n_mols) contributes no rows and sets
 * *status (optional device int32) to 1. */
#define FNB_ARENA_MAX_KINDS 24
#define FNB_ARENA_MAX_JOBS 32
#define FNB_ARENA_COPY32 0
#define FNB_ARENA_INDEX 1
#define FNB_ARENA_FILL 2
typedef struct fnb_arena_kind {
  const int32_t *counts;
  const int64_t *prefix;
} fnb_arena_kind;
typedef struct fnb_arena_job {
  const void *src;
  void *dst;
  int32_t kind;
  int32_t offset_kind;   /* FNB_ARENA_INDEX only */
  int32_t width;         /* FNB_ARENA_COPY32: elements per row */
  int32_t mode;
} fnb_arena_job;
size_t fnb_arena_workspace_bytes(int64_t n_batch, int n_kinds);
/* kinds / jobs are HOST arrays (copied into the launch parameters); workspace is 16-byte aligned device memory. */
int fnb_arena_assemble(const int64_t *mol_ids, int64_t n_batch, int64_t n_mols, const fnb_arena_kind *kinds,
                       int n_kinds, const fnb_arena_job *jobs, int n_jobs, void *workspace, size_t workspace_bytes,
                       int32_t *status, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* FRAGNET_B200_H */
