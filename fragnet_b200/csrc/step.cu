// One pretraining step as ONE library call: on-device collate, encoder forward, heads, loss, heads backward, encoder
// backward -- the body of the reference's Trainer.train loop (fragnet/train/pretrain/pretrain_utils.py:12-30:
// model(batch) -> four MSE terms -> loss.backward()) without a Python boundary between the ~150 launches.
//
// Why: at batch 1024 the device needs ~2.2 ms for the step and the host needed ~2.4 ms to ENQUEUE it through
// autograd.Function / ctypes round trips (profiles/r1o_host_profile.log); issued from here the same launches cost
// ~3 us each.  Everything lives in one caller-provided workspace whose layout is a pure function of the batch sizes.
// The optimizer update (fnb_adam_step over the flat parameter buffer) and, with several GPUs, the gradient
// all-reduce stay separate calls so that NCCL can sit between them.
#include "common.cuh"

namespace {

// Sizes-only view of the plan a batch will get (what the workspace-size functions of the sub-programs read).
fnb_batch_plan sizes_plan(const fnb_batch_inputs *in) {
  fnb_batch_plan p{};
  p.bond.n_nodes = in->n_bonds;        p.bond.n_edges = in->n_bond_edges;            p.bond.n_real_edges = in->n_bond_edges;
  p.atom.n_nodes = in->n_atoms;        p.atom.n_edges = in->n_bonds + in->n_atoms;   p.atom.n_real_edges = in->n_bonds;
  p.fbond.n_nodes = in->n_fbond_nodes; p.fbond.n_edges = in->n_fbond_edges;          p.fbond.n_real_edges = in->n_fbond_edges;
  p.frag.n_nodes = in->n_frags;        p.frag.n_edges = in->n_fbond_nodes;           p.frag.n_real_edges = in->n_fbond_nodes;
  p.n_atoms = in->n_atoms; p.n_frags = in->n_frags; p.n_graphs = in->n_graphs;
  return p;
}

// the encoder options of a step (fnb_pretrain_step_args and fnb_finetune_step_args name these fields alike)
template <class StepArgs>
fnb_encoder_opts opts_of(const StepArgs *a) {
  fnb_encoder_opts o{};
  o.n_layers = a->n_layers; o.post_act = 1; o.drop_p = a->drop_p; o.training = a->training; o.seed = a->seed;
  o.offset = a->offset; o.precision = a->precision; o.save_for_backward = a->backward ? 1 : 0;
  return o;
}

struct StepBufs {
  char *plan_arena; size_t plan_bytes;
  char *enc_ws; size_t enc_bytes;
  char *head_ws; size_t head_bytes;
  char *head_bws; size_t head_bws_bytes;
  char *enc_bws; size_t enc_bws_bytes;
  float *out_atoms, *out_frags, *out_bond, *out_fbond;
  float *bond_angle, *dihedral, *energy;
  float *d_bond_angle, *d_dihedral, *d_energy;
  float *g_atoms, *g_frags, *g_edge;
};

bool args_ok(const fnb_pretrain_step_args *a) {
  return a && a->n_layers >= 1 && a->n_layers <= 16 && a->layers && a->heads && a->batch.n_atoms >= 0 &&
         a->batch.n_frags >= 0 && a->batch.n_bonds >= 0 && a->batch.n_graphs >= 0;
}

size_t step_layout(const fnb_pretrain_step_args *a, char *base, StepBufs *out) {
  const fnb_batch_inputs *in = &a->batch;
  const fnb_batch_plan sp = sizes_plan(in);
  const fnb_encoder_opts o = opts_of(a);
  const int64_t Na = in->n_atoms, Nf = in->n_frags, Nb = in->n_bonds, Nfb = in->n_fbond_nodes, G = in->n_graphs;
  Arena ar{base, 0};
  StepBufs b{};
  b.plan_bytes = fnb_batch_plan_bytes(in);
  b.plan_arena = ar.bytes(b.plan_bytes);
  b.enc_bytes = fnb_encoder_workspace_bytes(&sp, &o, a->layers);
  b.enc_ws = ar.bytes(b.enc_bytes);
  b.head_bytes = fnb_pretrain_heads_workspace_bytes(Na, Nb, G);
  b.head_ws = ar.bytes(b.head_bytes);
  b.out_atoms = ar.take<float>(Na * kD); b.out_frags = ar.take<float>(Nf * kD);
  b.out_bond = ar.take<float>(Nb * kD);  b.out_fbond = ar.take<float>(Nfb * kD);
  b.bond_angle = ar.take<float>(Na); b.dihedral = ar.take<float>(Nb); b.energy = ar.take<float>(G);
  if (a->backward) {
    b.d_bond_angle = ar.take<float>(Na); b.d_dihedral = ar.take<float>(Nb); b.d_energy = ar.take<float>(G);
    b.g_atoms = ar.take<float>(Na * kD); b.g_frags = ar.take<float>(Nf * kD); b.g_edge = ar.take<float>(Nb * kD);
    b.head_bws_bytes = fnb_pretrain_heads_bwd_workspace_bytes(Na, Nb, G);
    b.head_bws = ar.bytes(b.head_bws_bytes);
    b.enc_bws_bytes = fnb_encoder_bwd_workspace_bytes(&sp, &o, a->layers);
    b.enc_bws = ar.bytes(b.enc_bws_bytes);
  }
  if (out) *out = b;
  return ar.total();
}

// The first half of both step programs: the on-device collate of the batch (north-star kernel a) and the encoder
// forward (FragNet.forward, gat2.py:381-442).  The collate runs on an auxiliary stream, underneath the plan-independent
// head of the forward pass (input dropout, operand padding, layer-0 projections), or was done ahead of the step by
// fnb_pretrain_plan_prefetch (`prefetched`: its arena, on its own stream, underneath the previous step).
int collate_and_encode(const fnb_batch_inputs *in, const void *prefetched, char *plan_arena, size_t plan_bytes,
                       const fnb_encoder_opts *o, const fnb_layer_params *layers, const fnb_encoder_io *eio,
                       char *enc_ws, size_t enc_bytes, void *scratch, void *stream, const FnbAux &aux, bool two,
                       fnb_batch_plan *plan_out) {
  fnb_batch_plan plan{};
  cudaEvent_t plan_ready = nullptr, plan_complete = nullptr;
  if (two && prefetched) {
    RC(fnb_batch_plan_view(in, const_cast<void *>(prefetched), fnb_batch_plan_bytes(in), &plan));
    plan_ready = aux.p_fwd;
    plan_complete = aux.p_done;
  } else if (two) {
    cudaStream_t s = (cudaStream_t)stream;
    RC((int)cudaEventRecord(aux.ready[1], s));               // the batch tensors are complete on the caller's stream
    RC((int)cudaStreamWaitEvent(aux.wstream, aux.ready[1], 0));
    RC(fnb_batch_plan_build_impl(in, plan_arena, plan_bytes, &plan, (void *)aux.wstream, aux.plan_fwd));
    RC((int)cudaEventRecord(aux.wjoin, aux.wstream));
    plan_ready = aux.plan_fwd;       // forward CSRs: what the first attention kernels wait for
    plan_complete = aux.wjoin;       // + reverse CSRs, per-molecule arrays: waited for behind those kernels
  } else {
    RC(fnb_batch_plan_build(in, plan_arena, plan_bytes, &plan, stream));
  }
  RC(fnb_encoder_forward_impl(&plan, o, layers, eio, enc_ws, enc_bytes, scratch, stream, plan_ready, plan_complete));
  // the collate of the next batch (fnb_pretrain_plan_prefetch) starts here: underneath the heads, where one or two
  // kernels are in flight, rather than underneath the forward, whose chains it slowed (gpurun_out/r5q)
  if (two) RC((int)cudaEventRecord(aux.step_begin, (cudaStream_t)stream));
  *plan_out = plan;
  return 0;
}

}  // namespace

extern "C" size_t fnb_pretrain_step_workspace_bytes(const fnb_pretrain_step_args *a) {
  if (!args_ok(a)) return 0;
  return step_layout(a, nullptr, nullptr);
}

extern "C" uint64_t fnb_pretrain_step_rng_span(const fnb_pretrain_step_args *a) {
  if (!args_ok(a)) return 0;
  const fnb_batch_plan sp = sizes_plan(&a->batch);
  const fnb_encoder_opts o = opts_of(a);
  return fnb_encoder_rng_span(&sp, &o, a->layers);
}

extern "C" int fnb_pretrain_step(const fnb_pretrain_step_args *a, void *workspace, size_t workspace_bytes, void *scratch,
                                 void *stream) {
  if (!a || !workspace || !scratch) return FNB_ERR_NULL;
  if (!args_ok(a)) return FNB_ERR_SIZE;
  if (!a->loss || !a->x_atoms || !a->x_bond || !a->x_fbond || !a->t_bond_angle || !a->t_dihedral || !a->t_energy)
    return FNB_ERR_NULL;
  if (a->backward && (!a->layer_grads || !a->head_grads)) return FNB_ERR_NULL;
  const fnb_batch_inputs *in = &a->batch;
  // every loss term needs at least one element (nn.MSELoss of an empty tensor is NaN upstream)
  if (in->n_atoms < 1 || in->n_bonds < 1 || in->n_graphs < 1 || !in->batch || !in->frag_batch) return FNB_ERR_SIZE;
  if (reinterpret_cast<uintptr_t>(workspace) & 255u) return FNB_ERR_ALIGN;
  StepBufs B;
  if (step_layout(a, (char *)workspace, &B) > workspace_bytes) return FNB_ERR_WORKSPACE;

  FnbAux aux{};
  const bool two = fnb_aux_streams(&aux) == 0;
  fnb_batch_plan plan{};
  fnb_encoder_opts o = opts_of(a);
  fnb_encoder_io eio{};
  eio.x_atoms = a->x_atoms; eio.x_bond = a->x_bond; eio.x_fbond = a->x_fbond;
  eio.out_atoms = B.out_atoms; eio.out_frags = B.out_frags; eio.out_bond = B.out_bond; eio.out_fbond = B.out_fbond;
  RC(collate_and_encode(in, a->plan_arena, B.plan_arena, B.plan_bytes, &o, a->layers, &eio, B.enc_ws, B.enc_bytes,
                        scratch, stream, aux, two, &plan));
  // ---- heads (PretrainTask.forward, pretrain_heads.py:64-102)
  fnb_pretrain_head_io hio{};
  hio.x_atoms = B.out_atoms; hio.x_frags = B.out_frags; hio.edge_feat = B.out_bond; hio.edge_index = in->edge_index;
  hio.mol_atom_ptr = plan.mol_atom_ptr; hio.mol_frag_ptr = plan.mol_frag_ptr; hio.batch32 = plan.batch32;
  hio.frag_batch32 = plan.frag_batch32;
  hio.n_atoms = in->n_atoms; hio.n_frags = in->n_frags; hio.n_edges = in->n_bonds; hio.n_graphs = in->n_graphs;
  hio.bond_length = a->bond_length;
  hio.bond_angle = a->bond_angle ? a->bond_angle : B.bond_angle;
  hio.dihedral = a->dihedral ? a->dihedral : B.dihedral;
  hio.energy = a->energy ? a->energy : B.energy;
  // Training without prediction outputs: the tails' forward, the loss and the gradients of the predictions are formed
  // inside the backward tails (fused loss) -- three launches and one synchronisation point between the heads fewer.
  const bool fuse_loss = a->backward && !a->bond_length && !a->bond_angle && !a->dihedral && !a->energy;
  RC(fnb_pretrain_heads_forward_impl(a->heads, &hio, a->precision, B.head_ws, B.head_bytes, scratch, stream, fuse_loss));
  // ---- loss (pretrain_utils.py:22-26): 2 x dihedral + bond angle + energy, and the gradients of the predictions
  fnb_mse_term terms[3];
  terms[0].pred = hio.dihedral;   terms[0].target = a->t_dihedral;   terms[0].n = in->n_bonds;  terms[0].weight = 2.f;
  terms[1].pred = hio.bond_angle; terms[1].target = a->t_bond_angle; terms[1].n = in->n_atoms;  terms[1].weight = 1.f;
  terms[2].pred = hio.energy;     terms[2].target = a->t_energy;     terms[2].n = in->n_graphs; terms[2].weight = 1.f;
  terms[0].grad = B.d_dihedral; terms[1].grad = B.d_bond_angle; terms[2].grad = B.d_energy;
  if (!fuse_loss) RC(fnb_mse_sum_loss(terms, 3, a->loss, scratch, stream));
  if (!a->backward) return 0;
  // ---- backward: heads, then the encoder
  hio.g_dihedral = B.d_dihedral; hio.g_bond_angle = B.d_bond_angle; hio.g_energy = B.d_energy;
  hio.g_atoms = B.g_atoms; hio.g_frags = B.g_frags; hio.g_edge = B.g_edge;
  const fnb_mse_term fused[3] = {terms[1], terms[0], terms[2]};   // bond angle, dihedral, energy
  // (the heads' weight gradients keep running on the auxiliary streams; the encoder backward ends by joining them)
  RC(fnb_pretrain_heads_backward_impl(a->heads, a->head_grads, &hio, a->precision, B.head_ws, B.head_bytes, B.head_bws,
                                      B.head_bws_bytes, scratch, stream, 1, fuse_loss ? fused : nullptr, a->loss));
  eio.g_atoms = B.g_atoms; eio.g_frags = B.g_frags; eio.g_bond = B.g_edge; eio.g_fbond = nullptr;
  RC(fnb_encoder_backward(&plan, &o, a->layers, a->layer_grads, &eio, B.enc_ws, B.enc_bytes, B.enc_bws, B.enc_bws_bytes,
                          scratch, stream));
  if (two) RC((int)cudaStreamWaitEvent((cudaStream_t)stream, aux.h_done, 0));   // energy head's first-layer weight gradient
  return 0;
}

extern "C" int fnb_pretrain_plan_prefetch(const fnb_batch_inputs *next, void *arena, size_t arena_bytes, void *batch_ready) {
  if (!next || !arena) return FNB_ERR_NULL;
  if (!next->batch || !next->frag_batch) return FNB_ERR_SIZE;
  FnbAux aux{};
  if (fnb_aux_streams(&aux) != 0) return FNB_ERR_MODE;
  // Starts once the encoder forward of the step launched last is complete (aux.step_begin is recorded there): by then
  // the arena's previous tenant -- the step before that one, two arenas alternate -- is long finished.
  RC((int)cudaStreamWaitEvent(aux.pstream, aux.step_begin, 0));
  if (batch_ready) RC((int)cudaStreamWaitEvent(aux.pstream, (cudaEvent_t)batch_ready, 0));
  fnb_batch_plan plan{};
  RC(fnb_batch_plan_build_impl(next, arena, arena_bytes, &plan, (void *)aux.pstream, aux.p_fwd));
  RC((int)cudaEventRecord(aux.p_done, aux.pstream));
  return 0;
}


// ---------------------------------------------------------------------------------------------------------------------
// One finetuning step (TrainerFineTune.train_regr / train_clsf_bce, fragnet/train/utils.py:330-470, on FragNetFineTune):
// collate, encoder forward, readout cat(sum atoms, sum fragments) (gat2.py:820-823), FTHead forward, loss, FTHead
// backward, readout backward, encoder backward -- in stream order on the caller's stream, the encoder's own forks aside.
namespace {

bool ft_args_ok(const fnb_finetune_step_args *a) {
  return a && a->variant >= FNB_VARIANT_GAT2 && a->variant <= FNB_VARIANT_EDGE && a->n_layers >= 1 && a->n_layers <= 16 && a->layers && a->batch.n_atoms >= 0 && a->batch.n_frags >= 0 &&
         a->batch.n_bonds >= 0 && a->batch.n_graphs >= 1 && a->first_trained_layer >= 0 &&
         a->first_trained_layer <= a->n_layers && fnb_mlp_check(a->head, a->n_head_layers, a->batch.n_graphs, 2 * kD, 0) == 0;
}

// Layers 0 .. first_trained_layer - 1 of the encoder are frozen; first_trained_layer == n_layers freezes all of it: the
// forward then saves nothing and the backward ends in the head.
bool encoder_trained(const fnb_finetune_step_args *a) { return a->first_trained_layer < a->n_layers; }

fnb_encoder_opts ft_opts_of(const fnb_finetune_step_args *a) {
  fnb_encoder_opts o = opts_of(a);
  o.first_trained_layer = a->first_trained_layer;
  o.save_for_backward = a->backward && encoder_trained(a);
  o.pool_frags = a->variant == FNB_VARIANT_LITE;
  o.skip_fbond = a->variant != FNB_VARIANT_GAT2;
  return o;
}

// The batch as the variant sees it (fnb_finetune_step_args.variant): the graphs it lacks are emptied.
fnb_batch_inputs ft_inputs(const fnb_finetune_step_args *a) {
  fnb_batch_inputs in = a->batch;
  if (a->variant != FNB_VARIANT_GAT2) in.n_fbond_edges = 0;
  if (a->variant == FNB_VARIANT_LITE) in.n_fbond_nodes = 0;
  return in;
}

struct FtBufs {
  char *plan_arena; size_t plan_bytes;
  char *enc_ws; size_t enc_bytes;
  char *enc_bws; size_t enc_bws_bytes;
  float *out_atoms, *out_frags, *out_bond, *out_fbond;
  float *readout, *xd0, *pred;
  float *xd[FNB_MLP_MAX_LAYERS], *u[FNB_MLP_MAX_LAYERS], *dz[FNB_MLP_MAX_LAYERS];
  float *d_readout, *g_atoms, *g_frags, *rec;
  float *cnx_table, *d_cnx_table;   // EDGE: the fragment graph's edge term [Ef,4] and its gradient
};

size_t ft_layout(const fnb_finetune_step_args *a, char *base, FtBufs *out) {
  const fnb_batch_inputs in_v = ft_inputs(a), *in = &in_v;
  const fnb_batch_plan sp = sizes_plan(in);
  const fnb_encoder_opts o = ft_opts_of(a);
  const bool enc = a->backward && encoder_trained(a);
  const int64_t Na = in->n_atoms, Nf = in->n_frags, Nb = in->n_bonds, Nfb = in->n_fbond_nodes, G = in->n_graphs;
  const fnb_mlp_layer *L = a->head;
  const int n = a->n_head_layers;
  Arena ar{base, 0};
  FtBufs b{};
  b.plan_bytes = fnb_batch_plan_bytes(in);
  b.plan_arena = ar.bytes(b.plan_bytes);
  b.enc_bytes = fnb_encoder_workspace_bytes(&sp, &o, a->layers);
  b.enc_ws = ar.bytes(b.enc_bytes);
  b.out_atoms = ar.take<float>(Na * kD); b.out_frags = ar.take<float>(Nf * kD);
  b.out_bond = ar.take<float>(Nb * kD);  b.out_fbond = ar.take<float>(Nfb * kD);
  b.readout = ar.take<float>(G * 2 * kD);
  if (L[0].p_in > 0.f) b.xd0 = ar.take<float>(G * 2 * kD);
  b.pred = ar.take<float>(G * L[n - 1].out_dim);
  // backward: u[l] and dz[l] where layer l + 1's input gradient runs (dz[n-1]: the loss gradient)
  for (int l = 0; l + 1 < n; ++l) {
    b.xd[l + 1] = ar.take<float>(G * L[l].out_dim);
    if (a->backward && fnb_mlp_needs_dx(L, l + 1, enc)) b.u[l] = ar.take<float>(G * L[l].out_dim);
  }
  if (a->backward) {
    for (int l = 0; l < n; ++l)
      if (l == n - 1 || fnb_mlp_needs_dx(L, l + 1, enc)) b.dz[l] = ar.take<float>(G * L[l].out_dim);
    if (enc) b.d_readout = ar.take<float>(G * 2 * kD);
    b.rec = ar.take<float>(fnb_mlp_dw_record_floats(L, n, G));
  }
  if (enc) {
    b.g_atoms = ar.take<float>(Na * kD); b.g_frags = ar.take<float>(Nf * kD);
    b.enc_bws_bytes = fnb_encoder_bwd_workspace_bytes(&sp, &o, a->layers);
    b.enc_bws = ar.bytes(b.enc_bws_bytes);
  }
  if (a->variant == FNB_VARIANT_EDGE) {
    b.cnx_table = ar.take<float>(Nfb * 4);
    if (enc) b.d_cnx_table = ar.take<float>(Nfb * 4);
  }
  if (out) *out = b;
  return ar.total();
}

}  // namespace

extern "C" size_t fnb_finetune_step_workspace_bytes(const fnb_finetune_step_args *a) {
  if (!ft_args_ok(a)) return 0;
  return ft_layout(a, nullptr, nullptr);
}

extern "C" uint64_t fnb_finetune_step_rng_span(const fnb_finetune_step_args *a) {
  if (!ft_args_ok(a)) return 0;
  const fnb_batch_inputs in = ft_inputs(a);
  const fnb_batch_plan sp = sizes_plan(&in);
  const fnb_encoder_opts o = ft_opts_of(a);
  return fnb_encoder_rng_span(&sp, &o, a->layers) +
         fnb_mlp_rng(a->head, a->n_head_layers, a->batch.n_graphs, 0, nullptr, nullptr);
}

extern "C" int fnb_finetune_step(const fnb_finetune_step_args *a, void *workspace, size_t workspace_bytes, void *scratch,
                                 void *stream) {
  if (!a || !workspace || !scratch) return FNB_ERR_NULL;
  if (!a->head || !a->layers) return FNB_ERR_NULL;
  if (a->n_layers < 1 || a->n_layers > 16) return FNB_ERR_SIZE;
  if (a->first_trained_layer < 0 || a->first_trained_layer > a->n_layers) return FNB_ERR_SIZE;
  if (a->variant < FNB_VARIANT_GAT2 || a->variant > FNB_VARIANT_EDGE) return FNB_ERR_MODE;
  const bool edge = a->variant == FNB_VARIANT_EDGE;
  if (edge && (!a->cnx_attr || !a->W_cnx || !a->b_cnx)) return FNB_ERR_NULL;
  const fnb_batch_inputs in_v = ft_inputs(a), *in = &in_v;
  if (in->n_atoms < 1 || in->n_bonds < 0 || in->n_frags < 0 || in->n_graphs < 1 || !in->batch || !in->frag_batch)
    return FNB_ERR_SIZE;
  RC(fnb_mlp_check(a->head, a->n_head_layers, in->n_graphs, 2 * kD, a->backward));
  if (a->loss_kind != FNB_LOSS_MSE && a->loss_kind != FNB_LOSS_BCE_MASKED) return FNB_ERR_MODE;
  if (!a->loss || !a->target || !a->x_atoms || !a->x_bond) return FNB_ERR_NULL;
  if (!a->x_fbond && a->variant == FNB_VARIANT_GAT2) return FNB_ERR_NULL;
  const bool enc_bwd = a->backward && encoder_trained(a);
  if (a->backward && !enc_bwd) {   // a backward that trains nothing is a caller's mistake
    bool head_trained = false;
    for (int l = 0; l < a->n_head_layers; ++l) head_trained |= a->head[l].dW != nullptr;
    if (!head_trained) return FNB_ERR_MODE;
  }
  if (enc_bwd && !a->layer_grads) return FNB_ERR_NULL;
  if (enc_bwd && edge && (!a->dW_cnx || !a->db_cnx || !a->layer_grads[a->n_layers - 1].f)) return FNB_ERR_NULL;
  if (reinterpret_cast<uintptr_t>(workspace) & 255u) return FNB_ERR_ALIGN;
  FtBufs B;
  if (ft_layout(a, (char *)workspace, &B) > workspace_bytes) return FNB_ERR_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream;
  const fnb_mlp_layer *L = a->head;
  const int n = a->n_head_layers;
  const int64_t G = in->n_graphs, n_out = G * L[n - 1].out_dim;

  // ---- collate + encoder forward
  FnbAux aux{};
  const bool two = fnb_aux_streams(&aux) == 0;
  fnb_batch_plan plan{};
  fnb_encoder_opts o = ft_opts_of(a);
  fnb_encoder_io eio{};
  eio.x_atoms = a->x_atoms; eio.x_bond = a->x_bond; eio.x_fbond = a->x_fbond;
  eio.out_atoms = B.out_atoms; eio.out_frags = B.out_frags; eio.out_bond = B.out_bond; eio.out_fbond = B.out_fbond;
  const fnb_layer_params &top = a->layers[a->n_layers - 1];
  if (edge) {   // gat2_edge: the fragment graph's edge term from the connection attributes (gat2_edge.py:152-158)
    RC(fnb_cnx_table_fwd(a->cnx_attr, in->n_fbond_nodes, a->W_cnx, a->b_cnx, top.f, B.cnx_table, s));
    eio.frag_table = B.cnx_table;
  }
  RC(collate_and_encode(in, a->plan_arena, B.plan_arena, B.plan_bytes, &o, a->layers, &eio, B.enc_ws, B.enc_bytes,
                        scratch, stream, aux, two, &plan));
  // ---- readout: [G,256] = cat(sum over each molecule's atoms, sum over its fragments)
  RC(fnb_segment_sum(plan.mol_atom_ptr, nullptr, G, B.out_atoms, B.readout, 2 * kD, nullptr, 0, 0, 0, nullptr, stream));
  RC(fnb_segment_sum(plan.mol_frag_ptr, nullptr, G, B.out_frags, B.readout + kD, 2 * kD, nullptr, 0, 0, 0, nullptr,
                     stream));
  // ---- head forward; its dropout sites follow the encoder's
  FnbMlpRun r{};
  r.L = L; r.n = n; r.G = G; r.training = a->training; r.seed = a->seed;
  fnb_mlp_rng(L, n, G, a->offset + fnb_encoder_rng_span(&plan, &o, a->layers), r.in_base, r.out_base);
  r.x0 = B.readout;
  r.xd[0] = (a->training && L[0].p_in > 0.f) ? B.xd0 : B.readout;
  for (int l = 0; l + 1 < n; ++l) { r.xd[l + 1] = B.xd[l + 1]; r.u[l] = B.u[l]; }
  r.out = a->predictions ? a->predictions : B.pred;
  RC(fnb_mlp_forward(&r, s));
  // ---- loss (and, training, the gradient of the predictions)
  float *d_pred = a->backward ? B.dz[n - 1] : nullptr;
  if (a->loss_kind == FNB_LOSS_MSE) {
    fnb_mse_term t{};
    t.pred = r.out; t.target = a->target; t.n = n_out; t.weight = 1.f; t.grad = d_pred;
    RC(fnb_mse_sum_loss(&t, 1, a->loss, scratch, stream));
  } else {
    RC(fnb_bce_masked_loss(r.out, a->target, n_out, a->loss, d_pred, s));
  }
  if (!a->backward) return 0;
  // ---- head backward, readout backward, encoder backward (the last two only where the encoder trains)
  for (int l = 0; l < n; ++l) r.dz[l] = B.dz[l];
  r.dx0 = B.d_readout; r.rec = B.rec;
  RC(fnb_mlp_backward(&r, s));
  if (!enc_bwd) return 0;
  RC(fnb_segment_gather(B.d_readout, 2 * kD, plan.batch32, in->n_atoms, nullptr, B.g_atoms, stream));
  RC(fnb_segment_gather(B.d_readout + kD, 2 * kD, plan.frag_batch32, in->n_frags, nullptr, B.g_frags, stream));
  eio.g_atoms = B.g_atoms; eio.g_frags = B.g_frags; eio.g_bond = nullptr; eio.g_fbond = nullptr;
  eio.d_frag_table = B.d_cnx_table;
  RC(fnb_encoder_backward(&plan, &o, a->layers, a->layer_grads, &eio, B.enc_ws, B.enc_bytes, B.enc_bws, B.enc_bws_bytes,
                          scratch, stream));
  // gat2_edge: the edge term's gradient to cnx_attr_transform and to the edge slice of f, which the encoder left zero;
  // behind the encoder backward on this stream (it ends by joining its side streams)
  if (edge)
    RC(fnb_cnx_table_bwd(a->cnx_attr, B.d_cnx_table, in->n_fbond_nodes, a->W_cnx, a->b_cnx, top.f, a->dW_cnx, a->db_cnx,
                         a->layer_grads[a->n_layers - 1].f, scratch, s));
  return 0;
}
