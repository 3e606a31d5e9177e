// Whole-encoder programs: FragNet.forward / its backward as ONE library call each.
//
// Reference: FragNet.forward (fragnet/model/gat/gat2.py:381-442) runs num_layer x FragNetLayerA.forward
// (gat2.py:121-330: bond graph -> atom graph -> atom->fragment pooling -> fragment-connection graph -> fragment
// graph) with ReLU(Dropout(.)) on the four outputs of every layer (gat2.py:414-418, 436-440).  Upstream that is a few
// hundred eager torch ops per step; the first version of this library still paid ~190 Python->C calls and ~300
// allocator calls per training step and was host-bound (DESIGN.md section 3).  Here the host side of the sequence is
// C++: one call issues every launch of the pass back to back on the caller's stream, all intermediates come out of
// one caller-allocated workspace whose layout is a pure function of the sizes, and nothing synchronises.
//
// Per layer, forward: 3 projections (tcgen05 TF32 or FP32), 3 tiled attention kernels (4 in the layer that runs
// the fragment block, plus the pooling).  Folded into those launches: edge-embedding constants, output masks,
// ReLU(Dropout), the consumer graph's edge term, the fragment graph's node scalars.
// Backward: per graph one destination pass + one source pass (parameter-gradient reductions inside), the edge-table
// backward with the ReLU(Dropout) backward folded in, and the projection backward (dX, dW).
#include "common.cuh"

namespace {

constexpr int AB_STRIDE = 96, AB_T = 0, AB_E = 32, AB_S = 64;    // a_b / f_a_b = [target 32 | edge 32 | source 32]
constexpr int A_STRIDE = 192, A_T = 0, A_E = 32, A_S = 160;      // a / f     = [target 32 | edge 128 | source 32]

struct LayerBufs {
  float *xa0;                                                   // layer 0: Dropout(x_atoms) (training only)
  float *x_pad[3], *W_pad[3];                                   // layer 0, TF32: inputs / weights zero-padded to k_pad columns
  int k_pad[3];                                                 // (order: bond, atom, fbond; 0 = no padding needed)
  float *hb, *Sb, *pre_bond, *y_bond, *p_b, *se_atom;
  float *ha, *Sa, *pre_atom, *y_atom, *p_a;
  float *hfb, *Sfb, *pre_fbond, *y_fbond, *p_fb, *se_frag;
  float *hf, *Sf, *pre_frag, *y_frag, *p_f;
};

struct Sizes {
  int64_t Na, Nb, Nfb, Nf, Ea, Eb, Efb, Ef;   // E* include appended self loops (atom graph)
};

Sizes sizes_of(const fnb_batch_plan *p) {
  Sizes s;
  s.Na = p->atom.n_nodes; s.Nb = p->bond.n_nodes; s.Nfb = p->fbond.n_nodes; s.Nf = p->frag.n_nodes;
  s.Ea = p->atom.n_edges; s.Eb = p->bond.n_edges; s.Efb = p->fbond.n_edges; s.Ef = p->frag.n_edges;
  return s;
}

bool input_dropout(const fnb_encoder_opts *o) { return o->post_act && o->training && o->drop_p > 0.f; }

// Layer-0 feature widths (167 / 17 / 6) are not addressable by TMA (row pitch must be a multiple of 16 bytes) and not a
// multiple of the 32-column K block of the tensor-core kernels: in TF32 mode the inputs and weights are zero-padded
// once per pass to the next multiple of 32 columns and take the same tcgen05 kernels as every other layer.
int pad_width(const fnb_encoder_opts *o, int K) {
  if (!fnb_tc_precision(o->precision) || (K & 31) == 0 || K > 224) return 0;
  return (K + 31) & ~31;
}

// Forward workspace layout (identical in fnb_encoder_forward / _backward / _workspace_bytes).
size_t layout(const fnb_batch_plan *plan, const fnb_encoder_opts *o, const fnb_layer_params *L, char *base,
              LayerBufs *bufs) {
  const Sizes z = sizes_of(plan);
  Arena a{base, 0};
  for (int l = 0; l < o->n_layers; ++l) {
    LayerBufs b{};
    const bool last = l == o->n_layers - 1;
    const bool keep = o->save_for_backward != 0 && l >= o->first_trained_layer;   // frozen layers: nothing to save
    const bool want_p = keep || L[l].want_attention;
    const bool frag = L[l].run_frag_block != 0;
    const bool pool_out = last && o->pool_frags;   // gat2_lite: the pooled pre-activation atoms are the fragment output
    if (l == 0 && input_dropout(o)) b.xa0 = a.take<float>(z.Na * L[0].K_atom);
    if (l == 0) {
      const int ks[3] = {L[0].K_bond, L[0].K_atom, L[0].K_fbond};
      const int64_t ns[3] = {z.Nb, z.Na, z.Nfb};
      for (int j = 0; j < 3; ++j) {
        b.k_pad[j] = j == 2 && o->skip_fbond ? 0 : pad_width(o, ks[j]);
        if (b.k_pad[j]) {
          b.x_pad[j] = a.take<float>(ns[j] * b.k_pad[j]);
          b.W_pad[j] = a.take<float>((size_t)kD * b.k_pad[j]);
        }
      }
    }
    b.hb = a.take<float>(z.Nb * kD);
    b.Sb = a.take<float>(z.Nb * 8);
    b.se_atom = a.take<float>(z.Nb * 4);
    b.ha = a.take<float>(z.Na * kD);
    b.Sa = a.take<float>(z.Na * 8);
    b.hfb = a.take<float>(z.Nfb * kD);
    b.Sfb = a.take<float>(z.Nfb * 8);
    if (want_p) {
      b.p_b = a.take<float>(z.Eb * 4);
      b.p_a = a.take<float>(z.Ea * 4);
      b.p_fb = a.take<float>(z.Efb * 4);
    }
    if (o->post_act) {
      // pre-activations only where something downstream reads them: the bond features feed d alpha_e of the atom
      // block's backward; the atom features feed the pooling; the fragment-connection features feed d alpha_e of
      // the fragment block.  Post-activations of the last layer go straight to the caller's outputs.
      if (keep) b.pre_bond = a.take<float>(z.Nb * kD);
      if (frag || pool_out) b.pre_atom = a.take<float>(z.Na * kD);
      if (frag && keep) b.pre_fbond = a.take<float>(z.Nfb * kD);
      if (!last) {
        b.y_bond = a.take<float>(z.Nb * kD);
        b.y_atom = a.take<float>(z.Na * kD);
        b.y_fbond = a.take<float>(z.Nfb * kD);
      }
    }
    if (frag) {
      b.hf = a.take<float>(z.Nf * kD);
      b.Sf = a.take<float>(z.Nf * 8);
      b.se_frag = a.take<float>(z.Nfb * 4);
      if (want_p) b.p_f = a.take<float>(z.Ef * 4);
      if (o->post_act && !last) b.y_frag = a.take<float>(z.Nf * kD);   // dead output of a non-final layer
    }
    if (bufs) bufs[l] = b;
  }
  return a.total();
}

struct BwdBufs {
  float *g_bond, *dz_b, *dSt_b, *dh_b, *dh_b2, *dx_bond;   // dh: one buffer per layer parity, so that a layer's
  float *g_atom, *dz_a, *dz_a2, *dSt_a, *dh_a, *dh_a2, *dx_atom;   // source pass never waits for the weight-gradient GEMM above it
  float *g_fbond, *dz_fb, *dSt_fb, *dh_fb, *dx_fbond;
  float *g_frag, *dz_f, *dSt_f, *d_hf;
  float *Wt;   // [n_layers][3][128*128] transposed K=128 projection weights
  float *scratch2;   // scratch of the fragment-connection chain when it runs on the auxiliary stream
  float *scratch3;   // scratch of the weight-gradient stream
  float *scratch4;   // scratch of the atom-graph stream
  float *scratch5;   // scratch of the edge-term stream
  float *scratch6;   // scratch of the atom chain's weight-gradient stream
};

size_t bwd_layout(const fnb_batch_plan *plan, const fnb_encoder_opts *o, char *base, BwdBufs *out) {
  const Sizes z = sizes_of(plan);
  Arena a{base, 0};
  BwdBufs b{};
  b.g_bond = a.take<float>(z.Nb * kD); b.dz_b = a.take<float>(z.Eb * 4); b.dSt_b = a.take<float>(z.Nb * 4);
  b.dh_b = a.take<float>(z.Nb * kD); b.dh_b2 = a.take<float>(z.Nb * kD); b.dx_bond = a.take<float>(z.Nb * kD);
  b.g_atom = a.take<float>(z.Na * kD); b.dz_a = a.take<float>(z.Ea * 4); b.dz_a2 = a.take<float>(z.Ea * 4);
  b.dSt_a = a.take<float>(z.Na * 4);
  b.dh_a = a.take<float>(z.Na * kD); b.dh_a2 = a.take<float>(z.Na * kD); b.dx_atom = a.take<float>(z.Na * kD);
  b.g_fbond = a.take<float>(z.Nfb * kD); b.dz_fb = a.take<float>(z.Efb * 4); b.dSt_fb = a.take<float>(z.Nfb * 4);
  b.dh_fb = a.take<float>(z.Nfb * kD); b.dx_fbond = a.take<float>(z.Nfb * kD);
  b.g_frag = a.take<float>(z.Nf * kD); b.dz_f = a.take<float>(z.Ef * 4); b.dSt_f = a.take<float>(z.Nf * 4);
  b.d_hf = a.take<float>(z.Nf * kD);
  b.Wt = a.take<float>((size_t)(o->n_layers - o->first_trained_layer) * 3 * kD * kD);   // trained layers only
  b.scratch2 = a.take<float>(kScratchFloats);
  b.scratch3 = a.take<float>(kScratchFloats);
  b.scratch4 = a.take<float>(kScratchFloats);
  b.scratch5 = a.take<float>(kScratchFloats);
  b.scratch6 = a.take<float>(kScratchFloats);
  if (out) *out = b;
  return a.total();
}

// RNG counters consumed by one dropout site over n elements.
uint64_t span(int64_t n) { return (uint64_t)((n + 3) / 4); }

// Counter bases of the dropout sites, in a fixed order: input, then per layer bond, atom, fbond, frag.
struct RngPlan {
  uint64_t input;
  uint64_t bond[16], atom[16], fbond[16], frag[16];
  uint64_t total;
};

RngPlan rng_plan(const fnb_batch_plan *plan, const fnb_encoder_opts *o, const fnb_layer_params *L) {
  const Sizes z = sizes_of(plan);
  RngPlan p{};
  uint64_t c = o->offset;
  p.input = c;
  c += span(z.Na * (int64_t)L[0].K_atom);
  for (int l = 0; l < o->n_layers && l < 16; ++l) {
    p.bond[l] = c;  c += span(z.Nb * kD);
    p.atom[l] = c;  c += span(z.Na * kD);
    p.fbond[l] = c; c += span(z.Nfb * kD);
    p.frag[l] = c;  c += span(z.Nf * kD);
  }
  p.total = c - o->offset;
  return p;
}

fnb_post_act post_of(const fnb_encoder_opts *o, uint64_t counter) {
  fnb_post_act pa;
  pa.p = o->drop_p; pa.training = o->training; pa.relu = 1; pa.seed = o->seed; pa.offset = counter;
  return pa;
}

// dst[r, 0:k_pad] = [src[r, 0:K] | 0]: up to 6 matrices per launch (blockIdx.y).
struct PadJobs {
  const float *src[6];
  float *dst[6];
  int64_t rows[6];
  int K[6], k_pad[6];
  int n;
  // job `drop_job` (or -1): nn.Dropout (gat2.py:396) applied on the way -- element i of the UNPADDED matrix draws the
  // same bit as in k_dropout_relu_fwd (counter offset + i / 4, position i % 4), so the two forms are interchangeable
  int drop_job;
  float drop_scale;
  uint32_t drop_threshold;
  uint64_t seed, offset;
};
__device__ __forceinline__ float dropped(const PadJobs &j, float v, int64_t i) {
  const uint2 r = dropout_bits(j.seed, j.offset + (uint64_t)(i >> 2));
  const uint32_t w = (i & 2) ? r.y : r.x;
  const uint32_t bits = (i & 1) ? (w >> 16) : (w & 0xffffu);
  return bits >= j.drop_threshold ? v * j.drop_scale : 0.f;
}
__global__ void __launch_bounds__(256) k_pad_cols(PadJobs j) {
  pdl_wait();
  const int job = blockIdx.y;
  const int K = j.K[job], kp = j.k_pad[job];
  const bool drop = job == j.drop_job;
  const int64_t total = j.rows[job] * (kp >> 2);
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / (kp >> 2);
    const int c = (int)(i - r * (kp >> 2)) * 4;
    const float *sp = j.src[job] + r * K + c;
    float4 v;
    v.x = c < K ? __ldg(sp) : 0.f;
    v.y = c + 1 < K ? __ldg(sp + 1) : 0.f;
    v.z = c + 2 < K ? __ldg(sp + 2) : 0.f;
    v.w = c + 3 < K ? __ldg(sp + 3) : 0.f;
    if (drop) {
      const int64_t e = r * K + c;
      if (c < K) v.x = dropped(j, v.x, e);
      if (c + 1 < K) v.y = dropped(j, v.y, e + 1);
      if (c + 2 < K) v.z = dropped(j, v.z, e + 2);
      if (c + 3 < K) v.w = dropped(j, v.w, e + 3);
    }
    st4(j.dst[job] + r * kp + c, v);
  }
}

// Rows listed in `rows` of up to two [N,128] tensors -- and of the [N,4] edge term the consumer graph reads in their
// place (<0, alpha_e> = 0) -- are zeroed: the list form of the masks of gat2.py:173-176, :227-231, :275-278.
__global__ void k_zero_rows(float *__restrict__ a, float *__restrict__ b, float *__restrict__ se,
                            const int *__restrict__ rows, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n * 32; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = __ldg(rows + (i >> 5));
    const int c = (int)(i & 31) * 4;
    if (a) st4(a + r * kD + c, make_float4(0.f, 0.f, 0.f, 0.f));
    if (b) st4(b + r * kD + c, make_float4(0.f, 0.f, 0.f, 0.f));
    if (se && c == 0) st4(se + r * 4, make_float4(0.f, 0.f, 0.f, 0.f));
  }
}

// out[e, 0:4] = src[index[e], 0:4]: gradient of an external edge table (slot order -> edge-id order).
__global__ void __launch_bounds__(256) k_gather_rows4(const float *__restrict__ src, const int *__restrict__ index,
                                                       float *__restrict__ out, int64_t n) {
  pdl_wait();
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e < n) st4(out + e * 4, ldg4(src + (int64_t)__ldg(index + e) * 4));
}

int check_common(const fnb_batch_plan *plan, const fnb_encoder_opts *o, const fnb_layer_params *L,
                 const fnb_encoder_io *io) {
  if (!plan || !o || !L || !io) return FNB_ERR_NULL;
  if (o->n_layers < 1 || o->n_layers > 16) return FNB_ERR_SIZE;
  if (o->first_trained_layer < 0 || o->first_trained_layer > o->n_layers) return FNB_ERR_SIZE;
  if (!o->post_act && o->n_layers != 1) return FNB_ERR_MODE;
  if (!(o->drop_p >= 0.f && o->drop_p < 1.f)) return FNB_ERR_SIZE;
  const Sizes z = sizes_of(plan);
  // a graph without nodes (gat2_lite runs with empty fragment-side graphs) has no feature rows to point at
  if ((z.Na > 0 && (!io->x_atoms || !io->out_atoms)) || (z.Nb > 0 && (!io->x_bond || !io->out_bond)) ||
      (z.Nfb > 0 && !o->skip_fbond && (!io->x_fbond || !io->out_fbond)))
    return FNB_ERR_NULL;
  if (o->pool_frags && (!o->post_act || (z.Nf > 0 && !io->out_frags))) return FNB_ERR_MODE;
  if (z.Na != plan->n_atoms || z.Nf != plan->n_frags) return FNB_ERR_SIZE;
  // the atom graph's edges are the bond graph's nodes, the fragment graph's edges the fragment-connection nodes
  if (plan->atom.n_real_edges != z.Nb || plan->frag.n_real_edges != z.Nfb) return FNB_ERR_SIZE;
  for (int l = 0; l < o->n_layers; ++l) {
    if (l > 0 && (L[l].K_atom != kD || L[l].K_bond != kD || L[l].K_fbond != kD)) return FNB_ERR_SIZE;
    if (L[l].run_frag_block && !io->out_frags && l == o->n_layers - 1) return FNB_ERR_NULL;
    // the pooled output replaces the fragment block; a skipped fragment-connection chain emits no fragment edge term
    if (L[l].run_frag_block && (o->pool_frags || (o->skip_fbond && !io->frag_table))) return FNB_ERR_MODE;
  }
  return 0;
}

}  // namespace

extern "C" size_t fnb_encoder_workspace_bytes(const fnb_batch_plan *plan, const fnb_encoder_opts *opts,
                                              const fnb_layer_params *layers) {
  if (!plan || !opts || !layers || opts->n_layers < 1 || opts->n_layers > 16) return 0;
  if (opts->first_trained_layer < 0 || opts->first_trained_layer > opts->n_layers) return 0;
  return layout(plan, opts, layers, nullptr, nullptr);
}

extern "C" size_t fnb_encoder_bwd_workspace_bytes(const fnb_batch_plan *plan, const fnb_encoder_opts *opts,
                                                  const fnb_layer_params *layers) {
  (void)layers;
  if (!plan || !opts || opts->n_layers < 1 || opts->n_layers > 16) return 0;
  if (opts->first_trained_layer < 0 || opts->first_trained_layer > opts->n_layers) return 0;
  return bwd_layout(plan, opts, nullptr, nullptr);
}

extern "C" uint64_t fnb_encoder_rng_span(const fnb_batch_plan *plan, const fnb_encoder_opts *opts,
                                            const fnb_layer_params *layers) {
  if (!plan || !opts || !layers || opts->n_layers < 1 || opts->n_layers > 16) return 0;
  return rng_plan(plan, opts, layers).total;
}

extern "C" int fnb_encoder_forward(const fnb_batch_plan *plan, const fnb_encoder_opts *o, const fnb_layer_params *L,
                                   const fnb_encoder_io *io, void *workspace, size_t workspace_bytes, void *scratch,
                                   void *stream_) {
  return fnb_encoder_forward_impl(plan, o, L, io, workspace, workspace_bytes, scratch, stream_, nullptr, nullptr);
}

// plan_ready: optional event after which the ARRAYS of `plan` are complete (its sizes and pointers are valid at call
// time).  fnb_pretrain_step builds the plan on an auxiliary stream while the plan-independent head of the forward
// (input dropout, operand padding, the three layer-0 projections) runs; the first attention kernel of every stream
// waits for the event.
int fnb_encoder_forward_impl(const fnb_batch_plan *plan, const fnb_encoder_opts *o, const fnb_layer_params *L,
                             const fnb_encoder_io *io, void *workspace, size_t workspace_bytes, void *scratch,
                             void *stream_, cudaEvent_t plan_ready, cudaEvent_t plan_complete) {
  RC(check_common(plan, o, L, io));
  if (!workspace || !scratch) return FNB_ERR_NULL;
  LayerBufs B[16];
  if (layout(plan, o, L, (char *)workspace, B) > workspace_bytes) return FNB_ERR_WORKSPACE;
  const Sizes z = sizes_of(plan);
  const RngPlan ph = rng_plan(plan, o, L);
  cudaStream_t stream = (cudaStream_t)stream_;

  const float *xa = io->x_atoms, *xb = io->x_bond, *xfb = io->x_fbond;
  // nn.Dropout on the raw atom features (gat2.py:396).  When layer 0 takes the padded operands anyway and nobody asks
  // for d x_atoms (whose backward reads the dropped copy), the padding kernel applies it on the way: one launch and one
  // pass over x_atoms fewer at the very head of the step.
  const bool drop_in_pad = input_dropout(o) && B[0].k_pad[1] != 0 && !o->need_dx_atoms;
  if (input_dropout(o) && !drop_in_pad) {
    RC(fnb_dropout_relu_fwd(xa, B[0].xa0, z.Na * (int64_t)L[0].K_atom, o->drop_p, 1, 0, o->seed, ph.input, stream_));
    xa = B[0].xa0;
  }
  {  // layer-0 operands padded for the tensor-core path (one launch for inputs and weights)
    PadJobs pj{};
    pj.drop_job = -1;
    const float *xs[3] = {xb, xa, xfb}, *ws[3] = {L[0].Wb, L[0].Wa, L[0].Wfb};
    const int ks[3] = {L[0].K_bond, L[0].K_atom, L[0].K_fbond};
    const int64_t ns[3] = {z.Nb, z.Na, z.Nfb};
    int64_t most = 0;
    for (int j = 0; j < 3; ++j)
      if (B[0].k_pad[j]) {
        const int64_t rows[2] = {ns[j], kD};
        const float *src[2] = {xs[j], ws[j]};
        float *dst[2] = {B[0].x_pad[j], B[0].W_pad[j]};
        for (int t = 0; t < 2; ++t) {
          const int k = pj.n++;
          if (j == 1 && t == 0 && drop_in_pad) {
            pj.drop_job = k;
            pj.drop_scale = 1.f / (1.f - o->drop_p);
            pj.drop_threshold = (uint32_t)(o->drop_p * 65536.0f + 0.5f);
            pj.seed = o->seed; pj.offset = ph.input;
          }
          pj.src[k] = src[t]; pj.dst[k] = dst[t]; pj.rows[k] = rows[t]; pj.K[k] = ks[j]; pj.k_pad[k] = B[0].k_pad[j];
          if (rows[t] * (B[0].k_pad[j] >> 2) > most) most = rows[t] * (B[0].k_pad[j] >> 2);
        }
      }
    if (pj.n && most > 0) {
      int64_t blocks = (most + 255) / 256;
      if (blocks > kNumSMs * 8) blocks = kNumSMs * 8;
      if (cudaError_t le = fnb_launch(k_pad_cols, dim3((unsigned)blocks, pj.n), dim3(256), 0, stream, pj)) return (int)le;
      FNB_CHECK_LAUNCH();
    }
  }
  // The fragment-connection chain (projection_fb + its attention block, every layer) depends on nothing the bond /
  // atom chain produces until the fragment block: it runs on the auxiliary stream, concurrently with the big graphs.
  FnbAux aux{};
  const bool two = fnb_aux_streams(&aux) == 0;
  cudaStream_t sB = two ? aux.stream : stream;
  void *sB_ = (void *)sB;
  bool pending = false;   // work queued on sB that the caller's stream has not waited for yet
  if (two) {
    RC((int)cudaEventRecord(aux.fork, stream));
    RC((int)cudaStreamWaitEvent(sB, aux.fork, 0));
  }
  cudaStream_t sA = two ? aux.astream : stream;
  void *sA_ = (void *)sA;
  bool a_pending = false;
  auto join = [&]() -> int {
    if (two && pending) {
      RC((int)cudaEventRecord(aux.join, sB));
      RC((int)cudaStreamWaitEvent(stream, aux.join, 0));
      pending = false;
    }
    if (two && a_pending) {
      RC((int)cudaEventRecord(aux.a_join, sA));
      RC((int)cudaStreamWaitEvent(stream, aux.a_join, 0));
      a_pending = false;
    }
    return 0;
  };
  for (int l = 0; l < o->n_layers; ++l) {
    const fnb_layer_params &P = L[l];
    LayerBufs &b = B[l];
    const bool last = l == o->n_layers - 1;
    const bool frag = P.run_frag_block != 0;
    const bool want_p = (o->save_for_backward != 0 && l >= o->first_trained_layer) || P.want_attention;
    // layer-0 operands may be the zero-padded copies (TF32 path)
    const bool pb = l == 0 && b.k_pad[0], pa = l == 0 && b.k_pad[1], pf = l == 0 && b.k_pad[2];
    const float *xb_in = pb ? b.x_pad[0] : xb, *Wb_in = pb ? b.W_pad[0] : P.Wb;
    const float *xa_in = pa ? b.x_pad[1] : xa, *Wa_in = pa ? b.W_pad[1] : P.Wa;
    const float *xfb_in = pf ? b.x_pad[2] : xfb, *Wfb_in = pf ? b.W_pad[2] : P.Wfb;
    const int Kb_in = pb ? b.k_pad[0] : P.K_bond, Ka_in = pa ? b.k_pad[1] : P.K_atom, Kfb_in = pf ? b.k_pad[2] : P.K_fbond;
    // where the four results of this layer go
    float *pre_bond = o->post_act ? b.pre_bond : io->out_bond;
    float *pre_atom = o->post_act ? b.pre_atom : io->out_atoms;
    float *pre_fbond = o->post_act ? b.pre_fbond : io->out_fbond;
    float *pre_frag = o->post_act ? nullptr : io->out_frags;
    float *y_bond = o->post_act ? (last ? io->out_bond : b.y_bond) : nullptr;
    float *y_atom = o->post_act ? (last ? io->out_atoms : b.y_atom) : nullptr;
    float *y_fbond = o->post_act ? (last ? io->out_fbond : b.y_fbond) : nullptr;
    float *y_frag = o->post_act ? (last ? io->out_frags : b.y_frag) : nullptr;

    // ---- atom chain (gat2.py:179-231) on its own stream: the projection needs only the previous layer's atoms (produced
    // on this same stream), the attention block additionally the bond block's edge term of this layer
    if (two && l == 0) {
      RC((int)cudaEventRecord(aux.a_fork, stream));
      RC((int)cudaStreamWaitEvent(sA, aux.a_fork, 0));
    }
    RC(fnb_proj_fwd(xa_in, Wa_in, P.ba, z.Na, Ka_in, P.a, A_STRIDE, A_T, A_S, b.ha, b.Sa, o->precision, sA_));
    // ---- bond graph (gat2.py:138-176); epilogue emits the atom graph's edge term <new_bond[e], a_e[h]>
    RC(fnb_proj_fwd(xb_in, Wb_in, P.bb, z.Nb, Kb_in, P.a_b, AB_STRIDE, AB_T, AB_S, b.hb, b.Sb, o->precision, stream_));
    {
      fnb_gat_fwd_args f{};
      f.h = b.hb; f.S = b.Sb; f.edge_mode = FNB_EDGE_AFFINE1; f.We = P.We_b; f.be = P.be_b;
      f.alpha_e = P.a_b + AB_E; f.alpha_stride = AB_STRIDE; f.out = pre_bond; f.y = y_bond;
      f.post = post_of(o, ph.bond[l]); f.p_saved = want_p ? b.p_b : nullptr;
      f.mask_lo = P.bond_mask >= 0 ? P.bond_mask : -1; f.mask_hi = P.bond_mask >= 0 ? P.bond_mask + 2 : -1;
      f.next_alpha_e = P.a + A_E; f.next_alpha_stride = A_STRIDE; f.next_Se = b.se_atom;
      if (plan_ready && l == 0) RC((int)cudaStreamWaitEvent(stream, plan_ready, 0));
      RC(fnb_gat_fwd_tiled(&plan->bond, &f, stream_));
      // everything later on this stream (pooling, readout, the backward) may read the rest of the plan
      if (plan_complete && l == 0) RC((int)cudaStreamWaitEvent(stream, plan_complete, 0));
      if (P.bond_mask_rows && P.n_bond_mask_rows > 0) {
        k_zero_rows<<<(int)((P.n_bond_mask_rows * 32 + 255) / 256), 256, 0, stream>>>(pre_bond, y_bond, b.se_atom,
                                                                                    P.bond_mask_rows, P.n_bond_mask_rows);
        FNB_CHECK_LAUNCH();
      }
    }
    // ---- atom graph with self loops (gat2.py:179-231)
    if (two) {
      RC((int)cudaEventRecord(aux.a_dz, stream));          // the bond block of this layer is queued
      RC((int)cudaStreamWaitEvent(sA, aux.a_dz, 0));
    }
    {
      fnb_gat_fwd_args f{};
      f.h = b.ha; f.S = b.Sa; f.edge_mode = FNB_EDGE_TABLE; f.edge_table = b.se_atom; f.out = pre_atom; f.y = y_atom;
      f.post = post_of(o, ph.atom[l]); f.p_saved = want_p ? b.p_a : nullptr;
      f.mask_lo = P.atom_mask >= 0 ? P.atom_mask : -1; f.mask_hi = P.atom_mask >= 0 ? P.atom_mask + 1 : -1;
      if (plan_ready && l == 0 && two) RC((int)cudaStreamWaitEvent(sA, plan_ready, 0));
      RC(fnb_gat_fwd_tiled(&plan->atom, &f, sA_));
      if (plan_complete && l == 0 && two) RC((int)cudaStreamWaitEvent(sA, plan_complete, 0));
      if (P.atom_mask_list && P.n_atom_mask > 0) {
        k_zero_rows<<<(int)((P.n_atom_mask * 32 + 255) / 256), 256, 0, sA>>>(pre_atom, y_atom, nullptr, P.atom_mask_list,
                                                                           P.n_atom_mask);
        FNB_CHECK_LAUNCH();
      }
      a_pending = true;
    }
    // ---- fragment-connection graph (gat2.py:239-278); epilogue emits the fragment graph's edge term
    if (!o->skip_fbond) {
      RC(fnb_proj_fwd(xfb_in, Wfb_in, P.bfb, z.Nfb, Kfb_in, P.f_a_b, AB_STRIDE, AB_T, AB_S, b.hfb, b.Sfb, o->precision,
                      sB_));
      pending = true;
      fnb_gat_fwd_args f{};
      f.h = b.hfb; f.S = b.Sfb; f.edge_mode = FNB_EDGE_AFFINE6; f.We = P.We_fb; f.be = P.be_fb;
      f.alpha_e = P.f_a_b + AB_E; f.alpha_stride = AB_STRIDE; f.out = pre_fbond; f.y = y_fbond;
      f.post = post_of(o, ph.fbond[l]); f.p_saved = want_p ? b.p_fb : nullptr;
      f.mask_lo = P.frag_bond_mask >= 0 ? 2 * P.frag_bond_mask : -1;
      f.mask_hi = P.frag_bond_mask >= 0 ? 2 * P.frag_bond_mask + 2 : -1;
      if (frag) { f.next_alpha_e = P.f + A_E; f.next_alpha_stride = A_STRIDE; f.next_Se = b.se_frag; }
      if (plan_ready && l == 0 && two) RC((int)cudaStreamWaitEvent(sB, plan_ready, 0));
      RC(fnb_gat_fwd_tiled(&plan->fbond, &f, sB_));
      if (plan_complete && l == 0 && two) RC((int)cudaStreamWaitEvent(sB, plan_complete, 0));
      if (P.fbond_mask_rows && P.n_fbond_mask_rows > 0) {
        k_zero_rows<<<(int)((P.n_fbond_mask_rows * 32 + 255) / 256), 256, 0, sB>>>(
            pre_fbond, y_fbond, frag ? b.se_frag : nullptr, P.fbond_mask_rows, P.n_fbond_mask_rows);
        FNB_CHECK_LAUNCH();
      }
    }
    const bool pool_out = last && o->pool_frags;
    if (frag || pool_out || P.want_attention) RC(join());
    // ---- gat2_lite's fragment output (gat2_lite.py:140, 205-212): ReLU(Dropout(pooled pre-activation atoms)) at the
    // last layer's fragment site, pooled into out_frags and activated in place
    if (pool_out) {
      RC(fnb_segment_sum(plan->pool_rowptr, plan->pool_col, z.Nf, pre_atom, io->out_frags, kD, nullptr, 0, 0, 0, nullptr,
                         stream_));
      RC(fnb_dropout_relu_fwd(io->out_frags, io->out_frags, z.Nf * kD, o->drop_p, o->training, 1, o->seed, ph.frag[l],
                              stream_));
    }
    // ---- atom -> fragment pooling (gat2.py:234) and the fragment graph (gat2.py:283-316): only where its output lives
    if (frag) {
      RC(fnb_segment_sum(plan->pool_rowptr, plan->pool_col, z.Nf, pre_atom, b.hf, kD, P.f, A_STRIDE, A_T, A_S, b.Sf,
                         stream_));
      fnb_gat_fwd_args f{};
      f.h = b.hf; f.S = b.Sf; f.edge_mode = FNB_EDGE_TABLE; f.edge_table = io->frag_table ? io->frag_table : b.se_frag;
      f.out = pre_frag; f.y = y_frag;
      f.post = post_of(o, ph.frag[l]); f.p_saved = want_p ? b.p_f : nullptr; f.mask_lo = f.mask_hi = -1;
      RC(fnb_gat_fwd_tiled(&plan->frag, &f, stream_));
    }
    if (P.want_attention) {  // by-source attention sums (gat2.py:165,219,268,312)
      if (io->attn_bonds) RC(fnb_attn_by_source(plan->bond.rrowptr, plan->bond.rslot, b.p_b, z.Nb, io->attn_bonds, stream_));
      if (io->attn_atoms) RC(fnb_attn_by_source(plan->atom.rrowptr, plan->atom.rslot, b.p_a, z.Na, io->attn_atoms, stream_));
      if (io->attn_fbonds)
        RC(fnb_attn_by_source(plan->fbond.rrowptr, plan->fbond.rslot, b.p_fb, z.Nfb, io->attn_fbonds, stream_));
      if (io->attn_frags && frag)
        RC(fnb_attn_by_source(plan->frag.rrowptr, plan->frag.rslot, b.p_f, z.Nf, io->attn_frags, stream_));
    }
    xa = y_atom; xb = y_bond; xfb = y_fbond;   // inputs of the next layer (post_act mode only has further layers)
  }
  RC(join());
  return 0;
}

extern "C" int fnb_encoder_backward(const fnb_batch_plan *plan, const fnb_encoder_opts *o, const fnb_layer_params *L,
                                    const fnb_layer_grads *G, const fnb_encoder_io *io, void *workspace,
                                    size_t workspace_bytes, void *bwd_workspace, size_t bwd_workspace_bytes,
                                    void *scratch, void *stream_) {
  RC(check_common(plan, o, L, io));
  if (!G || !workspace || !bwd_workspace || !scratch) return FNB_ERR_NULL;
  if (!o->save_for_backward) return FNB_ERR_MODE;
  LayerBufs B[16];
  BwdBufs W;
  if (layout(plan, o, L, (char *)workspace, B) > workspace_bytes) return FNB_ERR_WORKSPACE;
  if (bwd_layout(plan, o, (char *)bwd_workspace, &W) > bwd_workspace_bytes) return FNB_ERR_WORKSPACE;
  const Sizes z = sizes_of(plan);
  cudaStream_t stream = (cudaStream_t)stream_;
  const float scale = (o->post_act && o->training && o->drop_p > 0.f) ? 1.f / (1.f - o->drop_p) : 1.f;
  bool counters_cleared = false;
  const bool tf32 = fnb_tc_precision(o->precision);
  const int x3 = o->precision == FNB_PRECISION_TF32X3;
  // layers below first_trained_layer are frozen: the pass ends at that layer, which needs no input gradient
  const int first = o->first_trained_layer;

  // W^T of every K = 128 projection in one launch per 16 matrices (used by the tensor-core dX GEMMs)
  int wt_slot[16][3];
  {
    const float *mats[48];
    int nm = 0;
    for (int l = first; l < o->n_layers; ++l) {
      const float *ws[3] = {L[l].Wb, L[l].Wa, L[l].Wfb};
      const int ks[3] = {L[l].K_bond, L[l].K_atom, L[l].K_fbond};
      for (int j = 0; j < 3; ++j) {
        wt_slot[l][j] = -1;
        if (tf32 && ks[j] == kD && !(j == 2 && o->skip_fbond) &&
            (l > first || (l == 0 && (j == 0 ? o->need_dx_bond : (j == 1 ? o->need_dx_atoms : o->need_dx_fbond))))) {
          wt_slot[l][j] = nm;
          mats[nm++] = ws[j];
        }
      }
    }
    for (int c = 0; c < nm; c += 16) {
      TransposeBatch tb{};
      tb.count = nm - c < 16 ? nm - c : 16;
      for (int i = 0; i < tb.count; ++i) tb.W[i] = mats[c + i];
      if (c == 0) {   // the side streams' arrival counters, cleared here instead of by a memset behind every fork
        tb.zero[0] = W.scratch2; tb.zero[1] = W.scratch3; tb.zero[2] = W.scratch4; tb.zero[3] = W.scratch5;
        tb.zero[4] = W.scratch6;
        tb.n_zero = 5;
        counters_cleared = true;
      }
      RC(fnb_tc_transpose128_batched(tb, W.Wt + (size_t)c * kD * kD, stream));
    }
  }
  auto wt_of = [&](int layer, int j) -> const float * {
    return wt_slot[layer][j] >= 0 ? W.Wt + (size_t)wt_slot[layer][j] * kD * kD : nullptr;
  };

  // The fragment-connection blocks of all layers form one chain that only needs the fragment block of the last
  // layer: it runs on the auxiliary stream with its own scratch, concurrently with the atom / bond blocks.
  FnbAux aux{};
  const bool two = fnb_aux_streams(&aux) == 0;
  cudaStream_t sB = two ? aux.stream : stream;
  void *sB_ = (void *)sB;
  void *scratchB = two ? (void *)W.scratch2 : scratch;
  bool forked = false;
  auto fork = [&]() -> int {   // everything queued on the caller's stream so far is visible to sB
    if (two && !forked) {
      RC((int)cudaEventRecord(aux.fork, stream));
      RC((int)cudaStreamWaitEvent(sB, aux.fork, 0));
      if (!counters_cleared) RC((int)cudaMemsetAsync(W.scratch2, 0, kScratchCounters * sizeof(float), sB));
      forked = true;
    }
    return 0;
  };

  // Weight gradients of the atom / bond projections: nothing waits for them before the end of the pass, so they run
  // on a third stream; the caller's stream only waits before it overwrites the dh buffer such a GEMM is reading.
  // (one stream per chain: graph 0 = atom, 1 = bond)
  cudaStream_t sWs[2] = {two ? aux.wstream2 : stream, two ? aux.wstream : stream};
  void *scratchWs[2] = {two ? (void *)W.scratch6 : scratch, two ? (void *)W.scratch3 : scratch};
  bool w_used[2] = {false, false}, w_pending[2][2] = {{false, false}, {false, false}};   // [graph][layer parity]
  auto done_ev = [&](int i, int par) { return par ? aux.done2[i] : aux.done[i]; };
  auto w_begin = [&](int i, cudaStream_t producer) -> int {   // dh of graph i (0 atom, 1 bond) is complete on `producer`
    if (!two) return 0;
    RC((int)cudaEventRecord(aux.ready[i], producer));
    RC((int)cudaStreamWaitEvent(sWs[i], aux.ready[i], 0));
    if (!w_used[i]) {
      if (!counters_cleared) RC((int)cudaMemsetAsync(scratchWs[i], 0, kScratchCounters * sizeof(float), sWs[i]));
      w_used[i] = true;
    }
    return 0;
  };
  auto w_end = [&](int i, int par) -> int {
    if (!two) return 0;
    RC((int)cudaEventRecord(done_ev(i, par), sWs[i]));
    w_pending[i][par] = true;
    return 0;
  };
  // before the dh buffer `par` of graph i is overwritten, i.e. two layers later (or at the end of the pass)
  auto w_wait = [&](int i, int par, cudaStream_t waiter) -> int {
    if (two && w_pending[i][par]) {
      RC((int)cudaStreamWaitEvent(waiter, done_ev(i, par), 0));
      w_pending[i][par] = false;
    }
    return 0;
  };
  // The atom blocks of all layers form a chain of their own (dy_atom of layer l-1 is the dX of layer l's atom
  // projection); it meets the bond chain only where the edge-term kernel needs dz of the atom graph.  It runs on a
  // fourth stream; the bond chain on the caller's stream is the critical path.
  cudaStream_t sA = two ? aux.astream : stream;
  void *sA_ = (void *)sA;
  void *scratchA = two ? (void *)W.scratch4 : scratch;
  bool a_forked = false, a_table_pending = false;
  bool e_used = false, e_pending[2] = {false, false};

  // gradients arriving at the four outputs of the current layer (post-activation copies in post_act mode)
  const float *dy_atom = io->g_atoms, *dy_bond = io->g_bond, *dy_fbond = io->g_fbond, *dy_frag = io->g_frags;
  for (int l = o->n_layers - 1; l >= first; --l) {
    const fnb_layer_params &P = L[l];
    const fnb_layer_grads &D = G[l];
    LayerBufs &b = B[l];
    const bool last = l == o->n_layers - 1;
    const bool frag = P.run_frag_block != 0;
    const float *xa = l == 0 ? (b.xa0 ? b.xa0 : io->x_atoms) : B[l - 1].y_atom;
    const float *xb = l == 0 ? io->x_bond : B[l - 1].y_bond;
    const float *xfb = l == 0 ? io->x_fbond : B[l - 1].y_fbond;
    const float *y_bond = o->post_act ? (last ? io->out_bond : b.y_bond) : nullptr;
    const float *y_atom = o->post_act ? (last ? io->out_atoms : b.y_atom) : nullptr;
    const float *y_fbond = o->post_act ? (last ? io->out_fbond : b.y_fbond) : nullptr;
    const float *y_frag = o->post_act ? (last ? io->out_frags : b.y_frag) : nullptr;
    const float *pre_bond = o->post_act ? b.pre_bond : io->out_bond;
    const float *pre_fbond = o->post_act ? b.pre_fbond : io->out_fbond;
    const bool need_dx = l > first;
    const int par = l & 1;
    float *dh_a = par ? W.dh_a2 : W.dh_a, *dh_b = par ? W.dh_b2 : W.dh_b;
    // dz of the atom graph is double-buffered by layer parity like dh: its last reader, the edge-term kernel that forms
    // d a[:, edge slice], runs on the weight-gradient stream -- on the atom chain it sat between this layer's dX GEMM
    // and the next layer's destination pass, whose dz the bond chain (the critical path) waits for (~40 us per layer,
    // gpurun_out/r4l_device_profile.log)
    float *dz_a = par ? W.dz_a2 : W.dz_a;

    // ---- fragment graph block (only where it ran and a gradient arrives)
    const float *d_hf = nullptr;
    bool frag_bwd = frag && dy_frag != nullptr;
    if (frag_bwd) {
      if (!D.f) return FNB_ERR_NULL;
      fnb_gat_bwd_args a{};
      a.h = b.hf; a.dout = W.g_frag; a.p_saved = b.p_f; a.edge_mode = FNB_EDGE_TABLE; a.alpha = P.f;
      a.alpha_stride = A_STRIDE; a.off_t = A_T; a.off_e = A_E; a.off_s = A_S; a.dz = W.dz_f; a.dSt = W.dSt_f;
      a.dh = W.d_hf; a.d_alpha = D.f; a.d_bias = nullptr; a.scratch = scratch;
      FnbDstFuse fz{};      // ReLU(Dropout) backward of dy_frag inside the destination pass
      fz.dy = dy_frag; fz.y = y_frag; fz.scale = scale;
      // external edge term (gat2_edge): nothing in here writes the edge slice of d f -- it flows back through
      // d_frag_table on the caller's side -- so the whole tensor starts from zero
      if (io->frag_table) RC((int)cudaMemsetAsync(D.f, 0, 4 * A_STRIDE * sizeof(float), stream));
      RC(fnb_gat_bwd_tiled_fused(&plan->frag, &a, &fz, nullptr, nullptr, stream_));
      if (io->frag_table && io->d_frag_table && plan->frag.n_real_edges > 0) {
        const int64_t n = plan->frag.n_real_edges;
        if (cudaError_t le = fnb_launch(k_gather_rows4, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, stream, W.dz_f,
                                        plan->frag.slot_of_eid, io->d_frag_table, n))
          return (int)le;
        FNB_CHECK_LAUNCH();
      }
      d_hf = W.d_hf;
    }
    if (last && o->pool_frags && dy_frag) {   // gat2_lite: the gradient of the pooled rows, dy (y > 0) / (1 - p)
      RC(fnb_dropout_relu_bwd(dy_frag, y_frag, W.d_hf, z.Nf * kD, o->drop_p, o->training, stream_));
      d_hf = W.d_hf;     // the atom graph's destination pass hands it to the member atoms
    }
    const bool frag_feeds_fbond = frag_bwd && !io->frag_table;   // gat2: the fragment graph's edges ARE the fbond rows
    // ---- fragment-connection graph block
    if (!o->skip_fbond) {
      RC(fork());
      // incoming gradient = ReLU(Dropout) backward of dy_fbond + (last layer) the fragment graph's edge term
      // sum_h dz_f alpha_e, assembled inside the destination pass; d f[:, edge slice] by the edge-table kernel
      const bool have = frag_feeds_fbond || dy_fbond != nullptr;
      if (frag_feeds_fbond)
        RC(fnb_edge_table_bwd_fused(&plan->frag, W.dz_f, pre_fbond, P.f, A_STRIDE, A_E, nullptr, nullptr, nullptr, scale,
                                    nullptr, D.f, scratchB, sB_));
      if (have) {
        fnb_gat_bwd_args a{};
        a.h = b.hfb; a.dout = W.g_fbond; a.p_saved = b.p_fb; a.edge_mode = FNB_EDGE_AFFINE6; a.We = P.We_fb;
        a.be = P.be_fb; a.alpha = P.f_a_b; a.alpha_stride = AB_STRIDE; a.off_t = AB_T; a.off_e = AB_E; a.off_s = AB_S;
        a.dz = W.dz_fb; a.dSt = W.dSt_fb; a.dh = W.dh_fb; a.d_alpha = D.f_a_b; a.d_bias = D.bfb; a.dWe = D.We_fb;
        a.dbe = D.be_fb; a.scratch = scratchB;
        FnbDstFuse fz{};
        fz.dz_up = frag_feeds_fbond ? W.dz_f : nullptr; fz.slot_of_eid = plan->frag.slot_of_eid; fz.alpha_up = P.f + A_E;
        fz.alpha_up_stride = A_STRIDE; fz.dy = dy_fbond; fz.y = dy_fbond ? y_fbond : nullptr; fz.scale = scale;
        RC(fnb_gat_bwd_tiled_fused(&plan->fbond, &a, &fz, nullptr, nullptr, sB_));
        float *dx = need_dx ? W.dx_fbond : (l == 0 && o->need_dx_fbond ? io->dx_fbond : nullptr);
        if (l == 0 && b.k_pad[2] && !dx)
          RC(fnb_tc_dw_launch(W.dh_fb, b.x_pad[2], z.Nfb, b.k_pad[2], P.K_fbond, D.Wfb, scratch_body(scratchB), sB, x3));
        else
          RC(fnb_proj_bwd_impl(xfb, P.Wfb, wt_of(l, 2), W.dh_fb, z.Nfb, P.K_fbond, dx, D.Wfb, nullptr, o->precision,
                               scratchB, sB_));
        dy_fbond = need_dx ? W.dx_fbond : nullptr;
      } else {
        dy_fbond = nullptr;
      }
      if (!have) {  // no gradient reaches this block: its parameters get zeros
        RC((int)cudaMemsetAsync(D.f_a_b, 0, 4 * AB_STRIDE * 4, sB));
        RC((int)cudaMemsetAsync(D.bfb, 0, kD * 4, sB));
        RC((int)cudaMemsetAsync(D.We_fb, 0, 32 * 6 * 4, sB));
        RC((int)cudaMemsetAsync(D.be_fb, 0, 32 * 4, sB));
        RC((int)cudaMemsetAsync(D.Wfb, 0, (size_t)kD * P.K_fbond * 4, sB));
      }
    }
    // ---- atom graph block: incoming gradient = activation backward + pooling backward
    {
      const bool have = dy_atom != nullptr || d_hf != nullptr;
      if (have) {
        if (two && !a_forked) {   // the caller's gradients and the fragment block's pooled gradient are visible to sA
          RC((int)cudaEventRecord(aux.a_fork, stream));
          RC((int)cudaStreamWaitEvent(sA, aux.a_fork, 0));
          if (!counters_cleared) RC((int)cudaMemsetAsync(W.scratch4, 0, kScratchCounters * sizeof(float), sA));
          a_forked = true;
        }
        if (two && a_table_pending) {   // the edge-term kernel of the layer above has consumed dz of the atom graph
          RC((int)cudaStreamWaitEvent(sA, aux.a_table, 0));
          a_table_pending = false;
        }
        fnb_gat_bwd_args a{};
        a.h = b.ha; a.dout = W.g_atom; a.p_saved = b.p_a; a.edge_mode = FNB_EDGE_TABLE; a.alpha = P.a;
        a.alpha_stride = A_STRIDE; a.off_t = A_T; a.off_e = A_E; a.off_s = A_S; a.dz = dz_a; a.dSt = W.dSt_a;
        a.dh = dh_a; a.d_alpha = D.a; a.d_bias = D.ba; a.scratch = scratchA;
        RC(w_wait(0, par, sA));
        if (two && e_pending[par]) {      // the edge-term kernel two layers up has read this parity's dz buffer
          RC((int)cudaStreamWaitEvent(sA, aux.e_done[par], 0));
          e_pending[par] = false;
        }
        // the bond graph's destination pass (caller's stream) only needs dz of this graph: the event sits between the
        // two launches
        FnbDstFuse fza{};     // ReLU(Dropout) backward of dy_atom + pooling backward of the fragment gradient
        fza.dy = dy_atom; fza.y = dy_atom ? y_atom : nullptr; fza.scale = scale; fza.pool = d_hf; fza.seg_of = plan->a2f;
        RC(fnb_gat_bwd_tiled_fused(&plan->atom, &a, &fza, two ? aux.a_dz : nullptr, nullptr, sA_));
        if (two) RC((int)cudaStreamWaitEvent(stream, aux.a_dz, 0));
        RC(w_begin(0, sA));
        float *dx = need_dx ? W.dx_atom : (l == 0 && o->need_dx_atoms ? io->dx_atoms : nullptr);
        // layer 0 with padded operands: d Wa always from the padded copy, which holds exactly what the forward
        // multiplied (dropped or not).  The unpadded dropped copy xa0 exists only if the forward call already had
        // need_dx_atoms set; with input dropout applied inside the padding kernel it was never written.
        if (dx) RC(fnb_proj_bwd_dx(P.Wa, wt_of(l, 1), dh_a, z.Na, P.K_atom, dx, o->precision, scratchA, sA_));
        if (l == 0 && b.k_pad[1])
          RC(fnb_tc_dw_launch(dh_a, b.x_pad[1], z.Na, b.k_pad[1], P.K_atom, D.Wa, scratch_body(scratchWs[0]), sWs[0], x3));
        else
          RC(fnb_proj_bwd_dw(xa, dh_a, z.Na, P.K_atom, D.Wa, nullptr, o->precision, scratchWs[0], (void *)sWs[0]));
        RC(w_end(0, par));
        // bond features were this graph's edge vectors (gat2.py:203-208): the head-vector gradient of that term is
        // nobody's input.  On the atom chain it delayed the next layer's dz (which the bond chain, the critical path,
        // waits for) by ~40 us per layer; behind the weight-gradient GEMMs it piled up at the end of the pass
        // (gpurun_out/r4l, r4m): it gets a stream of its own and this parity's dz buffer to itself until e_done[par].
        // The row gradient is assembled inside the bond graph's destination pass.
        if (two) {
          RC((int)cudaEventRecord(aux.e_ready, sA));
          RC((int)cudaStreamWaitEvent(aux.estream, aux.e_ready, 0));
          if (!e_used) {
            if (!counters_cleared) RC((int)cudaMemsetAsync(W.scratch5, 0, kScratchCounters * sizeof(float), aux.estream));
            e_used = true;
          }
          RC(fnb_edge_table_bwd_fused(&plan->atom, dz_a, pre_bond, P.a, A_STRIDE, A_E, nullptr, nullptr, nullptr, scale,
                                      nullptr, D.a, W.scratch5, (void *)aux.estream));
          RC((int)cudaEventRecord(aux.e_done[par], aux.estream));
          e_pending[par] = true;
        } else {
          RC(fnb_edge_table_bwd_fused(&plan->atom, dz_a, pre_bond, P.a, A_STRIDE, A_E, nullptr, nullptr, nullptr, scale,
                                      nullptr, D.a, scratchA, sA_));
        }
        dy_atom = need_dx ? W.dx_atom : nullptr;
      } else {
        RC((int)cudaMemsetAsync(D.a, 0, 4 * A_STRIDE * 4, stream));
        RC((int)cudaMemsetAsync(D.ba, 0, kD * 4, stream));
        RC((int)cudaMemsetAsync(D.Wa, 0, (size_t)kD * P.K_atom * 4, stream));
        dy_atom = nullptr;
      }
      // ---- bond graph block
      if (have || dy_bond) {
        fnb_gat_bwd_args a{};
        a.h = b.hb; a.dout = W.g_bond; a.p_saved = b.p_b; a.edge_mode = FNB_EDGE_AFFINE1; a.We = P.We_b; a.be = P.be_b;
        a.alpha = P.a_b; a.alpha_stride = AB_STRIDE; a.off_t = AB_T; a.off_e = AB_E; a.off_s = AB_S; a.dz = W.dz_b;
        a.dSt = W.dSt_b; a.dh = dh_b; a.d_alpha = D.a_b; a.d_bias = D.bb; a.dWe = D.We_b; a.dbe = D.be_b;
        a.scratch = scratch;
        // incoming gradient = edge term of the atom graph (dz_a) + ReLU(Dropout) backward of dy_bond, assembled by
        // the destination pass; the atom chain may overwrite dz_a once that launch is done
        FnbDstFuse fz{};
        fz.dz_up = have ? dz_a : nullptr; fz.slot_of_eid = plan->atom.slot_of_eid; fz.alpha_up = P.a + A_E;
        fz.alpha_up_stride = A_STRIDE; fz.g_base = y_bond ? nullptr : dy_bond; fz.dy = y_bond ? dy_bond : nullptr;
        fz.y = y_bond && dy_bond ? y_bond : nullptr; fz.scale = scale;
        // (the weight-gradient GEMM two layers above read this dh buffer: only the source pass has to wait for it)
        const bool wait_w = two && w_pending[1][par];
        w_pending[1][par] = false;
        RC(fnb_gat_bwd_tiled_fused(&plan->bond, &a, &fz, two && have ? aux.a_table : nullptr,
                                   wait_w ? done_ev(1, par) : nullptr, stream_));
        if (two && have) a_table_pending = true;
        RC(w_begin(1, stream));
        float *dx = need_dx ? W.dx_bond : (l == 0 && o->need_dx_bond ? io->dx_bond : nullptr);
        if (l == 0 && b.k_pad[0] && !dx) {
          RC(fnb_tc_dw_launch(dh_b, b.x_pad[0], z.Nb, b.k_pad[0], P.K_bond, D.Wb, scratch_body(scratchWs[1]), sWs[1], x3));
        } else {
          RC(fnb_proj_bwd_dx(P.Wb, wt_of(l, 0), dh_b, z.Nb, P.K_bond, dx, o->precision, scratch, stream_));
          RC(fnb_proj_bwd_dw(xb, dh_b, z.Nb, P.K_bond, D.Wb, nullptr, o->precision, scratchWs[1], (void *)sWs[1]));
        }
        RC(w_end(1, par));
        dy_bond = need_dx ? W.dx_bond : nullptr;
      } else {
        RC((int)cudaMemsetAsync(D.a_b, 0, 4 * AB_STRIDE * 4, stream));
        RC((int)cudaMemsetAsync(D.bb, 0, kD * 4, stream));
        RC((int)cudaMemsetAsync(D.We_b, 0, 32 * 4, stream));
        RC((int)cudaMemsetAsync(D.be_b, 0, 32 * 4, stream));
        RC((int)cudaMemsetAsync(D.Wb, 0, (size_t)kD * P.K_bond * 4, stream));
        dy_bond = nullptr;
      }
    }
    if (!frag_bwd && D.f) RC((int)cudaMemsetAsync(D.f, 0, 4 * A_STRIDE * 4, stream));
    dy_frag = nullptr;   // the fragment output of a lower layer is dead (overwritten unread, gat2.py:234)
  }
  if (two && forked) {
    RC((int)cudaEventRecord(aux.join, sB));
    RC((int)cudaStreamWaitEvent(stream, aux.join, 0));
  }
  if (two && a_forked) {
    RC((int)cudaEventRecord(aux.a_join, sA));
    RC((int)cudaStreamWaitEvent(stream, aux.a_join, 0));
  }
  for (int i = 0; i < 2; ++i)
    for (int p2 = 0; p2 < 2; ++p2) RC(w_wait(i, p2, stream));
  if (two && e_used) {
    RC((int)cudaEventRecord(aux.e_join, aux.estream));
    RC((int)cudaStreamWaitEvent(stream, aux.e_join, 0));
  }
  // input dropout backward (gat2.py:396) when the caller wants d x_atoms: same RNG stream as the forward
  if (first == 0 && o->need_dx_atoms && io->dx_atoms && input_dropout(o)) {
    const RngPlan ph = rng_plan(plan, o, L);
    RC(fnb_dropout_relu_fwd(io->dx_atoms, io->dx_atoms, z.Na * (int64_t)L[0].K_atom, o->drop_p, 1, 0, o->seed, ph.input,
                            stream_));
  }
  return 0;
}
