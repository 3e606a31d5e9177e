// Shared device helpers for the fragnet_b200 kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "fragnet_b200.h"

#define FNB_ERR_NULL -1      // required pointer is NULL
#define FNB_ERR_SIZE -2      // negative / overflowing size
#define FNB_ERR_MODE -3      // unknown mode / unsupported width
#define FNB_ERR_WORKSPACE -4 // workspace too small
#define FNB_ERR_ALIGN -5     // pointer not 16-byte aligned

constexpr int kD = FNB_D;          // 128 features per node
constexpr int kH = FNB_H;          // 4 heads
constexpr int kHd = kD / kH;       // 32 features per head
constexpr float kNegSlope = 0.2f;  // nn.LeakyReLU(0.2), reference gat2.py:83
constexpr int kNumSMs = 148;       // B200
constexpr unsigned kFull = 0xffffffffu;

// Scratch floats a caller must provide to the backward entry points (fnb_scratch_bytes): the widest
// user is the projection weight gradient, kNumSMs CTAs x (128 x (K<=256) + 128) floats.
constexpr int kProjBwdMaxK = 256;
// The first kScratchCounters floats of every scratch buffer hold the arrival counters of cta_finish (zero between
// launches); everything else starts at scratch_body().
constexpr int kScratchCounters = 64;
constexpr size_t kScratchFloats = kScratchCounters + (size_t)kNumSMs * (128 * kProjBwdMaxK + 128);
static inline float *scratch_body(void *scratch) { return reinterpret_cast<float *>(scratch) + kScratchCounters; }

// Diagnostic only (bench.py's "gpu_launches"): kernels launched by this library in this process.
extern unsigned long long g_fnb_launches;
#define FNB_CHECK_LAUNCH()                              \
  do {                                                  \
    cudaError_t e__ = cudaGetLastError();               \
    if (e__ != cudaSuccess) return (int)e__;            \
    __atomic_fetch_add(&g_fnb_launches, 1ull, __ATOMIC_RELAXED); \
  } while (0)
// Returns a non-zero status (FNB_ERR_* or a cudaError_t) to the caller.
#define RC(expr)             \
  do {                       \
    const int rc__ = (expr); \
    if (rc__) return rc__;   \
  } while (0)
static inline bool fnb_aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
__device__ __forceinline__ bool fnb_is_aligned16_dev(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// Workspace carving: every buffer starts on a 256-byte boundary.  base == NULL only measures (take() returns NULL).
struct Arena {
  char *base;
  size_t off;
  template <class T>
  T *take(size_t n) {
    off = (off + 255) & ~(size_t)255;
    T *p = base ? reinterpret_cast<T *>(base + off) : nullptr;
    off += n * sizeof(T);
    return p;
  }
  char *bytes(size_t n) { return take<char>(n); }
  size_t total() const { return (off + 255) & ~(size_t)255; }   // bytes of the layout, a multiple of 256
};

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(kFull, v, o));
  return v;
}
// Sum over the 8 lanes that hold one head (lanes 8h .. 8h+7).
__device__ __forceinline__ float head_sum(float v) {
  v += __shfl_xor_sync(kFull, v, 1);
  v += __shfl_xor_sync(kFull, v, 2);
  v += __shfl_xor_sync(kFull, v, 4);
  return v;
}
__device__ __forceinline__ float dot4(const float4 &a, const float4 &b) {
  return a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w;
}
__device__ __forceinline__ float4 ldg4(const float *p) { return __ldg(reinterpret_cast<const float4 *>(p)); }
__device__ __forceinline__ float4 ld4(const float *p) { return *reinterpret_cast<const float4 *>(p); }
__device__ __forceinline__ void st4(float *p, const float4 &v) { *reinterpret_cast<float4 *>(p) = v; }
__device__ __forceinline__ float pick(const float4 &v, int i) {
  return i == 0 ? v.x : (i == 1 ? v.y : (i == 2 ? v.z : v.w));
}
__device__ __forceinline__ float leaky(float z) { return z > 0.f ? z : kNegSlope * z; }

// ---- programmatic dependent launch (PDL) ---------------------------------------------------------------------------
// A step is ~140 short kernels (10-40 us) in stream order; with the programmatic-stream-serialization attribute the
// next kernel's CTAs are scheduled while the last CTAs of the previous one drain, and block in pdl_wait() until the
// previous grid has completed and flushed.  Every kernel launched through fnb_launch() calls pdl_wait() before its
// first access to global memory and pdl_launch_dependents() once its main loop is done.  Both are no-ops for a
// kernel launched without the attribute (FNB_PDL=0 in the environment turns the attribute off).
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
bool fnb_pdl_enabled();
template <class... KArgs, class... Args>
inline cudaError_t fnb_launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                              Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = fnb_pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---- counter-based RNG for dropout masks (regenerated from (seed, counter), never stored) ------
// Philox4x32-10 cost ~135 instructions per group of 4 elements and made the fused forward epilogue the largest single
// consumer of issue slots (profiles/r1e: ~190 of ~407 warp instructions per node).  Dropout only needs independent,
// reproducible Bernoulli draws, so each group of 4 consecutive elements draws two 32-bit words from a 3-multiply
// integer mixer ("triple32", full avalanche) keyed by (seed, counter) and uses 16 bits per element:
// keep <=> r16 >= round(p * 65536).  ~35 instructions per group.
__device__ __forceinline__ uint32_t mix32(uint32_t x) {
  x ^= x >> 17; x *= 0xed5ad4bbu;
  x ^= x >> 11; x *= 0xac4c1b51u;
  x ^= x >> 15; x *= 0x31848babu;
  x ^= x >> 14;
  return x;
}

// ReLU(Dropout_p(v)) of the 4 consecutive elements with flat index 4*q .. 4*q+3; the counter of the group is
// offset + q, so a fused epilogue and the standalone elementwise kernel draw the same mask for the same element.
struct PostAct {
  float p, scale;      // drop probability, 1/(1-p)
  int training, relu;
  uint64_t seed, offset;
};
__device__ __forceinline__ uint2 dropout_bits(uint64_t seed, uint64_t counter) {
  const uint32_t lo = (uint32_t)counter, hi = (uint32_t)(counter >> 32);
  const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
  const uint32_t a = mix32(lo ^ k0) ^ (hi * 0x9E3779B1u);
  return make_uint2(mix32(a + k1), mix32(a ^ 0x85EBCA6Bu ^ k1));
}
__device__ __forceinline__ uint32_t dropout_threshold(float p) { return (uint32_t)(p * 65536.0f + 0.5f); }
__device__ __forceinline__ float4 post_act(const PostAct &pa, float4 v, uint64_t q) {
  if (pa.training && pa.p > 0.f) {
    const uint2 r = dropout_bits(pa.seed, pa.offset + q);
    const uint32_t th = dropout_threshold(pa.p);
    v.x *= (r.x & 0xffffu) >= th ? pa.scale : 0.f;
    v.y *= (r.x >> 16) >= th ? pa.scale : 0.f;
    v.z *= (r.y & 0xffffu) >= th ? pa.scale : 0.f;
    v.w *= (r.y >> 16) >= th ? pa.scale : 0.f;
  }
  if (pa.relu) {
    v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f);
  }
  return v;
}

// Full-warp sums of 4 values in 6 shuffles: on return every lane of head group k = lane/8 holds sum_lanes v[k].
__device__ __forceinline__ float warp_sum4(float v0, float v1, float v2, float v3) {
  const int lane = threadIdx.x & 31;
  const bool hi16 = lane & 16, hi8 = lane & 8;
  float x0 = hi16 ? v2 : v0, y0 = hi16 ? v0 : v2;
  float x1 = hi16 ? v3 : v1, y1 = hi16 ? v1 : v3;
  x0 += __shfl_xor_sync(kFull, y0, 16);
  x1 += __shfl_xor_sync(kFull, y1, 16);
  float z = hi8 ? x1 : x0, w = hi8 ? x0 : x1;
  z += __shfl_xor_sync(kFull, w, 8);
  z += __shfl_xor_sync(kFull, z, 4);
  z += __shfl_xor_sync(kFull, z, 2);
  z += __shfl_xor_sync(kFull, z, 1);
  return z;
}

// ---- deterministic parameter-gradient reduction without a second launch -----------------------
// Every CTA deposits one record of W floats; the last CTA of each group of 32 sums its group in CTA order, the last
// group to finish sums the group records in group order into s_final[W] (shared memory) and returns true in that one
// CTA (all its threads), after resetting the counters for the next launch on the stream.  Fixed summation tree =>
// run-to-run deterministic, no floating-point atomics, no extra launch.
// scratch layout (floats): [0,64) int counters (zero before first use) | [64, 64+64*W) group records | CTA records.
constexpr int kFinishGroup = 32;
template <int W>
__device__ __forceinline__ bool cta_finish(const float *s_rec, float *s_final, float *scratch) {
  __shared__ int s_last;
  int *counters = reinterpret_cast<int *>(scratch);
  float *grp = scratch + 64;
  float *rec = grp + 64 * W;
  const int b = blockIdx.x, nb = gridDim.x, g = b / kFinishGroup, ng = (nb + kFinishGroup - 1) / kFinishGroup;
  const int gsize = min(kFinishGroup, nb - g * kFinishGroup);
  for (int j = threadIdx.x; j < W; j += blockDim.x) rec[(int64_t)b * W + j] = s_rec[j];
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(&counters[1 + g], 1) == gsize - 1;
  __syncthreads();
  if (!s_last) return false;
  __threadfence();
  for (int j = threadIdx.x; j < W; j += blockDim.x) {
    const float *src = rec + (int64_t)g * kFinishGroup * W + j;
    float s = 0.f;
    for (int k = 0; k < gsize; ++k) s += __ldcg(src + (int64_t)k * W);
    grp[g * W + j] = s;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(&counters[0], 1) == ng - 1;
  __syncthreads();
  if (!s_last) return false;
  __threadfence();
  for (int j = threadIdx.x; j < W; j += blockDim.x) {
    float s = 0.f;
    for (int k = 0; k < ng; ++k) s += __ldcg(grp + k * W + j);
    s_final[j] = s;
  }
  if (threadIdx.x <= ng) counters[threadIdx.x] = 0;
  __syncthreads();
  return true;
}
constexpr size_t finish_scratch_floats(int W, int n_ctas) { return 64 + (size_t)64 * W + (size_t)n_ctas * W; }

// Up to 4 output segments of one partial record, reduced by a single launch (reduce.cu).
struct ReduceSegments {
  int n;
  int rec_off[4];       // float offset of the segment inside a record
  int width[4];         // number of columns
  int padded_width[4];  // filled by the launcher
  float *out[4];
  int row_len[4];       // out index = (j / row_len) * out_stride + j % row_len
  int valid_len[4];     // columns j % row_len >= valid_len are padding and are skipped (0 = row_len)
  int out_stride[4];
};
int fnb_launch_reduce_segments(const float *partials, int n_blocks, int pstride, ReduceSegments segs,
                               cudaStream_t stream);

// Auxiliary stream of the calling thread's current device (abi.cu); returns non-zero when only the caller's stream
// should be used.
struct FnbAux {
  cudaStream_t stream;       // independent chains (fragment-connection graph, energy head)
  cudaEvent_t fork, join;
  cudaStream_t wstream;      // weight-gradient GEMMs: nothing downstream waits for them until the end of the pass
  cudaStream_t wstream2;     // ... of the atom chain (encoder backward): the last bond-graph GEMM of a step, whose operand
                             // arrives last, then does not queue behind the atom chain's (20 us of the step's tail)
  cudaEvent_t ready[2], done[2], done2[2], wjoin;   // done / done2: even / odd layers (dh is double-buffered)
  cudaStream_t astream;      // atom-graph chain (it only meets the bond chain at the edge-term kernels)
  cudaEvent_t a_fork, a_dz, a_table, a_join;
  cudaEvent_t plan_fwd;      // forward half of the batch plan is complete (plan.cu)
  cudaStream_t estream;      // head-vector gradients of the 128-wide edge terms (nobody's input: off every chain)
  cudaEvent_t e_ready, e_done[2], e_join;
  cudaStream_t hstream;      // energy head (~1e3 rows, latency-bound): off the fragment-connection chain's stream
  cudaEvent_t h_done;
  cudaStream_t pstream;      // batch plan of the NEXT step (fnb_pretrain_plan_prefetch)
  cudaEvent_t p_fwd, p_done, step_begin;
};
int fnb_aux_streams(FnbAux *out);

// Destination pass of the attention backward with the incoming gradient assembled in the same launch (gat_tiled.cu:
// dst_grad_row): args->dout is WRITTEN by the destination pass and read by the source pass.  Between the two launches `after_dst`
// (optional) is recorded and `before_src` (optional) is waited for.
struct FnbDstFuse {
  const float *dz_up;        // [E_up,4] dz of the consumer graph (its real edge e = this graph's node e), or NULL
  const int *slot_of_eid;    // consumer graph's edge id -> slot
  const float *alpha_up;     // consumer head vector at its edge slice, [4, alpha_up_stride]
  int alpha_up_stride;
  const float *g_base, *dy, *y;   // y == NULL: dy is taken as is (bare-layer mode)
  float scale;
  const float *pool;         // [n_seg,128] gradient of sum-pooled rows to hand back to their members, or NULL
  const int *seg_of;         // [N]
};
int fnb_gat_bwd_tiled_fused(const fnb_graph *g, const fnb_gat_bwd_args *args, const FnbDstFuse *fuse,
                            cudaEvent_t after_dst, cudaEvent_t before_src, void *stream);

int fnb_encoder_forward_impl(const fnb_batch_plan *plan, const fnb_encoder_opts *opts, const fnb_layer_params *layers,
                             const fnb_encoder_io *io, void *workspace, size_t workspace_bytes, void *scratch,
                             void *stream, cudaEvent_t plan_ready, cudaEvent_t plan_complete);
int fnb_batch_plan_build_impl(const fnb_batch_inputs *in, void *arena, size_t arena_bytes, fnb_batch_plan *out,
                              void *stream, cudaEvent_t forward_ready);
// The plan struct of an arena that fnb_batch_plan_build filled (or is filling) for `in`: pointers only, no launch.
int fnb_batch_plan_view(const fnb_batch_inputs *in, void *arena, size_t arena_bytes, fnb_batch_plan *out);
int fnb_pretrain_heads_backward_impl(const fnb_pretrain_head_params *P, const fnb_pretrain_head_grads *D,
                                     const fnb_pretrain_head_io *io, int precision, void *workspace,
                                     size_t workspace_bytes, void *bwd_workspace, size_t bwd_workspace_bytes,
                                     void *scratch, void *stream, int defer_join, const fnb_mse_term *fused,
                                     float *loss_out);
int fnb_pretrain_heads_forward_impl(const fnb_pretrain_head_params *P, const fnb_pretrain_head_io *io, int precision,
                                    void *workspace, size_t workspace_bytes, void *scratch, void *stream,
                                    int skip_tails);

// Exact FP32 GEMM (proj.cu: k_mlp_gemm, FFMA, one k-ascending chain per output), for the projections' SIMT path and
// the finetuning head.  C[M,N] = sum_k A(m,k) B(k,n):
//   GEMM_FWD: A = x [M, K], B = W [N, K] (nn.Linear weight); epilogue z = acc (+ bias); z *= drop1; u = z;
//             C = act(z) * drop2, and optionally S (below).
//   GEMM_DX:  A = dz [M, K], B = W [K, N]; epilogue C = acc * drop1 * act'(u) * drop2 (u == NULL: no activation).
//   GEMM_DW:  through fnb_gemm_dw.
struct Drop {                       // one dropout site: element i of a [rows, width] tensor draws from base + i / 4
  float p, scale;
  uint64_t base;
  int on;
};
Drop fnb_drop(float p, int training, uint64_t base);
enum { GEMM_FWD = 0, GEMM_DX = 1, GEMM_DW = 2 };
struct GemmArgs {
  const float *A, *B;
  int M, N, K;
  float *C;
  uint64_t seed;
  const float *bias;        // FWD: [N] or NULL
  Drop drop1, drop2;
  int act;
  float *u;                 // FWD: written (may be NULL); DX: read (NULL = no activation between the layers)
  // FWD, N = 128 and no dropout or activation: S[m, h] = <C[m, 32h:32h+32], alpha[h, off_t:off_t+32]>, S[m, 4+h]
  // likewise at off_s (the per-node logit halves of the projections); NULL: not written
  const float *alpha;
  int alpha_stride, off_t, off_s;
  float *S;
  // DW (set by fnb_gemm_dw): per-chunk records [M*N dW | M db], record z at rec + z * rec_stride
  int k_chunk;
  float *rec;
  int64_t rec_stride;
};
int fnb_gemm(int mode, const GemmArgs &a, cudaStream_t stream);
// dW[out, in] = dz^T x and db[out] = column sums of dz (db may be NULL) over `rows` rows of dz [rows, out] and
// x [rows, in]: per-chunk records in `rec` (fnb_gemm_dw_record_floats), summed in a fixed order.
int fnb_gemm_dw(const float *dz, const float *x, int64_t rows, int out, int in, float *dW, float *db, float *rec,
                cudaStream_t stream);
size_t fnb_gemm_dw_record_floats(int64_t rows, int out, int in);

// Finetuning head (finetune.cu).  One run of an fnb_mlp_layer list over G rows; every buffer is caller-provided.
struct FnbMlpRun {
  const fnb_mlp_layer *L;
  int n;
  int64_t G;
  int training;
  uint64_t seed;
  uint64_t in_base[FNB_MLP_MAX_LAYERS], out_base[FNB_MLP_MAX_LAYERS];   // fnb_mlp_rng
  float *x0;                        // [G, L[0].in_dim] head input
  float *xd[FNB_MLP_MAX_LAYERS];    // [G, L[l].in_dim] what layer l multiplies; xd[0] == x0 when nothing drops there
  float *u[FNB_MLP_MAX_LAYERS];     // [G, L[l].out_dim] pre-activation of the hidden layers (NULL: not kept; the
                                    // backward reads u[l] where layer l + 1's input gradient runs)
  float *out;                       // [G, L[n-1].out_dim] predictions
  float *dz[FNB_MLP_MAX_LAYERS];    // backward: [G, L[l].out_dim] gradient of layer l's pre-dropout output; dz[n-1] is input
  float *dx0;                       // backward: [G, L[0].in_dim] gradient of x0 (NULL: not wanted)
  float *rec;                       // backward: fnb_mlp_dw_record_floats() floats
};
int fnb_mlp_check(const fnb_mlp_layer *L, int n, int64_t G, int in0, int backward);
uint64_t fnb_mlp_rng(const fnb_mlp_layer *L, int n, int64_t G, uint64_t offset, uint64_t *in_base, uint64_t *out_base);
// Weight-gradient records of the trained layers (dW != NULL).
size_t fnb_mlp_dw_record_floats(const fnb_mlp_layer *L, int n, int64_t G);
// Whether the backward runs layer l's input-gradient GEMM: a trained layer lies below l, or (want_dx0) the caller wants
// the gradient of the head input.
bool fnb_mlp_needs_dx(const fnb_mlp_layer *L, int l, bool want_dx0);
int fnb_mlp_forward(const FnbMlpRun *r, cudaStream_t stream);
int fnb_mlp_backward(const FnbMlpRun *r, cudaStream_t stream);
// loss[0] = mean of BCE-with-logits over the labels > -0.5 (NaN if none); grad (may be NULL) = its logit gradient.
int fnb_bce_masked_loss(const float *logits, const float *labels, int64_t n, float *loss, float *grad,
                        cudaStream_t stream);
// gat2_edge's fragment edge table (gat2_edge.py:152-158) and its gradient, exact FP32 (finetune.cu).  cnx: [n,8]
// connection attributes, W8 / b8: cnx_attr_transform [128,8] / [128], f: the last layer's head vectors [4,192].
//   table[e,h] = sum_k cnx[e,k] coef[k,h] + bias[h],  coef = W8^T f_e^T [8,4],  bias = b8 f_e^T [4],  f_e = f[:, 32:160]
// The backward writes dW8, db8 and the edge slice df[:, 32:160] (the rest of df is left alone); scratch: a step
// scratch whose arrival counters are zero (cta_finish).
int fnb_cnx_table_fwd(const float *cnx, int64_t n, const float *W8, const float *b8, const float *f, float *table,
                      cudaStream_t stream);
int fnb_cnx_table_bwd(const float *cnx, const float *d_table, int64_t n, const float *W8, const float *b8,
                      const float *f, float *dW8, float *db8, float *df, void *scratch, cudaStream_t stream);

// Tensor-core (tcgen05, TF32) projection path, tc_gemm.cu.  Returns FNB_ERR_MODE when the shape cannot use TMA.
// x3 != 0: 3xTF32 (error-compensated, FP32-grade) instead of one TF32 product.
int fnb_tc_proj_launch(const float *A, const float *B, const float *bias, int64_t M, int K, const float *alpha,
                       int alpha_stride, int off_t, int off_s, float *C, float *S, cudaStream_t stream, int x3);
int fnb_tc_transpose128_launch(const float *W, float *Wt, cudaStream_t stream);
// Up to 16 [128,128] matrices transposed by one launch: Wt_base + i * 128 * 128 = Ws[i]^T.
// zero[0..n_zero): scratch buffers whose arrival counters (first kScratchCounters floats) the launch clears on the way --
// the backward program's side streams then need no memset of their own between their fork and their first kernel.
struct TransposeBatch { const float *W[16]; int count; float *zero[6]; int n_zero; };
int fnb_tc_transpose128_batched(const TransposeBatch &b, float *Wt_base, cudaStream_t stream);
int fnb_proj_bwd_impl(const float *x, const float *W, const float *Wt_pre, const float *dh, int64_t n_rows, int K,
                      float *dx, float *dW, float *db, int precision, void *scratch, void *stream);
int fnb_proj_bwd_dx(const float *W, const float *Wt_pre, const float *dh, int64_t n_rows, int K, float *dx, int precision,
                    void *scratch, void *stream);
int fnb_proj_bwd_dw(const float *x, const float *dh, int64_t n_rows, int K, float *dW, float *db, int precision,
                    void *scratch, void *stream);
int fnb_tc_dw_launch(const float *dh, const float *x, int64_t n_rows, int x_cols, int k_out, float *dW, float *scratch,
                     cudaStream_t stream, int x3);
static inline bool fnb_tc_precision(int precision) {
  return precision == FNB_PRECISION_TF32 || precision == FNB_PRECISION_TF32X3;
}
