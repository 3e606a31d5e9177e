// The finetuning head (FTHead1-4 of FragNetFineTune, fragnet/model/gat/gat2.py:569-751) forward and backward, and the
// masked BCE-with-logits loss of TrainerFineTune (fragnet/train/utils.py:296-303, :406-470).
//
// A head is a list of linear layers (fnb_mlp_layer), each  y = act(drop_out(drop_in(x) W^T + b)).  Every layer is one
// launch of the library's FP32 FFMA GEMM (k_mlp_gemm, proj.cu: 64 x 64 tile, 4 x 4 outputs per thread) whose epilogue
// applies the bias, the dropout masks and the activation; the heads stay exact FP32 in every precision mode (as
// k_energy_head does for the energy head): rows are molecules (128 to a few thousand) and widths are whatever a hyper-parameter search picks,
// shapes the N = 128 tensor-core kernels do not cover.
//
// Buffers of a run (FnbMlpRun): xd[l] is what layer l multiplies (its input after its input dropout), u[l] its output
// after output dropout and before the activation.  The epilogue of layer l writes u[l] and xd[l+1] = drop_in_{l+1}(act(u[l]));
// the head input's own input dropout (FTHead1 / FTHead4) is one standalone dropout launch.  The backward needs no
// stored mask: the masks are regenerated from the counter hash of common.cuh.
//
// Backward, layer l from the last down:  dW_l = dz_l^T xd[l], db_l = column sums of dz_l (per-CTA partial records over
// row chunks, summed in a fixed order by k_reduce_partials: deterministic, no floating-point atomics), and one GEMM
// dz_l W_l whose epilogue folds what lies between xd[l] and u[l-1] -- the replayed input mask of layer l, the derivative
// of layer l-1's activation at u[l-1] and layer l-1's output mask -- so it writes dz_{l-1} directly (for l = 0: the
// gradient of the head input).  Each of these factors is evaluated once per element.  A frozen layer (dW = db = NULL)
// skips its weight-gradient GEMM and reduction; the input-gradient GEMMs stop where no trained layer lies below and the
// caller wants no gradient of the head input (dx0 = NULL).
#include <algorithm>

#include "common.cuh"

namespace {

// ---- masked BCE-with-logits (TrainerFineTune._bce): one CTA, fixed summation order -----------------------------------
constexpr int kBceThreads = 1024;
__global__ void __launch_bounds__(kBceThreads) k_bce_masked(const float *__restrict__ x, const float *__restrict__ y,
                                                             int64_t n, float *__restrict__ loss,
                                                             float *__restrict__ grad) {
  __shared__ float s_sum[kBceThreads / 32], s_cnt[kBceThreads / 32];
  __shared__ float s_inv;
  pdl_wait();
  float acc = 0.f, cnt = 0.f;
  for (int64_t i = threadIdx.x; i < n; i += kBceThreads) {
    const float xi = __ldg(x + i), yi = __ldg(y + i);
    if (yi > -0.5f) {
      acc += fmaxf(xi, 0.f) - xi * yi + log1pf(expf(-fabsf(xi)));
      cnt += 1.f;
    }
  }
  acc = warp_sum(acc);
  cnt = warp_sum(cnt);
  if ((threadIdx.x & 31) == 0) {
    s_sum[threadIdx.x >> 5] = acc;
    s_cnt[threadIdx.x >> 5] = cnt;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f, c = 0.f;
    for (int w = 0; w < kBceThreads / 32; ++w) {
      s += s_sum[w];
      c += s_cnt[w];
    }
    loss[0] = s / c;                         // no valid label: 0 / 0 = NaN, as the reference
    s_inv = 1.f / c;
  }
  __syncthreads();
  if (!grad) return;
  const float inv = s_inv;
  for (int64_t i = threadIdx.x; i < n; i += kBceThreads) {
    const float xi = __ldg(x + i), yi = __ldg(y + i);
    grad[i] = yi > -0.5f ? (1.f / (1.f + expf(-xi)) - yi) * inv : 0.f;
  }
}

// ---- gat2_edge's fragment edge table --------------------------------------------------------------------------------
// <cnx_attr_transform(cnx[e]), f_e[h]> = cnx[e] . (W8^T f_e[h]) + <b8, f_e[h]>: the 36 folded constants (coef[k,h] at
// k * 4 + h, bias[h] at 32 + h) are formed per CTA in a fixed order, one warp per constant.
constexpr int kCnxIn = 8, kCnxThreads = 256, kCnxConst = kCnxIn * kH + kH;
constexpr int kFStride = 192, kFEdge = 32;      // f = [target 32 | edge 128 | source 32] per head

__device__ __forceinline__ void cnx_fold(const float *__restrict__ W8, const float *__restrict__ b8,
                                         const float *__restrict__ f, float *s_c) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int o = warp; o < kCnxConst; o += kCnxThreads / 32) {
    const int k = o >> 2, h = o & 3;              // k == kCnxIn: the bias term
    float s = 0.f;
    for (int j = lane; j < kD; j += 32)
      s += (k < kCnxIn ? __ldg(W8 + j * kCnxIn + k) : __ldg(b8 + j)) * __ldg(f + h * kFStride + kFEdge + j);
    s = warp_sum(s);
    if (lane == 0) s_c[o] = s;
  }
  __syncthreads();
}

__device__ __forceinline__ void cnx_row(const float *__restrict__ cnx, int64_t e, float x[kCnxIn]) {
  const float4 lo = ldg4(cnx + e * kCnxIn), hi = ldg4(cnx + e * kCnxIn + 4);
  x[0] = lo.x; x[1] = lo.y; x[2] = lo.z; x[3] = lo.w; x[4] = hi.x; x[5] = hi.y; x[6] = hi.z; x[7] = hi.w;
}

__global__ void __launch_bounds__(kCnxThreads) k_cnx_table(const float *__restrict__ cnx, int64_t n,
                                                           const float *__restrict__ W8, const float *__restrict__ b8,
                                                           const float *__restrict__ f, float *__restrict__ table) {
  __shared__ float s_c[kCnxConst];
  pdl_wait();
  cnx_fold(W8, b8, f, s_c);
  for (int64_t e = blockIdx.x * (int64_t)kCnxThreads + threadIdx.x; e < n; e += (int64_t)gridDim.x * kCnxThreads) {
    float x[kCnxIn];
    cnx_row(cnx, e, x);
    float t[kH];
#pragma unroll
    for (int h = 0; h < kH; ++h) {
      float s = s_c[kCnxIn * kH + h];
#pragma unroll
      for (int k = 0; k < kCnxIn; ++k) s += x[k] * s_c[k * kH + h];
      t[h] = s;
    }
    st4(table + e * 4, make_float4(t[0], t[1], t[2], t[3]));
  }
}

// Backward: per-CTA records of dcoef = cnx^T d_table and dbias = column sums of d_table, summed in a fixed order by
// the last CTA (cta_finish), which then folds them through f_e and W8 / b8.
__global__ void __launch_bounds__(kCnxThreads) k_cnx_table_bwd(const float *__restrict__ cnx,
                                                               const float *__restrict__ d_table, int64_t n,
                                                               const float *__restrict__ W8, const float *__restrict__ b8,
                                                               const float *__restrict__ f, float *__restrict__ dW8,
                                                               float *__restrict__ db8, float *__restrict__ df,
                                                               float *scratch) {
  __shared__ float s_part[kCnxThreads / 32][kCnxConst];
  __shared__ float s_rec[kCnxConst], s_fin[kCnxConst];
  pdl_wait();
  float acc[kCnxConst];
#pragma unroll
  for (int o = 0; o < kCnxConst; ++o) acc[o] = 0.f;
  for (int64_t e = blockIdx.x * (int64_t)kCnxThreads + threadIdx.x; e < n; e += (int64_t)gridDim.x * kCnxThreads) {
    float x[kCnxIn];
    cnx_row(cnx, e, x);
    const float4 d = ldg4(d_table + e * 4);
    const float dv[kH] = {d.x, d.y, d.z, d.w};
#pragma unroll
    for (int h = 0; h < kH; ++h) {
#pragma unroll
      for (int k = 0; k < kCnxIn; ++k) acc[k * kH + h] += x[k] * dv[h];
      acc[kCnxIn * kH + h] += dv[h];
    }
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int o = 0; o < kCnxConst; ++o) {
    const float v = warp_sum(acc[o]);
    if (lane == 0) s_part[warp][o] = v;
  }
  __syncthreads();
  if (threadIdx.x < kCnxConst) {
    float s = 0.f;
    for (int w = 0; w < kCnxThreads / 32; ++w) s += s_part[w][threadIdx.x];
    s_rec[threadIdx.x] = s;
  }
  __syncthreads();
  if (!cta_finish<kCnxConst>(s_rec, s_fin, scratch)) return;
  // dW8[j,k] = sum_h dcoef[k,h] f_e[h,j];  db8[j] = sum_h dbias[h] f_e[h,j];
  // df[h, 32 + j] = sum_k W8[j,k] dcoef[k,h] + b8[j] dbias[h]
  for (int j = threadIdx.x; j < kD; j += kCnxThreads) {
    float fe[kH];
#pragma unroll
    for (int h = 0; h < kH; ++h) fe[h] = __ldg(f + h * kFStride + kFEdge + j);
    float w[kCnxIn];
#pragma unroll
    for (int k = 0; k < kCnxIn; ++k) {
      w[k] = __ldg(W8 + j * kCnxIn + k);
      float s = 0.f;
#pragma unroll
      for (int h = 0; h < kH; ++h) s += s_fin[k * kH + h] * fe[h];
      dW8[j * kCnxIn + k] = s;
    }
    float sb = 0.f;
#pragma unroll
    for (int h = 0; h < kH; ++h) sb += s_fin[kCnxIn * kH + h] * fe[h];
    db8[j] = sb;
    const float bj = __ldg(b8 + j);
#pragma unroll
    for (int h = 0; h < kH; ++h) {
      float s = bj * s_fin[kCnxIn * kH + h];
#pragma unroll
      for (int k = 0; k < kCnxIn; ++k) s += w[k] * s_fin[k * kH + h];
      df[h * kFStride + kFEdge + j] = s;
    }
  }
}

int cnx_grid(int64_t n) {
  const int64_t blocks = (n + kCnxThreads - 1) / kCnxThreads;
  return (int)(blocks < 1 ? 1 : (blocks > kNumSMs ? kNumSMs : blocks));
}

}  // namespace

int fnb_cnx_table_fwd(const float *cnx, int64_t n, const float *W8, const float *b8, const float *f, float *table,
                      cudaStream_t stream) {
  if (n < 0) return FNB_ERR_SIZE;
  if (n == 0) return 0;
  if (!cnx || !W8 || !b8 || !f || !table) return FNB_ERR_NULL;
  if (!fnb_aligned16(cnx) || !fnb_aligned16(table)) return FNB_ERR_ALIGN;
  if (cudaError_t le = fnb_launch(k_cnx_table, dim3(cnx_grid(n)), dim3(kCnxThreads), 0, stream, cnx, n, W8, b8, f, table))
    return (int)le;
  FNB_CHECK_LAUNCH();
  return 0;
}

int fnb_cnx_table_bwd(const float *cnx, const float *d_table, int64_t n, const float *W8, const float *b8,
                      const float *f, float *dW8, float *db8, float *df, void *scratch, cudaStream_t stream) {
  if (n < 0) return FNB_ERR_SIZE;
  if (!W8 || !b8 || !f || !dW8 || !db8 || !df || !scratch || (n > 0 && (!cnx || !d_table))) return FNB_ERR_NULL;
  if (!fnb_aligned16(cnx) || !fnb_aligned16(d_table)) return FNB_ERR_ALIGN;
  // (n == 0: one CTA writes zero gradients)
  if (cudaError_t le = fnb_launch(k_cnx_table_bwd, dim3(cnx_grid(n)), dim3(kCnxThreads), 0, stream, cnx, d_table, n, W8,
                                  b8, f, dW8, db8, df, reinterpret_cast<float *>(scratch)))
    return (int)le;
  FNB_CHECK_LAUNCH();
  return 0;
}

int fnb_mlp_check(const fnb_mlp_layer *L, int n, int64_t G, int in0, int backward) {
  if (!L) return FNB_ERR_NULL;
  if (n < 1 || n > FNB_MLP_MAX_LAYERS || G < 1) return FNB_ERR_SIZE;
  for (int l = 0; l < n; ++l) {
    const fnb_mlp_layer &y = L[l];
    if (!y.W || !y.b) return FNB_ERR_NULL;
    if (backward && (!y.dW != !y.db)) return FNB_ERR_NULL;          // both NULL: a frozen layer
    if (y.in_dim < 1 || y.out_dim < 1 || y.in_dim != (l == 0 ? in0 : L[l - 1].out_dim)) return FNB_ERR_SIZE;
    if ((int64_t)y.in_dim * y.out_dim + y.out_dim >= INT32_MAX || G * y.in_dim >= INT32_MAX || G * y.out_dim >= INT32_MAX)
      return FNB_ERR_SIZE;
    if (!(y.p_in >= 0.f && y.p_in < 1.f) || !(y.p_out >= 0.f && y.p_out < 1.f)) return FNB_ERR_SIZE;
    if (y.act < FNB_ACT_NONE || y.act > FNB_ACT_LEAKYRELU) return FNB_ERR_MODE;
  }
  if (L[n - 1].act != FNB_ACT_NONE || L[n - 1].p_out != 0.f) return FNB_ERR_MODE;   // the prediction is a bare linear
  return 0;
}

// Counter blocks of the head's dropout sites, in layer order (input site, then output site), from `offset` on; a site
// exists where its p is non-zero.  Returns the number of counters.
uint64_t fnb_mlp_rng(const fnb_mlp_layer *L, int n, int64_t G, uint64_t offset, uint64_t *in_base, uint64_t *out_base) {
  uint64_t c = offset;
  for (int l = 0; l < n; ++l) {
    if (in_base) in_base[l] = c;
    if (L[l].p_in > 0.f) c += ((uint64_t)G * L[l].in_dim + 3) / 4;
    if (out_base) out_base[l] = c;
    if (L[l].p_out > 0.f) c += ((uint64_t)G * L[l].out_dim + 3) / 4;
  }
  return c - offset;
}

bool fnb_mlp_needs_dx(const fnb_mlp_layer *L, int l, bool want_dx0) {
  for (int j = 0; j < l; ++j)
    if (L[j].dW) return true;
  return want_dx0;
}

size_t fnb_mlp_dw_record_floats(const fnb_mlp_layer *L, int n, int64_t G) {
  size_t most = 0;
  for (int l = 0; l < n; ++l)
    if (L[l].dW) most = std::max(most, fnb_gemm_dw_record_floats(G, L[l].out_dim, L[l].in_dim));
  return most;
}

int fnb_mlp_forward(const FnbMlpRun *r, cudaStream_t stream) {
  const fnb_mlp_layer *L = r->L;
  const fnb_mlp_layer &first = L[0];
  if (r->xd[0] != r->x0)
    RC(fnb_dropout_relu_fwd(r->x0, r->xd[0], r->G * first.in_dim, first.p_in, r->training, 0, r->seed, r->in_base[0],
                            stream));
  for (int l = 0; l < r->n; ++l) {
    GemmArgs a{};
    a.A = r->xd[l]; a.B = L[l].W; a.M = (int)r->G; a.N = L[l].out_dim; a.K = L[l].in_dim;
    a.bias = L[l].b; a.seed = r->seed; a.act = L[l].act;
    a.drop1 = fnb_drop(L[l].p_out, r->training, r->out_base[l]);
    const bool last = l == r->n - 1;
    a.drop2 = last ? fnb_drop(0.f, 0, 0) : fnb_drop(L[l + 1].p_in, r->training, r->in_base[l + 1]);
    a.u = last ? nullptr : r->u[l];
    a.C = last ? r->out : r->xd[l + 1];
    RC(fnb_gemm(GEMM_FWD, a, stream));
  }
  return 0;
}

int fnb_mlp_backward(const FnbMlpRun *r, cudaStream_t stream) {
  const fnb_mlp_layer *L = r->L;
  for (int l = r->n - 1; l >= 0; --l) {
    // weight and bias gradients: per-chunk records, then a fixed-order sum (not for a frozen layer)
    if (L[l].dW)
      RC(fnb_gemm_dw(r->dz[l], r->xd[l], r->G, L[l].out_dim, L[l].in_dim, L[l].dW, L[l].db, r->rec, stream));
    // input gradient, folded down to dz of the layer below (or the gradient of the head input): only while a trained
    // layer lies below, or the caller wants the head input's gradient
    if (!fnb_mlp_needs_dx(L, l, r->dx0 != nullptr)) break;
    GemmArgs d{};
    d.A = r->dz[l]; d.B = L[l].W; d.M = (int)r->G; d.N = L[l].in_dim; d.K = L[l].out_dim; d.seed = r->seed;
    d.drop1 = fnb_drop(L[l].p_in, r->training, r->in_base[l]);
    if (l > 0) {
      d.u = r->u[l - 1]; d.act = L[l - 1].act;
      d.drop2 = fnb_drop(L[l - 1].p_out, r->training, r->out_base[l - 1]);
      d.C = r->dz[l - 1];
    } else {
      d.drop2 = fnb_drop(0.f, 0, 0);
      d.C = r->dx0;
    }
    RC(fnb_gemm(GEMM_DX, d, stream));
  }
  return 0;
}

int fnb_bce_masked_loss(const float *logits, const float *labels, int64_t n, float *loss, float *grad,
                        cudaStream_t stream) {
  if (!logits || !labels || !loss) return FNB_ERR_NULL;
  if (n < 1) return FNB_ERR_SIZE;
  if (cudaError_t le = fnb_launch(k_bce_masked, dim3(1), dim3(kBceThreads), 0, stream, logits, labels, n, loss, grad))
    return (int)le;
  FNB_CHECK_LAUNCH();
  return 0;
}
