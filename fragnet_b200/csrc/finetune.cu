// The finetuning head (FTHead1-4 of FragNetFineTune, fragnet/model/gat/gat2.py:569-751) forward and backward, and the
// masked BCE-with-logits loss of TrainerFineTune (fragnet/train/utils.py:296-303, :406-470).
//
// A head is a list of linear layers (fnb_mlp_layer), each  y = act(drop_out(drop_in(x) W^T + b)).  Every layer is one
// launch of a register-tiled FP32 FFMA GEMM (64 x 64 tile, 4 x 4 outputs per thread) whose epilogue applies the bias,
// the dropout masks and the activation; the heads stay exact FP32 in every precision mode (as k_linear_rows does for
// the energy head): rows are molecules (128 to a few thousand) and widths are whatever a hyper-parameter search picks,
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
#include <cmath>

#include "common.cuh"

#define RC_INLINE(expr)      \
  do {                       \
    const int rc__ = (expr); \
    if (rc__) return rc__;   \
  } while (0)

namespace {

constexpr int BM = 64, BN = 64, BK = 16, kThreads = 256;
constexpr int SA = BM + 4;          // shared-memory row stride (floats): float4 aligned
constexpr int kDwTargetCtas = 2 * kNumSMs;

enum { MODE_FWD = 0, MODE_DX = 1, MODE_DW = 2 };

struct Drop {                       // one dropout site: element i of a [rows, width] tensor draws from base + i / 4
  float p, scale;
  uint64_t base;
  int on;
};

__device__ __forceinline__ float drop_factor(const Drop &d, uint64_t seed, int64_t i) {
  if (!d.on) return 1.f;
  const uint2 r = dropout_bits(seed, d.base + (uint64_t)(i >> 2));
  const int pos = (int)(i & 3);
  const uint32_t w = pos < 2 ? r.x : r.y;
  const uint32_t r16 = (pos & 1) ? (w >> 16) : (w & 0xffffu);
  return r16 >= dropout_threshold(d.p) ? d.scale : 0.f;
}

constexpr float kSeluAlpha = 1.6732632423543772f, kSeluScale = 1.0507009873554805f;

__device__ __forceinline__ float act_fwd(int act, float z) {
  switch (act) {
    case FNB_ACT_RELU: return fmaxf(z, 0.f);
    case FNB_ACT_CELU: return z > 0.f ? z : expm1f(z);
    case FNB_ACT_SILU: return z / (1.f + expf(-z));
    case FNB_ACT_GELU: return 0.5f * z * (1.f + erff(z * 0.70710678118654752f));
    case FNB_ACT_SELU: return kSeluScale * (z > 0.f ? z : kSeluAlpha * expm1f(z));
    case FNB_ACT_RELU6: return fminf(fmaxf(z, 0.f), 6.f);
    case FNB_ACT_LEAKYRELU: return z > 0.f ? z : 0.01f * z;
    default: return z;
  }
}

// d act / d z at z, with torch's choices at the kinks (relu: 0 at 0, relu6: 0 at 0 and 6, celu / selu: the exp branch
// at 0, leaky relu: the slope at 0).
__device__ __forceinline__ float act_grad(int act, float z) {
  switch (act) {
    case FNB_ACT_RELU: return z > 0.f ? 1.f : 0.f;
    case FNB_ACT_CELU: return z > 0.f ? 1.f : expf(z);
    case FNB_ACT_SILU: {
      const float s = 1.f / (1.f + expf(-z));
      return s * (1.f + z * (1.f - s));
    }
    case FNB_ACT_GELU:
      return 0.5f * (1.f + erff(z * 0.70710678118654752f)) + z * 0.39894228040143268f * expf(-0.5f * z * z);
    case FNB_ACT_SELU: return z > 0.f ? kSeluScale : kSeluScale * kSeluAlpha * expf(z);
    case FNB_ACT_RELU6: return (z > 0.f && z < 6.f) ? 1.f : 0.f;
    case FNB_ACT_LEAKYRELU: return z > 0.f ? 1.f : 0.01f;
    default: return 1.f;
  }
}

struct GemmArgs {
  // C[M,N] = sum_k A(m,k) B(k,n).  FWD: A = xd [M=G, K=in], B = W [N=out, K=in].  DX: A = dz [M=G, K=out],
  // B = W [K=out, N=in].  DW: A = dz [K=G, M=out], B = xd [K=G, N=in], K split into chunks of k_chunk rows (blockIdx.z).
  const float *A, *B;
  int M, N, K;
  float *C;                 // FWD / DX: [M,N]
  uint64_t seed;
  // FWD epilogue: z = acc + bias; z *= drop1; u = z; y = act(z) * drop2.  DX epilogue: v = acc * drop1 * act'(u) * drop2.
  const float *bias;
  Drop drop1, drop2;
  int act;
  float *u;                 // FWD: written (may be NULL); DX: read (NULL = no activation between the layers)
  // DW: per-chunk records [N*M dW | M db], record z at rec + z * rec_stride
  int k_chunk;
  float *rec;
  int64_t rec_stride;
};

// Loads one BK-deep slab of a 64-row operand tile into registers.  KC: the operand is K-contiguous (element (r, k) at
// p[r * ld + k]), else R-contiguous (p[k * ld + r]).  Thread t holds 4 elements; out-of-range elements are 0.
template <bool KC>
__device__ __forceinline__ void load_slab(const float *__restrict__ p, int ld, int r0, int nr, int k0, int k1,
                                          float v[4]) {
  const int t = threadIdx.x;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int kk = KC ? (t & 15) : (t >> 6) + 4 * i;
    const int r = KC ? (t >> 4) + 16 * i : (t & 63);
    const int k = k0 + kk, row = r0 + r;
    v[i] = (row < nr && k < k1) ? __ldg(KC ? p + (int64_t)row * ld + k : p + (int64_t)k * ld + row) : 0.f;
  }
}

template <bool KC>
__device__ __forceinline__ void store_slab(float (*s)[SA], const float v[4]) {
  const int t = threadIdx.x;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int kk = KC ? (t & 15) : (t >> 6) + 4 * i;
    const int r = KC ? (t >> 4) + 16 * i : (t & 63);
    s[kk][r] = v[i];
  }
}

template <int MODE>
__global__ void __launch_bounds__(kThreads) k_mlp_gemm(GemmArgs a) {
  constexpr bool A_KC = MODE != MODE_DW;      // FWD / DX: A rows are molecules, K contiguous; DW: A = dz, M contiguous
  constexpr bool B_KC = MODE == MODE_FWD;     // FWD: B = W [N, K]; DX: W [K, N]; DW: xd [K, N]
  __shared__ __align__(16) float As[BK][SA];
  __shared__ __align__(16) float Bs[BK][SA];
  pdl_wait();
  const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  int k0 = 0, k1 = a.K;
  if (MODE == MODE_DW) {
    k0 = blockIdx.z * a.k_chunk;
    k1 = min(a.K, k0 + a.k_chunk);
  }
  // leading dimensions: FWD A = xd [G, K], B = W [N, K]; DX A = dz [G, K], B = W [K, N]; DW A = dz [K, M], B = xd [K, N]
  const int lda = MODE == MODE_DW ? a.M : a.K;
  const int ldb = MODE == MODE_FWD ? a.K : a.N;
  const bool want_db = MODE == MODE_DW && blockIdx.x == 0;
  float acc[4][4] = {};
  float db_acc = 0.f;
  float ra[4], rb[4];
  load_slab<A_KC>(a.A, lda, m0, a.M, k0, k1, ra);
  load_slab<B_KC>(a.B, ldb, n0, a.N, k0, k1, rb);
  for (int kt = k0; kt < k1; kt += BK) {
    store_slab<A_KC>(As, ra);
    store_slab<B_KC>(Bs, rb);
    __syncthreads();
    if (kt + BK < k1) {                    // next slab's global loads are in flight during this slab's FMAs
      load_slab<A_KC>(a.A, lda, m0, a.M, kt + BK, k1, ra);
      load_slab<B_KC>(a.B, ldb, n0, a.N, kt + BK, k1, rb);
    }
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      const float4 av = *reinterpret_cast<const float4 *>(&As[kk][ty * 4]);
      const float4 bv = *reinterpret_cast<const float4 *>(&Bs[kk][tx * 4]);
      const float ar[4] = {av.x, av.y, av.z, av.w}, br[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(ar[i], br[j], acc[i][j]);
    }
    if (want_db && t < BM) {
#pragma unroll
      for (int kk = 0; kk < BK; ++kk) db_acc += As[kk][t];
    }
    __syncthreads();
  }
  pdl_launch_dependents();
  if constexpr (MODE == MODE_DW) {
    float *rec = a.rec + (int64_t)blockIdx.z * a.rec_stride;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int m = m0 + ty * 4 + i;
      if (m >= a.M) continue;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int n = n0 + tx * 4 + j;
        if (n < a.N) rec[(int64_t)m * a.N + n] = acc[i][j];
      }
    }
    if (want_db && t < BM && m0 + t < a.M) rec[(int64_t)a.M * a.N + m0 + t] = db_acc;
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int m = m0 + ty * 4 + i;
      if (m >= a.M) continue;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int n = n0 + tx * 4 + j;
        if (n >= a.N) continue;
        const int64_t idx = (int64_t)m * a.N + n;
        float v = acc[i][j];
        if (MODE == MODE_FWD) {
          v = (v + __ldg(a.bias + n)) * drop_factor(a.drop1, a.seed, idx);
          if (a.u) a.u[idx] = v;
          v = act_fwd(a.act, v) * drop_factor(a.drop2, a.seed, idx);
        } else {
          v *= drop_factor(a.drop1, a.seed, idx);
          if (a.u) v *= act_grad(a.act, __ldg(a.u + idx));
          v *= drop_factor(a.drop2, a.seed, idx);
        }
        a.C[idx] = v;
      }
    }
  }
}

Drop drop_of(float p, int training, uint64_t base) {
  Drop d{};
  d.on = training && p > 0.f;
  d.p = p;
  d.scale = d.on ? 1.f / (1.f - p) : 1.f;
  d.base = base;
  return d;
}

template <int MODE>
int launch_gemm(const GemmArgs &a, int splits, cudaStream_t stream) {
  const dim3 grid((a.N + BN - 1) / BN, (a.M + BM - 1) / BM, splits);
  if (cudaError_t le = fnb_launch(k_mlp_gemm<MODE>, grid, dim3(kThreads), 0, stream, a)) return (int)le;
  FNB_CHECK_LAUNCH();
  return 0;
}

// Row chunk of the weight-gradient GEMM: enough chunks to give ~2 CTAs per SM, each at least 64 rows.
int dw_chunk(int64_t G, int out, int in) {
  const int64_t tiles = (int64_t)((out + BM - 1) / BM) * ((in + BN - 1) / BN);
  int64_t splits = (kDwTargetCtas + tiles - 1) / tiles;
  const int64_t max_splits = (G + 63) / 64;
  if (splits > max_splits) splits = max_splits;
  if (splits < 1) splits = 1;
  int64_t chunk = (G + splits - 1) / splits;
  chunk = (chunk + BK - 1) / BK * BK;
  return (int)chunk;
}

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

}  // namespace

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
  for (int l = 0; l < n; ++l) {
    if (!L[l].dW) continue;
    const int chunk = dw_chunk(G, L[l].out_dim, L[l].in_dim);
    const size_t splits = (size_t)((G + chunk - 1) / chunk);
    const size_t f = splits * ((size_t)L[l].in_dim * L[l].out_dim + L[l].out_dim);
    if (f > most) most = f;
  }
  return most;
}

int fnb_mlp_forward(const FnbMlpRun *r, cudaStream_t stream) {
  const fnb_mlp_layer *L = r->L;
  const fnb_mlp_layer &first = L[0];
  if (r->xd[0] != r->x0)
    RC_INLINE(fnb_dropout_relu_fwd(r->x0, r->xd[0], r->G * first.in_dim, first.p_in, r->training, 0, r->seed, r->in_base[0],
                                   stream));
  for (int l = 0; l < r->n; ++l) {
    GemmArgs a{};
    a.A = r->xd[l]; a.B = L[l].W; a.M = (int)r->G; a.N = L[l].out_dim; a.K = L[l].in_dim;
    a.bias = L[l].b; a.seed = r->seed; a.act = L[l].act;
    a.drop1 = drop_of(L[l].p_out, r->training, r->out_base[l]);
    const bool last = l == r->n - 1;
    a.drop2 = last ? drop_of(0.f, 0, 0) : drop_of(L[l + 1].p_in, r->training, r->in_base[l + 1]);
    a.u = last ? nullptr : r->u[l];
    a.C = last ? r->out : r->xd[l + 1];
    RC_INLINE(launch_gemm<MODE_FWD>(a, 1, stream));
  }
  return 0;
}

int fnb_mlp_backward(const FnbMlpRun *r, cudaStream_t stream) {
  const fnb_mlp_layer *L = r->L;
  for (int l = r->n - 1; l >= 0; --l) {
    // weight and bias gradients: per-chunk records, then a fixed-order sum (not for a frozen layer)
    if (L[l].dW) {
      GemmArgs w{};
      w.A = r->dz[l]; w.B = r->xd[l]; w.M = L[l].out_dim; w.N = L[l].in_dim; w.K = (int)r->G;
      w.k_chunk = dw_chunk(r->G, L[l].out_dim, L[l].in_dim);
      w.rec = r->rec;
      w.rec_stride = (int64_t)L[l].in_dim * L[l].out_dim + L[l].out_dim;
      const int splits = (int)((r->G + w.k_chunk - 1) / w.k_chunk);
      RC_INLINE(launch_gemm<MODE_DW>(w, splits, stream));
      ReduceSegments segs{};
      segs.n = 2;
      segs.rec_off[0] = 0; segs.width[0] = L[l].in_dim * L[l].out_dim; segs.out[0] = L[l].dW;
      segs.row_len[0] = segs.width[0]; segs.out_stride[0] = segs.width[0];
      segs.rec_off[1] = L[l].in_dim * L[l].out_dim; segs.width[1] = L[l].out_dim; segs.out[1] = L[l].db;
      segs.row_len[1] = L[l].out_dim; segs.out_stride[1] = L[l].out_dim;
      RC_INLINE(fnb_launch_reduce_segments(r->rec, splits, (int)w.rec_stride, segs, stream));
    }
    // input gradient, folded down to dz of the layer below (or the gradient of the head input): only while a trained
    // layer lies below, or the caller wants the head input's gradient
    if (!fnb_mlp_needs_dx(L, l, r->dx0 != nullptr)) break;
    GemmArgs d{};
    d.A = r->dz[l]; d.B = L[l].W; d.M = (int)r->G; d.N = L[l].in_dim; d.K = L[l].out_dim; d.seed = r->seed;
    d.drop1 = drop_of(L[l].p_in, r->training, r->in_base[l]);
    if (l > 0) {
      d.u = r->u[l - 1]; d.act = L[l - 1].act;
      d.drop2 = drop_of(L[l - 1].p_out, r->training, r->out_base[l - 1]);
      d.C = r->dz[l - 1];
    } else {
      d.drop2 = drop_of(0.f, 0, 0);
      d.C = r->dx0;
    }
    RC_INLINE(launch_gemm<MODE_DX>(d, 1, stream));
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
