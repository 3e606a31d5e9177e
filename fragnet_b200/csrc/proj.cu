// Node/edge linear projections of the GAT2 blocks, fp32 (strict-parity path).
//
// Reference: nn.Linear projection_a / projection_b / projection_fb (fragnet/model/gat/gat2.py:142,
// 189, 247) followed by .view(N, H, d) and, per edge, two 32-wide dot products of the gathered rows
// with the head vector (gat2.py:148-150, 204-208, 252-254).  Here the projection kernel also emits the
// per-NODE halves of those dot products (S[n,0:4] target half, S[n,4:8] source half) from its
// epilogue while the output tile is still in registers, so the attention kernels never re-read
// 128-wide rows to form a logit (SURVEY.md App. A.5).
//
// This file holds every FP32 SIMT kernel of the projections, used for exact (<=1e-5) parity with the reference
// (FFMA-bound, not HBM-bound -- see DESIGN.md "projection" for the tensor-core kernels): the FFMA GEMM k_mlp_gemm, which
// also runs the finetuning head (finetune.cu), the row-sparse kernel for raw input features, k_linear_rows for few
// rows, and k_node_scalars.
#include "common.cuh"

namespace {

// ---- k_mlp_gemm: the register-tiled FP32 FFMA GEMM (GemmArgs, common.cuh) ---------------------------------------------
// 64 x 64 output tile per CTA, 4 x 4 outputs per thread, K in slabs of 16 whose global loads are in flight (in
// registers) while the previous slab's FMAs run.  Rows are on gridDim.x (no limit but INT32_MAX), columns on gridDim.y,
// weight-gradient row chunks on gridDim.z.
constexpr int BM = 64, BN = 64, BK = 16, kThreads = 256;
constexpr int SA = BM + 4;          // shared-memory row stride (floats): float4 aligned
constexpr int kDwTargetCtas = 2 * kNumSMs;

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
  constexpr bool A_KC = MODE != GEMM_DW;      // FWD / DX: A rows are molecules, K contiguous; DW: A = dz, M contiguous
  constexpr bool B_KC = MODE == GEMM_FWD;     // FWD: B = W [N, K]; DX: W [K, N]; DW: xd [K, N]
  __shared__ __align__(16) float As[BK][SA];
  __shared__ __align__(16) float Bs[BK][SA];
  pdl_wait();
  const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
  const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
  int k0 = 0, k1 = a.K;
  if (MODE == GEMM_DW) {
    k0 = blockIdx.z * a.k_chunk;
    k1 = min(a.K, k0 + a.k_chunk);
  }
  // leading dimensions: FWD A = xd [G, K], B = W [N, K]; DX A = dz [G, K], B = W [K, N]; DW A = dz [K, M], B = xd [K, N]
  const int lda = MODE == GEMM_DW ? a.M : a.K;
  const int ldb = MODE == GEMM_FWD ? a.K : a.N;
  const bool want_db = MODE == GEMM_DW && blockIdx.y == 0;
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
  if constexpr (MODE == GEMM_DW) {
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
        if (MODE == GEMM_FWD) {
          if (a.bias) v += __ldg(a.bias + n);
          v *= drop_factor(a.drop1, a.seed, idx);
          if (a.u) a.u[idx] = v;
          v = act_fwd(a.act, v) * drop_factor(a.drop2, a.seed, idx);
          acc[i][j] = v;
        } else {
          v *= drop_factor(a.drop1, a.seed, idx);
          if (a.u) v *= act_grad(a.act, __ldg(a.u + idx));
          v *= drop_factor(a.drop2, a.seed, idx);
        }
        a.C[idx] = v;
      }
    }
    if (MODE == GEMM_FWD && a.S) {
      // the thread's 4 columns lie in head c / 32, whose 32 columns the 8 threads tx & ~7 .. tx | 7 of this row group own
      const int c = n0 + tx * 4, head = c >> 5;
      const float *pt = a.alpha + head * a.alpha_stride + a.off_t + (c & 31);
      const float *ps = a.alpha + head * a.alpha_stride + a.off_s + (c & 31);
      const float4 at = make_float4(__ldg(pt), __ldg(pt + 1), __ldg(pt + 2), __ldg(pt + 3));
      const float4 as = make_float4(__ldg(ps), __ldg(ps + 1), __ldg(ps + 2), __ldg(ps + 3));
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float4 v = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
        const float st = head_sum(dot4(v, at)), ss = head_sum(dot4(v, as));
        const int m = m0 + ty * 4 + i;
        if ((tx & 7) == 0 && m < a.M) {
          a.S[(int64_t)m * 8 + head] = st;
          a.S[(int64_t)m * 8 + 4 + head] = ss;
        }
      }
    }
  }
}

// Row chunk of the weight-gradient GEMM: enough chunks to give ~2 CTAs per SM, each at least 64 rows.  With out = 128
// (two row tiles) that is at most kNumSMs chunks, which is what kScratchFloats holds for the projections.
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

template <int MODE>
int launch_gemm(const GemmArgs &a, int splits, cudaStream_t stream) {
  const dim3 grid((a.M + BM - 1) / BM, (a.N + BN - 1) / BN, splits);
  if (grid.y > 65535u || a.M > INT32_MAX - BM) return FNB_ERR_SIZE;
  if (cudaError_t le = fnb_launch(k_mlp_gemm<MODE>, grid, dim3(kThreads), 0, stream, a)) return (int)le;
  FNB_CHECK_LAUNCH();
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Row-sparse projections for the raw input features of layer 0 (K = 167 / 17 / 6: one-hot groups, a dozen non-zeros
// per row; features.py:43-139).  K is neither a multiple of 4 (no TMA, no tensor-core path) nor worth a dense FFMA
// sweep: a warp reads 32 feature values at a time, ballots the non-zeros and accumulates only those weight columns.
// Lane L owns output columns L, L+32, L+64, L+96 (one per head), so the weights -- staged as W[o][K+1] in shared
// memory, odd row stride -- are read conflict-free.  Skipping zeros is exact: fma(0, w, acc) == acc, so the result
// equals the dense k-ascending FFMA chain bit for bit.
constexpr int kSparseRowsPerIter = 4;

__global__ void __launch_bounds__(256) k_proj_rowsparse_fwd(const float *__restrict__ x, const float *__restrict__ W,
                                                             const float *__restrict__ bias, int64_t n_rows, int K,
                                                             const float *__restrict__ alpha, int alpha_stride,
                                                             int off_t, int off_s, float *__restrict__ h,
                                                             float *__restrict__ S) {
  pdl_wait();
  extern __shared__ float s_W[];  // [128][K+1]
  const int ld = K + 1;
  for (int idx = threadIdx.x; idx < 128 * K; idx += blockDim.x) s_W[(idx / K) * ld + idx % K] = __ldg(W + idx);
  __syncthreads();
  const int lane = threadIdx.x & 31;
  float b4[4], at[4], as[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    b4[i] = bias ? __ldg(bias + lane + 32 * i) : 0.f;
    at[i] = S ? __ldg(alpha + i * alpha_stride + off_t + lane) : 0.f;   // column lane + 32 i belongs to head i
    as[i] = S ? __ldg(alpha + i * alpha_stride + off_s + lane) : 0.f;
  }
  const int64_t w0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int n_chunks = (K + 31) >> 5;
  for (int64_t r0 = w0 * kSparseRowsPerIter; r0 < n_rows; r0 += nw * kSparseRowsPerIter) {
    float acc[kSparseRowsPerIter][4];
#pragma unroll
    for (int r = 0; r < kSparseRowsPerIter; ++r)
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[r][i] = b4[i];
    for (int c = 0; c < n_chunks; ++c) {
      const int k = c * 32 + lane;
      float xv[kSparseRowsPerIter];
#pragma unroll
      for (int r = 0; r < kSparseRowsPerIter; ++r)   // all loads of the iteration are in flight together
        xv[r] = (k < K && r0 + r < n_rows) ? __ldg(x + (r0 + r) * K + k) : 0.f;
#pragma unroll
      for (int r = 0; r < kSparseRowsPerIter; ++r) {
        unsigned m = __ballot_sync(kFull, xv[r] != 0.f);
        while (m) {
          const int bit = __ffs(m) - 1;
          m &= m - 1;
          const float xk = __shfl_sync(kFull, xv[r], bit);
          const float *w = s_W + lane * ld + c * 32 + bit;
#pragma unroll
          for (int i = 0; i < 4; ++i) acc[r][i] = fmaf(xk, w[32 * i * ld], acc[r][i]);
        }
      }
    }
#pragma unroll
    for (int r = 0; r < kSparseRowsPerIter; ++r) {
      const int64_t row = r0 + r;
      if (row >= n_rows) break;
#pragma unroll
      for (int i = 0; i < 4; ++i) h[row * kD + lane + 32 * i] = acc[r][i];
      if (S) {
        const float st = warp_sum4(acc[r][0] * at[0], acc[r][1] * at[1], acc[r][2] * at[2], acc[r][3] * at[3]);
        const float ss = warp_sum4(acc[r][0] * as[0], acc[r][1] * as[1], acc[r][2] * as[2], acc[r][3] * as[3]);
        if ((lane & 7) == 0) {
          S[row * 8 + (lane >> 3)] = st;
          S[row * 8 + 4 + (lane >> 3)] = ss;
        }
      }
    }
  }
}

inline bool rowsparse_shape(int K) { return (K & 3) != 0 || K < 32; }

// S for un-projected features: one warp per row.
__global__ void __launch_bounds__(256) k_node_scalars(const float *__restrict__ h, int64_t n_rows,
                                                      const float *__restrict__ alpha, int alpha_stride, int off_t,
                                                      int off_s, float *__restrict__ S) {
  const int lane = threadIdx.x & 31, head = lane >> 3;
  const float4 at = ldg4(alpha + (int64_t)head * alpha_stride + off_t + (lane & 7) * 4);
  const float4 as = ldg4(alpha + (int64_t)head * alpha_stride + off_s + (lane & 7) * 4);
  const int64_t w0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t wstride = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t n = w0; n < n_rows; n += wstride) {
    const float4 v = ldg4(h + n * kD + lane * 4);
    const float st = head_sum(dot4(v, at)), ss = head_sum(dot4(v, as));
    if ((lane & 7) == 0) {
      S[n * 8 + head] = st;
      S[n * 8 + 4 + head] = ss;
    }
  }
}

// Small-M linear layer: C[M, Nc] = A[M, Kd] @ op(B) (+ bias) for a few thousand rows at most (the energy head:
// one row per molecule, [G, 256] x [256 -> 128] forward and [G, 128] x [128 -> 256] input gradient).  The GEMM tiles 64
// rows per CTA: 16 CTAs at G = 1024 and 45 us of pure latency on the critical path between the encoder's forward and
// backward (gpurun_out/r4j_device_profile.log).  Here a CTA owns LR_ROWS = 8 rows (128 CTAs at G = 1024), a thread owns
// output columns t, t + 128, ... for all 8 rows: the A rows sit in shared memory (broadcast reads), every thread
// streams its own part of B once.  Exact FP32 (FFMA, k ascending).
constexpr int LR_ROWS = 8, LR_THREADS = 128, LR_MAXK = 256, LR_MAXC = 2;   // Nc <= LR_MAXC * LR_THREADS

template <bool TRANS_B>
__global__ void __launch_bounds__(LR_THREADS) k_linear_rows(GemmArgs g) {
  pdl_wait();
  __shared__ __align__(16) float sA[LR_ROWS][LR_MAXK];
  const int Kd = g.K, Nc = g.N, ldb = TRANS_B ? Kd : Nc;   // A [M, Kd], C [M, Nc]
  const int tid = threadIdx.x;
  const int64_t m0 = (int64_t)blockIdx.x * LR_ROWS;
  for (int i = tid; i < LR_ROWS * Kd; i += LR_THREADS) {
    const int r = i / Kd, k = i - r * Kd;
    sA[r][k] = (m0 + r < g.M) ? __ldg(g.A + (m0 + r) * Kd + k) : 0.f;
  }
  __syncthreads();
  float acc[LR_MAXC][LR_ROWS];
#pragma unroll
  for (int c = 0; c < LR_MAXC; ++c)
#pragma unroll
    for (int r = 0; r < LR_ROWS; ++r) acc[c][r] = 0.f;
  if (TRANS_B) {            // B = nn.Linear weight [Nc, Kd]: the thread reads its row(s) of B, 16 bytes at a time
#pragma unroll
    for (int c = 0; c < LR_MAXC; ++c) {
      const int n = tid + c * LR_THREADS;
      if (n >= Nc) break;
      const float *brow = g.B + (int64_t)n * ldb;
      for (int k0 = 0; k0 < Kd; k0 += 32) {        // 8 independent 16-byte loads in flight (Kd is a multiple of 32 here)
        float4 w[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) w[u] = (k0 + 4 * u < Kd) ? ldg4(brow + k0 + 4 * u) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int k = k0 + 4 * u;
          if (k >= Kd) break;
#pragma unroll
          for (int r = 0; r < LR_ROWS; ++r) {
            const float4 a = ld4(&sA[r][k]);
            acc[c][r] = fmaf(a.x, w[u].x, acc[c][r]);
            acc[c][r] = fmaf(a.y, w[u].y, acc[c][r]);
            acc[c][r] = fmaf(a.z, w[u].z, acc[c][r]);
            acc[c][r] = fmaf(a.w, w[u].w, acc[c][r]);
          }
        }
      }
    }
  } else {                  // B [Kd, Nc]: coalesced reads of B's rows
    for (int k0 = 0; k0 < Kd; k0 += 8) {             // 16 independent loads in flight per thread
      float w[8][LR_MAXC];
#pragma unroll
      for (int u = 0; u < 8; ++u)
#pragma unroll
        for (int c = 0; c < LR_MAXC; ++c) {
          const int n = tid + c * LR_THREADS;
          w[u][c] = (n < Nc && k0 + u < Kd) ? __ldg(g.B + (int64_t)(k0 + u) * ldb + n) : 0.f;
        }
#pragma unroll
      for (int u = 0; u < 8; ++u)
#pragma unroll
        for (int r = 0; r < LR_ROWS; ++r) {
          const float a = sA[r][(k0 + u) & (LR_MAXK - 1)];
#pragma unroll
          for (int c = 0; c < LR_MAXC; ++c) acc[c][r] = fmaf(a, w[u][c], acc[c][r]);
        }
    }
  }
#pragma unroll
  for (int c = 0; c < LR_MAXC; ++c) {
    const int n = tid + c * LR_THREADS;
    if (n >= Nc) break;
    const float b = g.bias ? __ldg(g.bias + n) : 0.f;
#pragma unroll
    for (int r = 0; r < LR_ROWS; ++r)
      if (m0 + r < g.M) g.C[(m0 + r) * Nc + n] = acc[c][r] + b;
  }
}

// Shapes k_linear_rows takes: few rows, K a multiple of 32 up to 256, at most 256 output columns, 16-byte aligned rows.
bool linear_rows_shape(const GemmArgs &g, bool trans_b) {
  return g.M > 0 && g.M <= 8192 && g.K <= LR_MAXK && (g.K & 31) == 0 && g.N <= LR_MAXC * LR_THREADS &&
         fnb_aligned16(g.A) && (!trans_b || fnb_aligned16(g.B));
}

template <bool TRANS_B>
int launch_linear_rows(const GemmArgs &g, cudaStream_t stream) {
  if (cudaError_t le = fnb_launch(k_linear_rows<TRANS_B>, dim3((unsigned)((g.M + LR_ROWS - 1) / LR_ROWS)), dim3(LR_THREADS), 0,
                                  stream, g))
    return (int)le;
  FNB_CHECK_LAUNCH();
  return 0;
}

// The FFMA GEMM indexes rows with int32.
inline bool gemm_rows_ok(int64_t n_rows) { return n_rows <= INT32_MAX - BM; }

}  // namespace

Drop fnb_drop(float p, int training, uint64_t base) {
  Drop d{};
  d.on = training && p > 0.f;
  d.p = p;
  d.scale = d.on ? 1.f / (1.f - p) : 1.f;
  d.base = base;
  return d;
}

int fnb_gemm(int mode, const GemmArgs &a, cudaStream_t stream) {
  if (mode == GEMM_FWD) return launch_gemm<GEMM_FWD>(a, 1, stream);
  if (mode == GEMM_DX) return launch_gemm<GEMM_DX>(a, 1, stream);
  return FNB_ERR_MODE;
}

size_t fnb_gemm_dw_record_floats(int64_t rows, int out, int in) {
  if (rows <= 0) return 0;
  const int chunk = dw_chunk(rows, out, in);
  return (size_t)((rows + chunk - 1) / chunk) * ((size_t)in * out + out);
}

int fnb_gemm_dw(const float *dz, const float *x, int64_t rows, int out, int in, float *dW, float *db, float *rec,
                cudaStream_t stream) {
  if (rows == 0) {
    if (cudaError_t e = cudaMemsetAsync(dW, 0, (size_t)out * in * sizeof(float), stream)) return (int)e;
    if (db)
      if (cudaError_t e = cudaMemsetAsync(db, 0, (size_t)out * sizeof(float), stream)) return (int)e;
    return 0;
  }
  GemmArgs w{};
  w.A = dz; w.B = x; w.M = out; w.N = in; w.K = (int)rows;
  w.k_chunk = dw_chunk(rows, out, in);
  w.rec = rec;
  w.rec_stride = (int64_t)in * out + out;
  const int splits = (int)((rows + w.k_chunk - 1) / w.k_chunk);
  if (const int rc = launch_gemm<GEMM_DW>(w, splits, stream)) return rc;
  ReduceSegments segs{};
  segs.n = db ? 2 : 1;
  segs.rec_off[0] = 0; segs.width[0] = in * out; segs.out[0] = dW; segs.row_len[0] = in * out; segs.out_stride[0] = in * out;
  segs.rec_off[1] = in * out; segs.width[1] = out; segs.out[1] = db; segs.row_len[1] = out; segs.out_stride[1] = out;
  return fnb_launch_reduce_segments(rec, splits, (int)w.rec_stride, segs, stream);
}

extern "C" int fnb_proj_fwd(const float *x, const float *W, const float *b, int64_t n_rows, int K, const float *alpha,
                            int alpha_stride, int off_t, int off_s, float *h, float *S, int precision, void *stream) {
  if (n_rows < 0 || K <= 0) return FNB_ERR_SIZE;
  if (n_rows == 0) return 0;
  if (!x || !W || !h) return FNB_ERR_NULL;
  if (S && !alpha) return FNB_ERR_NULL;
  if (!fnb_aligned16(h)) return FNB_ERR_ALIGN;
  // 3xTF32 with K > 128 (the energy head's [G, 256] readout) and few rows: the FFMA kernel is as fast as the
  // latency-bound tensor-core launch on <= 64 row tiles and exact FP32 (32 truncating accumulator additions at
  // K = 256 left that prediction at 9e-6 of the reference, against 3e-6 here)
  const bool small_wide = precision == FNB_PRECISION_TF32X3 && K > kD && n_rows <= 8192;
  if (fnb_tc_precision(precision) && !small_wide) {
    const int rc = fnb_tc_proj_launch(x, W, b, n_rows, K, S ? alpha : nullptr, alpha_stride, off_t, off_s, h, S,
                                      (cudaStream_t)stream, precision == FNB_PRECISION_TF32X3);
    if (rc != FNB_ERR_MODE) return rc;   // shapes TMA cannot address (K*4 % 16 != 0) take the SIMT kernel below
  } else if (precision != FNB_PRECISION_FP32 && !fnb_tc_precision(precision)) {
    return FNB_ERR_MODE;
  }
  if (rowsparse_shape(K) && K <= kProjBwdMaxK) {
    const size_t smem = (size_t)128 * (K + 1) * sizeof(float);
    static bool done[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (smem > 48 * 1024 && dev >= 0 && dev < 64 && !done[dev]) {
      const cudaError_t e = cudaFuncSetAttribute(k_proj_rowsparse_fwd, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 (int)((size_t)128 * (kProjBwdMaxK + 1) * sizeof(float)));
      if (e != cudaSuccess) return (int)e;
      done[dev] = true;
    }
    const int per_sm = smem > 64 * 1024 ? 2 : 4;
    int64_t blocks = (n_rows + 8 * kSparseRowsPerIter - 1) / (8 * kSparseRowsPerIter);
    if (blocks > kNumSMs * per_sm) blocks = kNumSMs * per_sm;
    k_proj_rowsparse_fwd<<<(int)blocks, 256, smem, (cudaStream_t)stream>>>(x, W, b, n_rows, K, alpha, alpha_stride, off_t,
                                                                          off_s, h, S);
    FNB_CHECK_LAUNCH();
    return 0;
  }
  if (!gemm_rows_ok(n_rows)) return FNB_ERR_SIZE;
  GemmArgs g{};
  g.A = x; g.B = W; g.M = (int)n_rows; g.N = kD; g.K = K; g.C = h; g.bias = b;
  if (!S && K > kD && linear_rows_shape(g, true)) return launch_linear_rows<true>(g, (cudaStream_t)stream);
  g.alpha = alpha; g.alpha_stride = alpha_stride; g.off_t = off_t; g.off_s = off_s; g.S = S;
  return launch_gemm<GEMM_FWD>(g, 1, (cudaStream_t)stream);
}

extern "C" int fnb_proj_bwd(const float *x, const float *W, const float *dh, int64_t n_rows, int K, float *dx,
                            float *dW, float *db, int precision, void *scratch, void *stream_) {
  return fnb_proj_bwd_impl(x, W, nullptr, dh, n_rows, K, dx, dW, db, precision, scratch, stream_);
}

// Wt_pre: optional W^T [K=128,128] already transposed by the caller (the encoder program transposes every layer's
// weights in one launch at the start of its backward pass).
// The two halves of the backward are separate so that a caller can run the weight gradient -- which nothing
// downstream waits for -- on another stream than the input gradient (which feeds the next block).
int fnb_proj_bwd_dx(const float *W, const float *Wt_pre, const float *dh, int64_t n_rows, int K, float *dx, int precision,
                    void *scratch, void *stream_) {
  if (n_rows < 0 || K <= 0 || K > kProjBwdMaxK) return FNB_ERR_SIZE;
  if (!dx || n_rows == 0) return 0;
  if (!W || !dh) return FNB_ERR_NULL;
  cudaStream_t stream = (cudaStream_t)stream_;
  if (fnb_tc_precision(precision) && K == kD) {
    // dx = dh @ W as the forward tensor-core kernel with B = W^T
    const float *Wt = Wt_pre;
    int rc = 0;
    if (!Wt) {
      if (!scratch) return FNB_ERR_NULL;
      rc = fnb_tc_transpose128_launch(W, scratch_body(scratch), stream);
      if (rc) return rc;
      Wt = scratch_body(scratch);
    }
    rc = fnb_tc_proj_launch(dh, Wt, nullptr, n_rows, kD, nullptr, 0, 0, 0, dx, nullptr, stream,
                            precision == FNB_PRECISION_TF32X3);
    if (rc != FNB_ERR_MODE) return rc;
  }
  if (!gemm_rows_ok(n_rows)) return FNB_ERR_SIZE;
  GemmArgs g{};
  g.A = dh; g.B = W; g.M = (int)n_rows; g.N = K; g.K = kD; g.C = dx;
  if (linear_rows_shape(g, false)) return launch_linear_rows<false>(g, stream);
  return launch_gemm<GEMM_DX>(g, 1, stream);
}

int fnb_proj_bwd_dw(const float *x, const float *dh, int64_t n_rows, int K, float *dW, float *db, int precision,
                    void *scratch, void *stream_) {
  if (n_rows < 0 || K <= 0 || K > kProjBwdMaxK) return FNB_ERR_SIZE;
  if (!x || !dh || !dW || !scratch) return FNB_ERR_NULL;
  cudaStream_t stream = (cudaStream_t)stream_;
  if (fnb_tc_precision(precision) && (K & 31) == 0 && K <= 256 && n_rows > 0 && !db) {
    // tensor-core path for every TMA-addressable width (K = 128: the attention projections; K = 256: the energy head)
    const int rc = fnb_tc_dw_launch(dh, x, n_rows, K, K, dW, scratch_body(scratch), stream,
                                    precision == FNB_PRECISION_TF32X3);
    if (rc != FNB_ERR_MODE) return rc;
  }
  if (!gemm_rows_ok(n_rows)) return FNB_ERR_SIZE;
  return fnb_gemm_dw(dh, x, n_rows, kD, K, dW, db, scratch_body(scratch), stream);
}

int fnb_proj_bwd_impl(const float *x, const float *W, const float *Wt_pre, const float *dh, int64_t n_rows, int K,
                      float *dx, float *dW, float *db, int precision, void *scratch, void *stream_) {
  if (n_rows < 0 || K <= 0 || K > kProjBwdMaxK) return FNB_ERR_SIZE;
  if (!x || !W || !dh || !dW || !scratch) return FNB_ERR_NULL;
  if (precision != FNB_PRECISION_FP32 && !fnb_tc_precision(precision)) return FNB_ERR_MODE;
  const int rc = fnb_proj_bwd_dx(W, Wt_pre, dh, n_rows, K, dx, precision, scratch, stream_);
  if (rc) return rc;
  return fnb_proj_bwd_dw(x, dh, n_rows, K, dW, db, precision, scratch, stream_);
}

extern "C" int fnb_node_scalars(const float *h, int64_t n_rows, const float *alpha, int alpha_stride, int off_t,
                                int off_s, float *S, void *stream) {
  if (n_rows < 0) return FNB_ERR_SIZE;
  if (n_rows == 0) return 0;
  if (!h || !alpha || !S) return FNB_ERR_NULL;
  if ((alpha_stride & 3) || (off_t & 3) || (off_s & 3) || !fnb_aligned16(alpha) || !fnb_aligned16(h))
    return FNB_ERR_ALIGN;
  int64_t blocks = (n_rows + 7) / 8;
  if (blocks > kNumSMs * 8) blocks = kNumSMs * 8;
  k_node_scalars<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(h, n_rows, alpha, alpha_stride, off_t, off_s, S);
  FNB_CHECK_LAUNCH();
  return 0;
}
