// Node/edge linear projections of the GAT2 blocks, fp32 (strict-parity path).
//
// Reference: nn.Linear projection_a / projection_b / projection_fb (fragnet/model/gat/gat2.py:142,
// 189, 247) followed by .view(N, H, d) and, per edge, two 32-wide dot products of the gathered rows
// with the head vector (gat2.py:148-150, 204-208, 252-254).  Here the projection kernel also emits the
// per-NODE halves of those dot products (S[n,0:4] target half, S[n,4:8] source half) from its
// epilogue while the output tile is still in registers, so the attention kernels never re-read
// 128-wide rows to form a logit (SURVEY.md App. A.5).
//
// This file is the fp32 SIMT implementation used for exact (<=1e-5) parity with the reference;
// FFMA-bound, not HBM-bound -- see DESIGN.md "projection" for the tensor-core plan.
#include "common.cuh"

namespace {

constexpr int BM = 64, BN = 128, BK = 32;
constexpr int kGemmThreads = 256;

struct GemmArgs {
  const float *A; int lda;      // [M, Kd]
  const float *B; int ldb;      // TRANS_B: [Nc, Kd] (nn.Linear weight), else [Kd, Nc]
  float *C; int ldc;            // [M, Nc]
  int64_t M; int Kd; int Nc;
  const float *bias;            // [Nc] or NULL
  const float *alpha; int alpha_stride, off_t, off_s;  // epilogue scalars (EPI only)
  float *S;                     // [M, 8] or NULL
};

template <bool TRANS_B, bool EPI>
__global__ void __launch_bounds__(kGemmThreads) k_gemm(GemmArgs g) {
  pdl_wait();
  __shared__ float As[BM][BK + 1];
  __shared__ __align__(16) float Bs[BK][BN];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int64_t m0 = (int64_t)blockIdx.x * BM;
  const int n0 = blockIdx.y * BN;
  float acc[4][8];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

  for (int k0 = 0; k0 < g.Kd; k0 += BK) {
#pragma unroll
    for (int i = 0; i < (BM * BK) / kGemmThreads; ++i) {
      const int idx = tid + i * kGemmThreads;
      const int k = idx & (BK - 1), r = idx / BK;
      const int64_t row = m0 + r;
      As[r][k] = (row < g.M && k0 + k < g.Kd) ? __ldg(g.A + row * g.lda + k0 + k) : 0.f;
    }
#pragma unroll
    for (int i = 0; i < (BK * BN) / kGemmThreads; ++i) {
      const int idx = tid + i * kGemmThreads;
      const int n = idx & (BN - 1), k = idx / BN;
      float v = 0.f;
      if (n0 + n < g.Nc && k0 + k < g.Kd)
        v = TRANS_B ? __ldg(g.B + (int64_t)(n0 + n) * g.ldb + k0 + k) : __ldg(g.B + (int64_t)(k0 + k) * g.ldb + n0 + n);
      Bs[k][n] = v;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      float a[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = As[ty * 4 + i][k];
      const float4 b0 = *reinterpret_cast<const float4 *>(&Bs[k][tx * 8]);
      const float4 b1 = *reinterpret_cast<const float4 *>(&Bs[k][tx * 8 + 4]);
      const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }

  const int c0 = n0 + tx * 8;
  if (g.bias) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float bj = (c0 + j < g.Nc) ? __ldg(g.bias + c0 + j) : 0.f;
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[i][j] += bj;
    }
  }
  const bool vec_ok = ((g.ldc & 3) == 0) && (c0 + 8 <= g.Nc) && fnb_is_aligned16_dev(g.C);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t row = m0 + ty * 4 + i;
    if (row >= g.M) continue;
    float *cp = g.C + row * g.ldc + c0;
    if (vec_ok) {
      st4(cp, make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]));
      st4(cp + 4, make_float4(acc[i][4], acc[i][5], acc[i][6], acc[i][7]));
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (c0 + j < g.Nc) cp[j] = acc[i][j];
    }
  }
  if (EPI && g.S) {
    // columns c0..c0+7 lie in head c0/32; the 4 threads tx&~3 .. tx|3 cover that head's 32 columns
    const int head = tx >> 2, within = (tx & 3) * 8;
    float at[8], as[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      at[j] = __ldg(g.alpha + head * g.alpha_stride + g.off_t + within + j);
      as[j] = __ldg(g.alpha + head * g.alpha_stride + g.off_s + within + j);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float st = 0.f, ss = 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        st = fmaf(acc[i][j], at[j], st);
        ss = fmaf(acc[i][j], as[j], ss);
      }
      st += __shfl_xor_sync(kFull, st, 1); st += __shfl_xor_sync(kFull, st, 2);
      ss += __shfl_xor_sync(kFull, ss, 1); ss += __shfl_xor_sync(kFull, ss, 2);
      const int64_t row = m0 + ty * 4 + i;
      if ((tx & 3) == 0 && row < g.M) {
        g.S[row * 8 + head] = st;
        g.S[row * 8 + 4 + head] = ss;
      }
    }
  }
}

// dW[o,k] = sum_n dh[n,o] x[n,k], db[o] = sum_n dh[n,o]; per-CTA partial over a contiguous row range.
constexpr int kDwRows = 32;
__global__ void __launch_bounds__(256) k_proj_dw(const float *__restrict__ dh, const float *__restrict__ x, int64_t n_rows,
                                                 int K, int64_t rows_per_block, float *__restrict__ partials,
                                                 int64_t rec_stride) {
  pdl_wait();
  __shared__ __align__(16) float dhs[kDwRows][128];
  __shared__ __align__(16) float xs[kDwRows][128];
  const int tid = threadIdx.x, tk = tid & 15, to = tid >> 4;
  const int kt0 = blockIdx.y * 128;
  const int64_t r_begin = (int64_t)blockIdx.x * rows_per_block;
  const int64_t r_end = min(n_rows, r_begin + rows_per_block);
  float acc[8][8], dbacc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    dbacc[i] = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
  }
  for (int64_t r0 = r_begin; r0 < r_end; r0 += kDwRows) {
#pragma unroll
    for (int i = 0; i < (kDwRows * 128) / 256; ++i) {
      const int idx = tid + i * 256;
      const int c = idx & 127, r = idx >> 7;
      const int64_t row = r0 + r;
      const bool in = row < r_end;
      dhs[r][c] = in ? __ldg(dh + row * 128 + c) : 0.f;
      xs[r][c] = (in && kt0 + c < K) ? __ldg(x + row * K + kt0 + c) : 0.f;
    }
    __syncthreads();
#pragma unroll 4
    for (int r = 0; r < kDwRows; ++r) {
      const float4 a0 = *reinterpret_cast<const float4 *>(&dhs[r][to * 8]);
      const float4 a1 = *reinterpret_cast<const float4 *>(&dhs[r][to * 8 + 4]);
      const float4 b0 = *reinterpret_cast<const float4 *>(&xs[r][tk * 8]);
      const float4 b1 = *reinterpret_cast<const float4 *>(&xs[r][tk * 8 + 4]);
      const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        dbacc[i] += a[i];
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
      }
    }
    __syncthreads();
  }
  float *rec = partials + (int64_t)blockIdx.x * rec_stride;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int o = to * 8 + i;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int k = kt0 + tk * 8 + j;
      if (k < K) rec[(int64_t)o * K + k] = acc[i][j];
    }
    if (tk == 0 && blockIdx.y == 0) rec[(int64_t)128 * K + o] = dbacc[i];
  }
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
// one row per molecule, [G, 256] x [256 -> 128] forward and [G, 128] x [128 -> 256] input gradient).  k_gemm tiles 64
// rows per CTA: 16 CTAs at G = 1024 and 45 us of pure latency on the critical path between the encoder's forward and
// backward (gpurun_out/r4j_device_profile.log).  Here a CTA owns LR_ROWS = 8 rows (128 CTAs at G = 1024), a thread owns
// output columns t, t + 128, ... for all 8 rows: the A rows sit in shared memory (broadcast reads), every thread
// streams its own part of B once.  Exact FP32 (FFMA, k ascending).
constexpr int LR_ROWS = 8, LR_THREADS = 128, LR_MAXK = 256, LR_MAXC = 2;   // Nc <= LR_MAXC * LR_THREADS

template <bool TRANS_B>
__global__ void __launch_bounds__(LR_THREADS) k_linear_rows(GemmArgs g) {
  pdl_wait();
  __shared__ __align__(16) float sA[LR_ROWS][LR_MAXK];
  const int tid = threadIdx.x;
  const int64_t m0 = (int64_t)blockIdx.x * LR_ROWS;
  for (int i = tid; i < LR_ROWS * g.Kd; i += LR_THREADS) {
    const int r = i / g.Kd, k = i - r * g.Kd;
    sA[r][k] = (m0 + r < g.M) ? __ldg(g.A + (m0 + r) * g.lda + k) : 0.f;
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
      if (n >= g.Nc) break;
      const float *brow = g.B + (int64_t)n * g.ldb;
      for (int k0 = 0; k0 < g.Kd; k0 += 32) {        // 8 independent 16-byte loads in flight (Kd is a multiple of 32 here)
        float4 w[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) w[u] = (k0 + 4 * u < g.Kd) ? ldg4(brow + k0 + 4 * u) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int k = k0 + 4 * u;
          if (k >= g.Kd) break;
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
    for (int k0 = 0; k0 < g.Kd; k0 += 8) {             // 16 independent loads in flight per thread
      float w[8][LR_MAXC];
#pragma unroll
      for (int u = 0; u < 8; ++u)
#pragma unroll
        for (int c = 0; c < LR_MAXC; ++c) {
          const int n = tid + c * LR_THREADS;
          w[u][c] = (n < g.Nc && k0 + u < g.Kd) ? __ldg(g.B + (int64_t)(k0 + u) * g.ldb + n) : 0.f;
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
    if (n >= g.Nc) break;
    const float b = g.bias ? __ldg(g.bias + n) : 0.f;
#pragma unroll
    for (int r = 0; r < LR_ROWS; ++r)
      if (m0 + r < g.M) g.C[(m0 + r) * g.ldc + n] = acc[c][r] + b;
  }
}

// Shapes k_linear_rows takes: few rows, K a multiple of 32 up to 256, at most 256 output columns, 16-byte aligned rows.
bool linear_rows_shape(int64_t M, int Kd, int Nc, const float *A, int lda, const float *B, int ldb, bool trans_b) {
  return M > 0 && M <= 8192 && Kd <= LR_MAXK && (Kd & 31) == 0 && Nc <= LR_MAXC * LR_THREADS && fnb_aligned16(A) &&
         (lda & 3) == 0 && (!trans_b || (fnb_aligned16(B) && (ldb & 3) == 0));
}

}  // namespace

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
  GemmArgs g;
  g.A = x; g.lda = K; g.B = W; g.ldb = K; g.C = h; g.ldc = kD; g.M = n_rows; g.Kd = K; g.Nc = kD; g.bias = b;
  g.alpha = alpha; g.alpha_stride = alpha_stride; g.off_t = off_t; g.off_s = off_s; g.S = S;
  if (!S && K > kD && linear_rows_shape(n_rows, K, kD, x, K, W, K, true)) {
    if (cudaError_t le = fnb_launch(k_linear_rows<true>, dim3((unsigned)((n_rows + LR_ROWS - 1) / LR_ROWS)), dim3(LR_THREADS), 0,
                                    (cudaStream_t)stream, g))
      return (int)le;
    FNB_CHECK_LAUNCH();
    return 0;
  }
  dim3 grid((unsigned)((n_rows + BM - 1) / BM), 1);
  if (cudaError_t le = fnb_launch(k_gemm<true, true>, grid, dim3(kGemmThreads), 0, (cudaStream_t)stream, g)) return (int)le;
  FNB_CHECK_LAUNCH();
  return 0;
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
  GemmArgs g;
  g.A = dh; g.lda = kD; g.B = W; g.ldb = K; g.C = dx; g.ldc = K; g.M = n_rows; g.Kd = kD; g.Nc = K; g.bias = nullptr;
  g.alpha = nullptr; g.alpha_stride = 0; g.off_t = 0; g.off_s = 0; g.S = nullptr;
  if (linear_rows_shape(n_rows, kD, K, dh, kD, W, K, false)) {
    if (cudaError_t le = fnb_launch(k_linear_rows<false>, dim3((unsigned)((n_rows + LR_ROWS - 1) / LR_ROWS)), dim3(LR_THREADS), 0,
                                    stream, g))
      return (int)le;
    FNB_CHECK_LAUNCH();
    return 0;
  }
  dim3 grid((unsigned)((n_rows + BM - 1) / BM), (unsigned)((K + BN - 1) / BN));
  if (cudaError_t le = fnb_launch(k_gemm<false, false>, grid, dim3(kGemmThreads), 0, stream, g)) return (int)le;
  FNB_CHECK_LAUNCH();
  return 0;
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
  int64_t nb = (n_rows + 255) / 256;
  if (nb > kNumSMs) nb = kNumSMs;
  if (nb < 1) nb = 1;
  int64_t rows_per_block = (n_rows + nb - 1) / nb;
  rows_per_block = ((rows_per_block + kDwRows - 1) / kDwRows) * kDwRows;
  if (rows_per_block < kDwRows) rows_per_block = kDwRows;
  const int64_t rec_stride = (int64_t)128 * K + 128;
  dim3 grid((unsigned)nb, (unsigned)((K + 127) / 128));
  if (cudaError_t le = fnb_launch(k_proj_dw, grid, dim3(256), 0, stream, dh, x, n_rows, K, rows_per_block, scratch_body(scratch),
                                  rec_stride))
    return (int)le;
  FNB_CHECK_LAUNCH();
  ReduceSegments segs{};
  segs.n = db ? 2 : 1;
  segs.rec_off[0] = 0;       segs.width[0] = 128 * K; segs.out[0] = dW; segs.row_len[0] = 128 * K; segs.out_stride[0] = 128 * K;
  segs.rec_off[1] = 128 * K; segs.width[1] = 128;     segs.out[1] = db; segs.row_len[1] = 128;     segs.out_stride[1] = 128;
  return fnb_launch_reduce_segments(scratch_body(scratch), (int)nb, (int)rec_stride, segs, stream);
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
