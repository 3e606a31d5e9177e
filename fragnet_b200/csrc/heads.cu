// Pretraining heads and loss as library programs: one call for the four heads' forward, one for their backward,
// one for the loss (value + gradients).
//
// Reference: PretrainTask.forward (fragnet/model/gat/pretrain_heads.py:64-102)
//   bond length : cat(x_atoms[ei0], x_atoms[ei1], edge_feat) [Ea,384] -> Linear(384,128) -> (ReLU, Linear) x3 (128-64-32-1)
//   bond angle  : x_atoms   [Na,128] -> Linear(128,64) ReLU Linear(64,32) ReLU Linear(32,1)
//   dihedral    : edge_feat [Ea,128] -> same stack
//   energy      : cat(scatter_add(x_atoms, batch), scatter_add(x_frags, frag_batch)) [G,256] -> 256-128-64-1
// and the training loss of Trainer.train (fragnet/train/pretrain/pretrain_utils.py:22-26).
// Upstream this is ~45 eager ops forward and ~90 kernels backward; the step was host-bound on them
// (profiles/r1n_device_profile.log: ~700 us of library kernels, ~2 ms of host time per step at batch 1024).
//
// Decomposition.  Every head is "wide first layer + narrow tail":
//   * the first layers of the per-atom / per-bond heads are dense [N,128]x[128,64] contractions over tens of
//     thousands of rows: they run on the projection kernels of this library (tcgen05 TF32 or FP32 FFMA, tc_gemm.cu /
//     proj.cu) with the 64-row weights zero-padded to 128 rows, so forward, dX and dW reuse three tested kernels;
//   * the 384-wide bond-length reduce layer never materialises the [Ea,384] concatenation: Linear(cat(a,b,e)) =
//     a W_a^T + b W_b^T + e W_e^T + bias, i.e. two [Na,128] and one [Ea,128] projections followed by a gather-add;
//   * their tails (64-32-1 per row, ~2 kFMA) are register-tiled FP32 kernels out of shared memory; the backward tail
//     recomputes the hidden layer, and reduces the parameter gradients of the tail (dW1 [MID,IN], db1, dW2, db2, db0)
//     over the rows of its tile into per-CTA records;
//   * the energy head (~1e3 molecules) is one kernel, k_energy_head, in the forward and in the backward program:
//     readout, first layer and tail (128-64-1), and in the backward the tail's gradients, the input gradient and the
//     fragments' readout backward; exact FP32 in every precision mode.  Only the weight gradient of its first layer
//     ([128,256], summed over the molecules) runs on the projection kernels.
// Parameter-gradient sums are fixed-order two-stage reductions: run-to-run deterministic, no atomics.

#include "common.cuh"

namespace {

constexpr int kPadMat = kD * kD;

// ---- forward / saved workspace ------------------------------------------------------------------------------------
struct FwdBufs {
  // saved for backward
  float *h0_ba, *h0_da;          // [Na,128], [Ea,128] first-layer pre-activations (columns 64.. are zero)
  float *readout;                // [G,256] (read by the weight gradient of the energy head's first layer)
  float *W0pad_ba, *W0pad_da;    // [128,128] rows 64.. zero
  float *W0padT_ba, *W0padT_da;  // transposes (B operand of the dX GEMM)
  // transient (bond-length head and padded operands)
  float *b0pad_ba, *b0pad_da, *b0pad_bl, *W0pad_bl, *Wr_a, *Wr_b, *Wr_e;
  float *U, *V, *T, *h0_bl;
};

size_t fwd_layout(int64_t Na, int64_t Ea, int64_t G, char *base, FwdBufs *out) {
  Arena a{base, 0};
  FwdBufs b{};
  b.h0_ba = a.take<float>(Na * kD);
  b.h0_da = a.take<float>(Ea * kD);
  b.readout = a.take<float>(G * 2 * kD);
  b.W0pad_ba = a.take<float>(kPadMat); b.W0pad_da = a.take<float>(kPadMat);
  b.W0padT_ba = a.take<float>(kPadMat); b.W0padT_da = a.take<float>(kPadMat);
  b.b0pad_ba = a.take<float>(kD); b.b0pad_da = a.take<float>(kD); b.b0pad_bl = a.take<float>(kD);
  b.W0pad_bl = a.take<float>(kPadMat);
  b.Wr_a = a.take<float>(kPadMat); b.Wr_b = a.take<float>(kPadMat); b.Wr_e = a.take<float>(kPadMat);
  b.U = a.take<float>(Na * kD); b.V = a.take<float>(Na * kD);
  b.T = a.take<float>(Ea * kD); b.h0_bl = a.take<float>(Ea * kD);
  if (out) *out = b;
  return a.total();
}

// ---- backward workspace -----------------------------------------------------------------------------------------------
// Tail kernels run 3 CTAs of 128 threads per SM (444 slots); a tile is 128 rows.  At 148 CTAs per head the 422 tiles of
// the dihedral head were 3 rounds on some CTAs while a third of the slots idled; 222 per head make it 2 rounds
// (k_mlp_tail_bwd2: 54 -> 40 us at batch 1 024).
constexpr int kTailCtasMax = kNumSMs * 3 / 2;
__host__ __device__ constexpr int rec_floats(int IN, int MID) { return (MID * IN + MID + MID + 1 + IN + 3) & ~3; }
constexpr int kRecSmall = rec_floats(64, 32);    // 2180
constexpr int kRecWide = rec_floats(128, 64);    // 8452

struct BwdBufs {
  float *dh0_ba, *dh0_da, *dh0_fc;   // [Na,128] [Ea,128] [G,128] gradients of the first-layer pre-activations
  float *dx_ba;                      // [Na,128] gradient of x_atoms through the bond-angle head
  float *d_readout;                  // [G,256]
  float *dWpad_ba, *dWpad_da;        // [128,128] (rows 64.. are zero)
  float *rec_ba, *rec_da, *rec_fc;   // per-CTA records of the tail gradients
  float *scratch2;                   // scratch of the energy-head chain (auxiliary stream)
  float *scratch3;                   // scratch of the weight-gradient stream
  float *loss_parts;                 // [4] per-head shares of the fused loss
};

size_t bwd_layout(int64_t Na, int64_t Ea, int64_t G, char *base, BwdBufs *out) {
  Arena a{base, 0};
  BwdBufs b{};
  b.dh0_ba = a.take<float>(Na * kD); b.dh0_da = a.take<float>(Ea * kD); b.dh0_fc = a.take<float>(G * kD);
  b.dx_ba = a.take<float>(Na * kD);
  b.d_readout = a.take<float>(G * 2 * kD);
  b.dWpad_ba = a.take<float>(kPadMat); b.dWpad_da = a.take<float>(kPadMat);
  b.rec_ba = a.take<float>((size_t)kTailCtasMax * kRecSmall);
  b.rec_da = a.take<float>((size_t)kTailCtasMax * kRecSmall);
  b.rec_fc = a.take<float>((size_t)kTailCtasMax * kRecWide);
  b.scratch2 = a.take<float>(kScratchFloats);
  b.scratch3 = a.take<float>(kScratchFloats);
  b.loss_parts = a.take<float>(4);
  if (out) *out = b;
  return a.total();
}

// ---- operand packing --------------------------------------------------------------------------------------------------
// job j < 3: dst[j] = [W0 (64 x 128); 0 (64 x 128)], dstT[j] = its transpose (optional), bias[j] = [b0; 0]
// job 3..5 : dst = Wr[:, 128 (j-3) : 128 (j-2)]  (the three 128-column blocks of the 384-wide reduce layer)
struct PackJobs {
  const float *W0[3], *b0[3];
  float *Wpad[3], *WpadT[3], *bpad[3];
  const float *Wr;
  float *Wr_blk[3];
};
__global__ void __launch_bounds__(256) k_head_pack(PackJobs p) {
  pdl_wait();
  const int job = blockIdx.y;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < kPadMat; i += gridDim.x * blockDim.x) {
    const int r = i >> 7, c = i & 127;
    if (job < 3) {
      if (!p.Wpad[job]) return;
      const float v = r < 64 ? __ldg(p.W0[job] + r * kD + c) : 0.f;
      p.Wpad[job][i] = v;
      if (p.WpadT[job]) p.WpadT[job][c * kD + r] = v;
      if (i < kD) p.bpad[job][i] = i < 64 ? __ldg(p.b0[job] + i) : 0.f;
    } else {
      if (!p.Wr_blk[job - 3]) return;
      p.Wr_blk[job - 3][i] = __ldg(p.Wr + r * 3 * kD + (job - 3) * kD + c);
    }
  }
}

// T[i,:] = ReLU(U[ei0[i],:] + V[ei1[i],:] + T[i,:])   (the activation in front of bl_layers[0], pretrain_heads.py:72-73)
__global__ void __launch_bounds__(256) k_bl_combine(const float *__restrict__ U, const float *__restrict__ V,
                                                    float *__restrict__ T, const int64_t *__restrict__ ei, int64_t n_edges) {
  pdl_wait();
  const int64_t total = n_edges * 32;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t e = i >> 5;
    const int c = (int)(i & 31) * 4;
    const int64_t a = __ldg(ei + e), b = __ldg(ei + n_edges + e);
    const float4 u = ldg4(U + a * kD + c), v = ldg4(V + b * kD + c), t = ld4(T + e * kD + c);
    st4(T + e * kD + c, make_float4(fmaxf(u.x + v.x + t.x, 0.f), fmaxf(u.y + v.y + t.y, 0.f),
                                    fmaxf(u.z + v.z + t.z, 0.f), fmaxf(u.w + v.w + t.w, 0.f)));
  }
}

// ---- tails --------------------------------------------------------------------------------------------------------------
// out[r] = b2 + sum_j W2[j] ReLU(b1[j] + sum_k W1[j,k] ReLU(h0[r,k])),   k < IN, j < MID, h0 rows have stride 128.
struct TailJob {
  const float *h0;        // [n,128] first-layer pre-activations
  int64_t n;
  const float *W1, *b1, *W2, *b2;
  float *out;             // forward: [n]
  const float *gout;      // backward: [n] gradient of out
  float *dh0;             // backward: [n,128] gradient of h0 (columns IN.. written as zero)
  float *rec;             // backward: per-CTA records
  // fused loss (training step): with target != NULL the kernel forms the prediction itself and uses
  // gout[r] = 2 * loss_coef * (pred[r] - target[r]); the CTA's share of loss_coef * sum (pred - target)^2 goes into the
  // spare slot at the end of its record
  const float *target;
  float loss_coef;
};
struct TailJobs {
  TailJob j[3];
  int n;
};

template <int IN, int MID>
__device__ __forceinline__ void load_tail_weights(const TailJob &job, float *sW1t, float *sb1, float *sW2, float *sb2) {
  for (int i = threadIdx.x; i < IN * MID; i += blockDim.x) {
    const int k = i / MID, j = i - k * MID;
    sW1t[i] = __ldg(job.W1 + j * IN + k);
  }
  for (int i = threadIdx.x; i < MID; i += blockDim.x) {
    sb1[i] = __ldg(job.b1 + i);
    sW2[i] = __ldg(job.W2 + i);
  }
  if (threadIdx.x == 0) sb2[0] = __ldg(job.b2);
}

// Forward tail of the big heads (IN = 64, MID = 32), register-tiled like k_mlp_tail_bwd2's first GEMM: the ReLU(h0) tile
// in shared memory, a thread computes 8 rows x 4 hidden units (10.7 FMA per LDS.128 instead of 4), the 32-wide dot
// with W2 is finished by three shuffles over the 8 threads that share a row group.
__global__ void __launch_bounds__(128, 4) k_mlp_tail_fwd2(TailJobs J) {
  pdl_wait();
  constexpr int IN = 64, MID = 32, ROWS = 128, SA = 68;
  const TailJob &job = J.j[blockIdx.y];
  __shared__ __align__(16) float sW1t[IN * MID];
  __shared__ __align__(16) float sA[ROWS * SA];
  __shared__ __align__(16) float sb1[MID], sW2[MID];
  __shared__ float sb2[1];
  const int tid = threadIdx.x;
  const int64_t n_tiles = (job.n + ROWS - 1) / ROWS;
  if (blockIdx.x >= n_tiles) return;
  load_tail_weights<IN, MID>(job, sW1t, sb1, sW2, sb2);
  const int rg = tid >> 3, g8 = tid & 7;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t r0 = tile * ROWS;
    __syncthreads();
#pragma unroll 4
    for (int it = 0; it < 16; ++it) {
      const int idx = it * 128 + tid, r = idx >> 4, c4 = idx & 15;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r0 + r < job.n) v = ldg4(job.h0 + (r0 + r) * kD + c4 * 4);
      st4(sA + r * SA + c4 * 4, make_float4(fmaxf(v.x, 0.f), fmaxf(v.y, 0.f), fmaxf(v.z, 0.f), fmaxf(v.w, 0.f)));
    }
    __syncthreads();
    float acc[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int q = 0; q < 4; ++q) acc[i][q] = 0.f;
#pragma unroll 2
    for (int k4 = 0; k4 < IN / 4; ++k4) {
      float4 w[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) w[u] = ld4(sW1t + (k4 * 4 + u) * MID + g8 * 4);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float4 a = ld4(sA + (rg + 16 * i) * SA + k4 * 4);
        const float av[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          acc[i][0] = fmaf(av[u], w[u].x, acc[i][0]);
          acc[i][1] = fmaf(av[u], w[u].y, acc[i][1]);
          acc[i][2] = fmaf(av[u], w[u].z, acc[i][2]);
          acc[i][3] = fmaf(av[u], w[u].w, acc[i][3]);
        }
      }
    }
    const float4 b1v = ld4(sb1 + g8 * 4), w2v = ld4(sW2 + g8 * 4);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float o = fmaxf(acc[i][0] + b1v.x, 0.f) * w2v.x + fmaxf(acc[i][1] + b1v.y, 0.f) * w2v.y +
                fmaxf(acc[i][2] + b1v.z, 0.f) * w2v.z + fmaxf(acc[i][3] + b1v.w, 0.f) * w2v.w;
      o += __shfl_xor_sync(kFull, o, 1);
      o += __shfl_xor_sync(kFull, o, 2);
      o += __shfl_xor_sync(kFull, o, 4);
      const int64_t row = r0 + rg + 16 * i;
      if (g8 == 0 && row < job.n) job.out[row] = o + sb2[0];
    }
  }
}

// Backward tail of the two big heads (IN = 64, MID = 32) as three register-tiled FP32 GEMMs per 128-row tile, all
// operands in shared memory (the first version was thread-per-row with broadcast weight loads and ran at the
// shared-memory return bandwidth, 4 FMA per LDS.128: 118 us for 80 k rows; here 11-16 FMA per LDS.128):
//   P1  H1pre[r,j] = b1[j] + sum_k A[r,k] W1[j,k]      thread = 8 rows x 4 j     A = ReLU(h0) tile, row-major
//       D1[r,j]    = H1pre > 0 ? g[r] W2[j] : 0        (+ per-thread partials of db1, dW2, db2)
//   P2  dh0[r,k]   = A[r,k] > 0 ? sum_j D1[r,j] W1[j,k] : 0    thread = 8 rows x 8 k   (+ db0 partials) -> global
//   P3  dW1[j,k]  += sum_r D1[r,j] A[r,k]              thread = 4 j x 4 k, accumulated over all tiles of the CTA
// Rows of a thread are interleaved (r = rg + 16 i) so that the 4 row groups of a warp hit distinct banks.
constexpr int TB_ROWS = 128, TB_SA = 68, TB_SD = 36;
constexpr size_t kTailBwd2Smem = sizeof(float) * (2 * 64 * 32 + TB_ROWS * TB_SA + TB_ROWS * TB_SD + TB_ROWS + 68);

__global__ void __launch_bounds__(128, 3) k_mlp_tail_bwd2(TailJobs J) {
  pdl_wait();
  constexpr int IN = 64, MID = 32, REC = rec_floats(64, 32);
  const TailJob &job = J.j[blockIdx.y];
  extern __shared__ __align__(16) float smem[];
  float *sW1t = smem;                       // [IN][MID]   W1t[k][j] = W1[j][k]
  float *sW1 = sW1t + IN * MID;             // [MID][IN]
  float *sA = sW1 + IN * MID;               // [TB_ROWS][TB_SA]
  float *sD1 = sA + TB_ROWS * TB_SA;        // [TB_ROWS][TB_SD]
  float *sg = sD1 + TB_ROWS * TB_SD;        // [TB_ROWS]
  float *sb1 = sg + TB_ROWS;                // [32] b1, [32] W2
  float *sred = sA;                         // [16][80] end-of-kernel partials (the tile is dead by then)
  const int tid = threadIdx.x;
  const int64_t n_tiles = (job.n + TB_ROWS - 1) / TB_ROWS;
  if (blockIdx.x >= n_tiles && blockIdx.x > 0) return;   // CTA 0 always runs: it writes a (possibly zero) record
  for (int i = tid; i < IN * MID; i += 128) {
    const float w = __ldg(job.W1 + i);      // i = j * IN + k
    sW1[i] = w;
    sW1t[(i & (IN - 1)) * MID + (i >> 6)] = w;
  }
  if (tid < MID) {
    sb1[tid] = __ldg(job.b1 + tid);
    sb1[32 + tid] = __ldg(job.W2 + tid);
  }
  if (tid == 0) sb1[64] = __ldg(job.b2);
  const bool fused = job.target != nullptr;
  float lossp = 0.f;
  const int rg = tid >> 3, g8 = tid & 7;    // P1: j = 4 g8 .. +3;  P2: k = 4 g8 .. +3 and 32 + 4 g8 .. +3
  const int jb = tid >> 4, kb = tid & 15;   // P3: j = 4 jb .. +3, k = 4 kb .. +3
  float wacc[4][4];
#pragma unroll
  for (int p_ = 0; p_ < 4; ++p_)
#pragma unroll
    for (int q = 0; q < 4; ++q) wacc[p_][q] = 0.f;
  float db1p[4] = {0.f, 0.f, 0.f, 0.f}, dw2p[4] = {0.f, 0.f, 0.f, 0.f}, db0p[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  float db2p = 0.f;

  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t r0 = tile * TB_ROWS;
    __syncthreads();   // previous tile fully consumed (also publishes the weights on the first pass)
    // ---- stage A = ReLU(h0[:, 0:64]) and g
#pragma unroll 4
    for (int it = 0; it < 16; ++it) {
      const int idx = it * 128 + tid, r = idx >> 4, c4 = idx & 15;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r0 + r < job.n) v = ldg4(job.h0 + (r0 + r) * kD + c4 * 4);
      st4(sA + r * TB_SA + c4 * 4, make_float4(fmaxf(v.x, 0.f), fmaxf(v.y, 0.f), fmaxf(v.z, 0.f), fmaxf(v.w, 0.f)));
    }
    sg[tid] = r0 + tid < job.n ? __ldg((fused ? job.target : job.gout) + r0 + tid) : 0.f;
    __syncthreads();
    // ---- P1
    {
      float acc[8][4];
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int q = 0; q < 4; ++q) acc[i][q] = 0.f;
#pragma unroll 2
      for (int k4 = 0; k4 < IN / 4; ++k4) {
        float4 w[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) w[u] = ld4(sW1t + (k4 * 4 + u) * MID + g8 * 4);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 a = ld4(sA + (rg + 16 * i) * TB_SA + k4 * 4);
          const float av[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            acc[i][0] = fmaf(av[u], w[u].x, acc[i][0]);
            acc[i][1] = fmaf(av[u], w[u].y, acc[i][1]);
            acc[i][2] = fmaf(av[u], w[u].z, acc[i][2]);
            acc[i][3] = fmaf(av[u], w[u].w, acc[i][3]);
          }
        }
      }
      const float4 b1v = ld4(sb1 + g8 * 4), w2v = ld4(sb1 + 32 + g8 * 4);
      const float b1a[4] = {b1v.x, b1v.y, b1v.z, b1v.w}, w2a[4] = {w2v.x, w2v.y, w2v.z, w2v.w};
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int r = rg + 16 * i;
        float g = sg[r];
        if (fused) {   // prediction of the row: the 8 lanes of a row group hold 4 hidden units each
          float o = fmaxf(acc[i][0] + b1a[0], 0.f) * w2a[0] + fmaxf(acc[i][1] + b1a[1], 0.f) * w2a[1] +
                    fmaxf(acc[i][2] + b1a[2], 0.f) * w2a[2] + fmaxf(acc[i][3] + b1a[3], 0.f) * w2a[3];
          o += __shfl_xor_sync(kFull, o, 1);
          o += __shfl_xor_sync(kFull, o, 2);
          o += __shfl_xor_sync(kFull, o, 4);
          const float diff = r0 + r < job.n ? (o + sb1[64]) - g : 0.f;   // g held the target
          g = 2.f * job.loss_coef * diff;
          if (g8 == 0) lossp = fmaf(job.loss_coef * diff, diff, lossp);
        }
        float d[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float pre = acc[i][q] + b1a[q];
          d[q] = pre > 0.f ? g * w2a[q] : 0.f;
          db1p[q] += d[q];
          dw2p[q] = fmaf(g, fmaxf(pre, 0.f), dw2p[q]);
        }
        if (g8 == 0) db2p += g;
        st4(sD1 + r * TB_SD + g8 * 4, make_float4(d[0], d[1], d[2], d[3]));
      }
    }
    __syncthreads();
    // ---- P2
    {
      float acc[8][8];
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int q = 0; q < 8; ++q) acc[i][q] = 0.f;
#pragma unroll 1
      for (int j4 = 0; j4 < MID / 4; ++j4) {
        float4 wl[4], wh[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          wl[u] = ld4(sW1 + (j4 * 4 + u) * IN + g8 * 4);
          wh[u] = ld4(sW1 + (j4 * 4 + u) * IN + 32 + g8 * 4);
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 dv = ld4(sD1 + (rg + 16 * i) * TB_SD + j4 * 4);
          const float da[4] = {dv.x, dv.y, dv.z, dv.w};
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            acc[i][0] = fmaf(da[u], wl[u].x, acc[i][0]);
            acc[i][1] = fmaf(da[u], wl[u].y, acc[i][1]);
            acc[i][2] = fmaf(da[u], wl[u].z, acc[i][2]);
            acc[i][3] = fmaf(da[u], wl[u].w, acc[i][3]);
            acc[i][4] = fmaf(da[u], wh[u].x, acc[i][4]);
            acc[i][5] = fmaf(da[u], wh[u].y, acc[i][5]);
            acc[i][6] = fmaf(da[u], wh[u].z, acc[i][6]);
            acc[i][7] = fmaf(da[u], wh[u].w, acc[i][7]);
          }
        }
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int r = rg + 16 * i;
        const float4 al = ld4(sA + r * TB_SA + g8 * 4), ah = ld4(sA + r * TB_SA + 32 + g8 * 4);
        float4 lo, hi;
        lo.x = al.x > 0.f ? acc[i][0] : 0.f; lo.y = al.y > 0.f ? acc[i][1] : 0.f;
        lo.z = al.z > 0.f ? acc[i][2] : 0.f; lo.w = al.w > 0.f ? acc[i][3] : 0.f;
        hi.x = ah.x > 0.f ? acc[i][4] : 0.f; hi.y = ah.y > 0.f ? acc[i][5] : 0.f;
        hi.z = ah.z > 0.f ? acc[i][6] : 0.f; hi.w = ah.w > 0.f ? acc[i][7] : 0.f;
        db0p[0] += lo.x; db0p[1] += lo.y; db0p[2] += lo.z; db0p[3] += lo.w;
        db0p[4] += hi.x; db0p[5] += hi.y; db0p[6] += hi.z; db0p[7] += hi.w;
        if (r0 + r < job.n) {
          float *dp = job.dh0 + (r0 + r) * kD;
          st4(dp + g8 * 4, lo);
          st4(dp + 32 + g8 * 4, hi);
          st4(dp + 64 + g8 * 4, make_float4(0.f, 0.f, 0.f, 0.f));   // columns 64.. of the padded first layer
          st4(dp + 96 + g8 * 4, make_float4(0.f, 0.f, 0.f, 0.f));
        }
      }
    }
    // ---- P3 (reads sD1 and sA only: no barrier needed after P2)
#pragma unroll 4
    for (int r = 0; r < TB_ROWS; ++r) {
      const float4 dv = ld4(sD1 + r * TB_SD + jb * 4), av = ld4(sA + r * TB_SA + kb * 4);
      const float da[4] = {dv.x, dv.y, dv.z, dv.w};
#pragma unroll
      for (int p_ = 0; p_ < 4; ++p_) {
        wacc[p_][0] = fmaf(da[p_], av.x, wacc[p_][0]);
        wacc[p_][1] = fmaf(da[p_], av.y, wacc[p_][1]);
        wacc[p_][2] = fmaf(da[p_], av.z, wacc[p_][2]);
        wacc[p_][3] = fmaf(da[p_], av.w, wacc[p_][3]);
      }
    }
  }
  // ---- CTA record: [dW1 MID*IN][db1 MID][dW2 MID][db2 1][db0 IN]
  float *rec = job.rec + (size_t)blockIdx.x * REC;
#pragma unroll
  for (int p_ = 0; p_ < 4; ++p_)
    st4(rec + (jb * 4 + p_) * IN + kb * 4, make_float4(wacc[p_][0], wacc[p_][1], wacc[p_][2], wacc[p_][3]));
  // vector sums: 16 row groups share every (g8) column set; combine them in fixed order through shared memory
  __syncthreads();
  float *mine = sred + rg * 80;            // [db1 32][dW2 32][db2 8 (one per g8, only g8 == 0 is non-zero)] ... db0 separately
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    mine[g8 * 4 + q] = db1p[q];
    mine[32 + g8 * 4 + q] = dw2p[q];
  }
  mine[64 + g8] = db2p;
  mine[72 + g8] = lossp;
  __syncthreads();
  if (tid < 66) {
    float s_ = 0.f;
    const int col = tid < 64 ? tid : (tid == 64 ? 64 : 72);   // 64: db2, 72: loss share (g8 == 0 slots)
    for (int g = 0; g < 16; ++g) s_ += sred[g * 80 + col];
    rec[tid < 65 ? MID * IN + col : MID * IN + 2 * MID + 1 + IN] = s_;
  }
  __syncthreads();
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    mine[g8 * 4 + q] = db0p[q];
    mine[32 + g8 * 4 + q] = db0p[4 + q];
  }
  __syncthreads();
  if (tid < 64) {
    float s_ = 0.f;
    for (int g = 0; g < 16; ++g) s_ += sred[g * 80 + tid];
    rec[MID * IN + 2 * MID + 1 + tid] = s_;
  }
}

// ---- the energy head as ONE kernel ----------------------------------------------------------------------------------
// pretrain_heads.py:93-102 for G ~ 1e3 molecules is six latency-bound launches in a chain (two readout sums, first
// layer, tail forward+backward, input gradient, readout backward) that the encoder backward has to wait for: 165 us in
// the step (gpurun_out/r5k_device_profile.log) for 70 MFLOP.  Here a CTA takes 8 molecules through the whole chain in
// shared memory: readout (written out for the weight-gradient GEMM of the first layer) -> h0 = W0 readout + b0 ->
// tail forward, loss share, tail backward -> dh0 (written out, same GEMM) -> d_readout = dh0 W0 (atom half written out
// for the caller's gather, fragment half scattered to the molecule's fragment rows here) and the per-CTA record of the
// tail's parameter gradients (SumBuilder::add_tail's layout).  Exact FP32, fixed summation order.
// The pointers that are set select the mode:
//   target : fused loss (training step): g = 2 loss_coef (pred - target), the loss share goes into the record;
//   gout   : the caller's gradient of the prediction, g = gout; the loss share is 0;
//   neither: forward only: readout and pred; the tail's backward is skipped and no record is written.
struct EnergyArgs {
  const int *atom_ptr, *frag_ptr;             // [G + 1] molecule boundaries
  const float *x_atoms, *x_frags;             // [Na,128], [Nf,128]
  const float *W0, *b0, *W1, *b1, *W2, *b2;   // fc head: [128,256] [128] [64,128] [64] [64] [1]
  const float *target, *gout;                 // [G]
  float loss_coef;
  int G;
  float *readout, *pred, *dh0, *d_readout, *g_frags, *rec;
};
constexpr int EH_ROWS = 8, EH_THREADS = 256, EH_IN0 = 2 * kD, EH_H = kD, EH_MID = 64;
constexpr size_t kEnergySmem =
    sizeof(float) * ((size_t)2 * EH_H * EH_MID + EH_ROWS * EH_IN0 + 2 * EH_ROWS * EH_H + 2 * EH_ROWS * EH_H +
                     3 * EH_ROWS * EH_MID + 2 * EH_MID + 4 * EH_ROWS);

__global__ void __launch_bounds__(EH_THREADS) k_energy_head(EnergyArgs a) {
  constexpr int REC = rec_floats(EH_H, EH_MID);
  extern __shared__ __align__(16) float smem[];
  float *sW1 = smem;                          // [MID][H]   W1[i][k]
  float *sW1t = sW1 + EH_MID * EH_H;          // [H][MID]   W1t[k][i]
  float *sA = sW1t + EH_MID * EH_H;           // [ROWS][256] readout, later d_readout
  float *sH = sA + EH_ROWS * EH_IN0;          // [ROWS][128] h0 (pre-activation)
  float *sD0 = sH + EH_ROWS * EH_H;           // [ROWS][128] dh0
  float *sP = sD0 + EH_ROWS * EH_H;           // [2][ROWS][128] K-halves of h0
  float *sH1 = sP + 2 * EH_ROWS * EH_H;       // [ROWS][MID] hidden pre-activation
  float *sD1 = sH1 + EH_ROWS * EH_MID;        // [ROWS][MID]
  float *sH1g = sD1 + EH_ROWS * EH_MID;       // [ROWS][MID] g * ReLU(hidden)
  float *sb1 = sH1g + EH_ROWS * EH_MID;       // [MID] b1, [MID] W2
  float *sG = sb1 + 2 * EH_MID;               // [ROWS] g, [ROWS] loss share, [2 * ROWS] spare
  const int tid = threadIdx.x;
  for (int i = tid; i < EH_MID * EH_H; i += EH_THREADS) {   // parameters: before the dependency wait
    const float w = __ldg(a.W1 + i);      // i = unit * H + k
    sW1[i] = w;
    sW1t[(i & (EH_H - 1)) * EH_MID + (i >> 7)] = w;
  }
  if (tid < EH_MID) {
    sb1[tid] = __ldg(a.b1 + tid);
    sb1[EH_MID + tid] = __ldg(a.W2 + tid);
  }
  const float b2 = __ldg(a.b2);
  pdl_wait();
  const bool fwd_only = !a.target && !a.gout;
  const int oj = tid >> 2, ok0 = (tid & 3) * 4;   // dW1 ownership: row oj, columns ok0 + 16 q .. +3
  float wacc[32];
#pragma unroll
  for (int q = 0; q < 32; ++q) wacc[q] = 0.f;
  float vacc = 0.f, b0acc = 0.f, b2acc = 0.f, lossacc = 0.f;
  const int n_tiles = (a.G + EH_ROWS - 1) / EH_ROWS;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int g0 = tile * EH_ROWS, rows = min(EH_ROWS, a.G - g0);
    __syncthreads();
    // ---- readout (pretrain_heads.py:93-96): [sum of atom rows | sum of fragment rows]; one warp per molecule, a lane
    // owns 4 columns, 8 row loads in flight (a thread per column walking 8 molecules in turn was 50 dependent round
    // trips: half of the kernel's time)
    {
      const int m = tid >> 5, lane = tid & 31;
      float4 sum[2] = {make_float4(0.f, 0.f, 0.f, 0.f), make_float4(0.f, 0.f, 0.f, 0.f)};
      if (m < rows) {
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          const int *ptr = half ? a.frag_ptr : a.atom_ptr;
          const float *x = (half ? a.x_frags : a.x_atoms) + lane * 4;
          const int b = __ldg(ptr + g0 + m), e = __ldg(ptr + g0 + m + 1);
          float4 s_ = make_float4(0.f, 0.f, 0.f, 0.f);
          int r = b;
          for (; r + 8 <= e; r += 8) {
            float4 v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) v[u] = ldg4(x + (int64_t)(r + u) * kD);
#pragma unroll
            for (int u = 0; u < 8; ++u) { s_.x += v[u].x; s_.y += v[u].y; s_.z += v[u].z; s_.w += v[u].w; }
          }
          for (; r < e; ++r) {
            const float4 v = ldg4(x + (int64_t)r * kD);
            s_.x += v.x; s_.y += v.y; s_.z += v.z; s_.w += v.w;
          }
          sum[half] = s_;
          st4(a.readout + (int64_t)(g0 + m) * EH_IN0 + half * kD + lane * 4, s_);
        }
      }
      st4(sA + m * EH_IN0 + lane * 4, sum[0]);
      st4(sA + m * EH_IN0 + kD + lane * 4, sum[1]);
    }
    __syncthreads();
    // ---- h0 = readout W0^T + b0: thread = (output j, K-half), 8 molecules each
    {
      const int j = tid & 127, kh = tid >> 7;
      float acc[EH_ROWS];
#pragma unroll
      for (int m = 0; m < EH_ROWS; ++m) acc[m] = 0.f;
      const float *wrow = a.W0 + (int64_t)j * EH_IN0 + kh * kD;
      for (int k0 = 0; k0 < kD; k0 += 32) {
        float4 w[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) w[u] = ldg4(wrow + k0 + 4 * u);
#pragma unroll
        for (int u = 0; u < 8; ++u)
#pragma unroll
          for (int m = 0; m < EH_ROWS; ++m) {
            const float4 av = ld4(sA + m * EH_IN0 + kh * kD + k0 + 4 * u);
            acc[m] = fmaf(av.x, w[u].x, acc[m]);
            acc[m] = fmaf(av.y, w[u].y, acc[m]);
            acc[m] = fmaf(av.z, w[u].z, acc[m]);
            acc[m] = fmaf(av.w, w[u].w, acc[m]);
          }
      }
#pragma unroll
      for (int m = 0; m < EH_ROWS; ++m) sP[(kh * EH_ROWS + m) * EH_H + j] = acc[m];
    }
    __syncthreads();
    for (int i = tid; i < EH_ROWS * EH_H; i += EH_THREADS)
      sH[i] = (sP[i] + sP[EH_ROWS * EH_H + i]) + __ldg(a.b0 + (i & (EH_H - 1)));
    __syncthreads();
    // ---- hidden layer: thread = (unit i, molecule pair)
    {
      const int i = tid & 63, mp = tid >> 6;
      float acc0 = sb1[i], acc1 = sb1[i];
      const float *h0a = sH + (2 * mp) * EH_H, *h0b = h0a + EH_H;
#pragma unroll 4
      for (int k = 0; k < EH_H; ++k) {
        const float w = sW1t[k * EH_MID + i];
        acc0 = fmaf(fmaxf(h0a[k], 0.f), w, acc0);
        acc1 = fmaf(fmaxf(h0b[k], 0.f), w, acc1);
      }
      sH1[(2 * mp) * EH_MID + i] = acc0;
      sH1[(2 * mp + 1) * EH_MID + i] = acc1;
    }
    __syncthreads();
    // ---- prediction, loss share, gradient of the prediction
    if (tid < EH_ROWS) {
      float o = b2;
      for (int i = 0; i < EH_MID; ++i) o = fmaf(fmaxf(sH1[tid * EH_MID + i], 0.f), sb1[EH_MID + i], o);
      if (a.target) {
        const float diff = tid < rows ? o - __ldg(a.target + g0 + tid) : 0.f;
        sG[tid] = 2.f * a.loss_coef * diff;
        sG[EH_ROWS + tid] = a.loss_coef * diff * diff;
      } else if (fwd_only) {
        if (tid < rows) a.pred[g0 + tid] = o;
      } else {
        sG[tid] = tid < rows ? __ldg(a.gout + g0 + tid) : 0.f;
        sG[EH_ROWS + tid] = 0.f;
      }
    }
    if (fwd_only) continue;   // the same for every thread of the CTA: the next tile's barriers stay matched
    __syncthreads();
    {
      const int i = tid & 63, mp = tid >> 6;
#pragma unroll
      for (int d = 0; d < 2; ++d) {
        const int m = 2 * mp + d;
        const float pre = sH1[m * EH_MID + i], g = sG[m];
        sD1[m * EH_MID + i] = pre > 0.f ? g * sb1[EH_MID + i] : 0.f;
        sH1g[m * EH_MID + i] = g * fmaxf(pre, 0.f);
      }
    }
    __syncthreads();
    // ---- dh0: thread = (column k, molecule quad)
    {
      const int k = tid & 127, mh = tid >> 7;
      float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
      for (int i = 0; i < EH_MID; ++i) {
        const float w = sW1[i * EH_H + k];
#pragma unroll
        for (int q = 0; q < 4; ++q) acc[q] = fmaf(sD1[(4 * mh + q) * EH_MID + i], w, acc[q]);
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int m = 4 * mh + q;
        const float v = sH[m * EH_H + k] > 0.f ? acc[q] : 0.f;
        sD0[m * EH_H + k] = v;
        if (m < rows) a.dh0[(int64_t)(g0 + m) * kD + k] = v;
      }
    }
    __syncthreads();
    // ---- parameter-gradient partials of the tail (registers, summed over the CTA's tiles)
    for (int m = 0; m < EH_ROWS; ++m) {
      const float d = sD1[m * EH_MID + oj];
      const float *hp = sH + m * EH_H + ok0;
#pragma unroll
      for (int q4 = 0; q4 < 8; ++q4) {
        const float4 hv = ld4(hp + q4 * 16);
        wacc[q4 * 4 + 0] = fmaf(d, fmaxf(hv.x, 0.f), wacc[q4 * 4 + 0]);
        wacc[q4 * 4 + 1] = fmaf(d, fmaxf(hv.y, 0.f), wacc[q4 * 4 + 1]);
        wacc[q4 * 4 + 2] = fmaf(d, fmaxf(hv.z, 0.f), wacc[q4 * 4 + 2]);
        wacc[q4 * 4 + 3] = fmaf(d, fmaxf(hv.w, 0.f), wacc[q4 * 4 + 3]);
      }
      if ((tid & 3) == 0) vacc += d;
      else if ((tid & 3) == 1) vacc += sH1g[m * EH_MID + oj];
      if (tid < EH_H) b0acc += sD0[m * EH_H + tid];
      if (tid == 0) {
        b2acc += sG[m];
        lossacc += sG[EH_ROWS + m];
      }
    }
    // ---- d_readout = dh0 W0: thread = column c of the 256, 8 molecules
    {
      const int c = tid;
      float acc[EH_ROWS];
#pragma unroll
      for (int m = 0; m < EH_ROWS; ++m) acc[m] = 0.f;
      for (int j0 = 0; j0 < EH_H; j0 += 32) {
        float w[32];
#pragma unroll
        for (int u = 0; u < 32; ++u) w[u] = __ldg(a.W0 + (int64_t)(j0 + u) * EH_IN0 + c);
#pragma unroll
        for (int u = 0; u < 32; ++u)
#pragma unroll
          for (int m = 0; m < EH_ROWS; ++m) acc[m] = fmaf(sD0[m * EH_H + j0 + u], w[u], acc[m]);
      }
#pragma unroll
      for (int m = 0; m < EH_ROWS; ++m) {
        sA[m * EH_IN0 + c] = acc[m];    // (the readout was last read two barriers ago)
        if (m < rows) a.d_readout[(int64_t)(g0 + m) * EH_IN0 + c] = acc[m];
      }
    }
    __syncthreads();
    // ---- readout backward of the fragments: every fragment row receives its molecule's gradient
    {
      const int c = tid & 127, sub = tid >> 7;
      for (int m = 0; m < rows; ++m) {
        const int fb = __ldg(a.frag_ptr + g0 + m), fe = __ldg(a.frag_ptr + g0 + m + 1);
        const float v = sA[m * EH_IN0 + kD + c];
        for (int f = fb + sub; f < fe; f += 2) a.g_frags[(int64_t)f * kD + c] = v;
      }
    }
  }
  // ---- CTA record: [dW1 MID*H][db1 MID][dW2 MID][db2 1][db0 H][loss]
  pdl_launch_dependents();
  if (fwd_only) return;
  float *rec = a.rec + (size_t)blockIdx.x * REC;
#pragma unroll
  for (int q4 = 0; q4 < 8; ++q4)
    st4(rec + oj * EH_H + ok0 + q4 * 16, make_float4(wacc[q4 * 4], wacc[q4 * 4 + 1], wacc[q4 * 4 + 2], wacc[q4 * 4 + 3]));
  if ((tid & 3) == 0) rec[EH_MID * EH_H + oj] = vacc;
  if ((tid & 3) == 1) rec[EH_MID * EH_H + EH_MID + oj] = vacc;
  if (tid == 0) {
    rec[EH_MID * EH_H + 2 * EH_MID] = b2acc;
    rec[EH_MID * EH_H + 2 * EH_MID + 1 + EH_H] = lossacc;
  }
  if (tid < EH_H) rec[EH_MID * EH_H + 2 * EH_MID + 1 + tid] = b0acc;
}

// Fixed-order sum of per-CTA records (or a plain copy with n_blocks = 1) into the gradient tensors: one launch for all
// heads.  out[seg][i] = sum_b src[b * stride + off + i], i < width.
struct SumJobs {
  const float *src[20];
  int n_blocks[20], stride[20], off[20], width[20];
  float *out[20];
  int n;
};
__global__ void __launch_bounds__(256) k_head_sum_records(SumJobs s) {
  pdl_wait();
  // one CTA = 64 consecutive outputs of one segment; the records are split over 4 thread groups (fixed assignment and
  // fixed combination order => deterministic), each load instruction reads 256 contiguous bytes of one record
  __shared__ float part[4][64];
  const int seg = blockIdx.y;
  const int i = blockIdx.x * 64 + (threadIdx.x & 63), grp = threadIdx.x >> 6;
  if (blockIdx.x * 64 >= s.width[seg]) return;
  const int nb = s.n_blocks[seg], stride = s.stride[seg];
  const float *src = s.src[seg] + s.off[seg];
  float acc = 0.f;
  if (i < s.width[seg])
    for (int b = grp; b < nb; b += 4) acc += __ldg(src + (size_t)b * stride + i);
  part[grp][threadIdx.x & 63] = acc;
  __syncthreads();
  if (grp == 0 && i < s.width[seg]) s.out[seg][i] = (part[0][threadIdx.x] + part[1][threadIdx.x]) + (part[2][threadIdx.x] + part[3][threadIdx.x]);
}

__global__ void k_loss_total(const float *__restrict__ parts, int n, float *__restrict__ loss) {
  pdl_wait();
  if (threadIdx.x == 0) {
    float s_ = 0.f;
    for (int i = 0; i < n; ++i) s_ += parts[i];
    loss[0] = s_;
  }
}

struct SumBuilder {
  SumJobs s{};
  int max_width = 0;
  void add(const float *src, int n_blocks, int stride, int off, int width, float *out) {
    if (!out || width <= 0 || s.n >= 20) return;
    const int k = s.n++;
    s.src[k] = src; s.n_blocks[k] = n_blocks; s.stride[k] = stride; s.off[k] = off; s.width[k] = width; s.out[k] = out;
    if (width > max_width) max_width = width;
  }
  // tail record of a head: [dW1][db1][dW2][db2][db0]
  void add_tail(const float *rec, int n_ctas, int IN, int MID, float *dW1, float *db1, float *dW2, float *db2, float *db0) {
    const int stride = rec_floats(IN, MID);
    add(rec, n_ctas, stride, 0, MID * IN, dW1);
    add(rec, n_ctas, stride, MID * IN, MID, db1);
    add(rec, n_ctas, stride, MID * IN + MID, MID, dW2);
    add(rec, n_ctas, stride, MID * IN + 2 * MID, 1, db2);
    add(rec, n_ctas, stride, MID * IN + 2 * MID + 1, IN, db0);
  }
  int launch(cudaStream_t stream) {
    if (s.n == 0) return 0;
    if (cudaError_t le = fnb_launch(k_head_sum_records, dim3((max_width + 63) / 64, s.n), dim3(256), 0, stream, s)) return (int)le;
    FNB_CHECK_LAUNCH();
    return 0;
  }
};

int tail_grid(int64_t n, int rows) {
  int64_t t = (n + rows - 1) / rows;
  if (t > kTailCtasMax) t = kTailCtasMax;
  if (t < 1) t = 1;
  return (int)t;
}

// The kernels that use more than 48 KB of dynamic shared memory opt in once per device, before their first launch.
int opt_in_smem() {
  static bool done[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) return FNB_ERR_SIZE;
  if (!done[dev]) {
    RC((int)cudaFuncSetAttribute(k_mlp_tail_bwd2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTailBwd2Smem));
    RC((int)cudaFuncSetAttribute(k_energy_head, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kEnergySmem));
    done[dev] = true;
  }
  return 0;
}

// The energy head's inputs, parameters and readout buffer; the caller sets the pointers of the mode (EnergyArgs).
EnergyArgs energy_args(const fnb_pretrain_head_params *P, const fnb_pretrain_head_io *io, float *readout) {
  EnergyArgs e{};
  e.atom_ptr = io->mol_atom_ptr; e.frag_ptr = io->mol_frag_ptr; e.x_atoms = io->x_atoms; e.x_frags = io->x_frags;
  e.W0 = P->fc.W0; e.b0 = P->fc.b0; e.W1 = P->fc.W1; e.b1 = P->fc.b1; e.W2 = P->fc.W2; e.b2 = P->fc.b2;
  e.G = (int)io->n_graphs; e.readout = readout;
  return e;
}

int check_io(const fnb_pretrain_head_params *P, const fnb_pretrain_head_io *io) {
  if (!P || !io) return FNB_ERR_NULL;
  if (io->n_atoms < 0 || io->n_frags < 0 || io->n_edges < 0 || io->n_graphs < 0) return FNB_ERR_SIZE;
  if (io->n_atoms >= INT32_MAX || io->n_edges >= INT32_MAX) return FNB_ERR_SIZE;
  const fnb_mlp3_params *m[4] = {&P->bl, &P->ba, &P->da, &P->fc};
  for (int i = 0; i < 4; ++i)
    if (!m[i]->W0 || !m[i]->b0 || !m[i]->W1 || !m[i]->b1 || !m[i]->W2 || !m[i]->b2) return FNB_ERR_NULL;
  if (!P->Wr || !P->br) return FNB_ERR_NULL;
  if ((io->n_atoms && !io->x_atoms) || (io->n_frags && !io->x_frags) || (io->n_edges && (!io->edge_feat || !io->edge_index)))
    return FNB_ERR_NULL;
  if (io->n_graphs && (!io->mol_atom_ptr || !io->mol_frag_ptr)) return FNB_ERR_NULL;
  if (!fnb_aligned16(io->x_atoms) || !fnb_aligned16(io->x_frags) || !fnb_aligned16(io->edge_feat)) return FNB_ERR_ALIGN;
  return 0;
}

}  // namespace

extern "C" size_t fnb_pretrain_heads_workspace_bytes(int64_t n_atoms, int64_t n_edges, int64_t n_graphs) {
  if (n_atoms < 0 || n_edges < 0 || n_graphs < 0) return 0;
  return fwd_layout(n_atoms, n_edges, n_graphs, nullptr, nullptr);
}

extern "C" size_t fnb_pretrain_heads_bwd_workspace_bytes(int64_t n_atoms, int64_t n_edges, int64_t n_graphs) {
  if (n_atoms < 0 || n_edges < 0 || n_graphs < 0) return 0;
  return bwd_layout(n_atoms, n_edges, n_graphs, nullptr, nullptr);
}

extern "C" int fnb_pretrain_heads_forward(const fnb_pretrain_head_params *P, const fnb_pretrain_head_io *io,
                                          int precision, void *workspace, size_t workspace_bytes, void *scratch,
                                          void *stream_) {
  return fnb_pretrain_heads_forward_impl(P, io, precision, workspace, workspace_bytes, scratch, stream_, 0);
}

// skip_tails != 0: only the first layers of the per-atom / per-bond heads (what the backward needs); the training step
// forms the predictions inside the backward tails and the energy kernel (fused loss) and never materialises them.
int fnb_pretrain_heads_forward_impl(const fnb_pretrain_head_params *P, const fnb_pretrain_head_io *io, int precision,
                                    void *workspace, size_t workspace_bytes, void *scratch, void *stream_,
                                    int skip_tails) {
  RC(check_io(P, io));
  if (!workspace || !scratch) return FNB_ERR_NULL;
  if (!skip_tails && (!io->bond_angle || !io->dihedral || !io->energy)) return FNB_ERR_NULL;
  const int64_t Na = io->n_atoms, Ea = io->n_edges, G = io->n_graphs;
  FwdBufs B;
  if (fwd_layout(Na, Ea, G, (char *)workspace, &B) > workspace_bytes) return FNB_ERR_WORKSPACE;
  cudaStream_t stream = (cudaStream_t)stream_;
  const bool want_bl = io->bond_length != nullptr && Ea > 0 && !skip_tails;

  // ---- energy head: ~1e3 rows, one latency-bound kernel on an auxiliary stream underneath the per-atom / per-bond
  // heads.  Training step (skip_tails): the backward program runs it, forward included.
  FnbAux aux{};
  const bool two = fnb_aux_streams(&aux) == 0;
  cudaStream_t sB = two ? aux.hstream : stream;
  {  // padded / split operands (one launch)
    PackJobs p{};
    p.W0[0] = P->ba.W0; p.b0[0] = P->ba.b0; p.Wpad[0] = B.W0pad_ba; p.WpadT[0] = B.W0padT_ba; p.bpad[0] = B.b0pad_ba;
    p.W0[1] = P->da.W0; p.b0[1] = P->da.b0; p.Wpad[1] = B.W0pad_da; p.WpadT[1] = B.W0padT_da; p.bpad[1] = B.b0pad_da;
    if (want_bl) {
      p.W0[2] = P->bl.W0; p.b0[2] = P->bl.b0; p.Wpad[2] = B.W0pad_bl; p.WpadT[2] = nullptr; p.bpad[2] = B.b0pad_bl;
      p.Wr = P->Wr; p.Wr_blk[0] = B.Wr_a; p.Wr_blk[1] = B.Wr_b; p.Wr_blk[2] = B.Wr_e;
    }
    if (cudaError_t le = fnb_launch(k_head_pack, dim3(16, want_bl ? 6 : 2), dim3(256), 0, stream, p)) return (int)le;
    FNB_CHECK_LAUNCH();
  }
  // ---- energy head (graph readout pretrain_heads.py:93-96, first layer, tail)
  if (G > 0 && !skip_tails) {
    RC(opt_in_smem());
    if (two) {
      RC((int)cudaEventRecord(aux.fork, stream));
      RC((int)cudaStreamWaitEvent(sB, aux.fork, 0));
    }
    EnergyArgs e = energy_args(P, io, B.readout);
    e.pred = io->energy;
    if (cudaError_t le = fnb_launch(k_energy_head, dim3(tail_grid(G, EH_ROWS)), dim3(EH_THREADS), kEnergySmem, sB, e))
      return (int)le;
    FNB_CHECK_LAUNCH();
  }
  // ---- first layers on the projection kernels
  RC(fnb_proj_fwd(io->x_atoms, B.W0pad_ba, B.b0pad_ba, Na, kD, nullptr, 0, 0, 0, B.h0_ba, nullptr, precision, stream_));
  RC(fnb_proj_fwd(io->edge_feat, B.W0pad_da, B.b0pad_da, Ea, kD, nullptr, 0, 0, 0, B.h0_da, nullptr, precision, stream_));
  if (want_bl) {
    RC(fnb_proj_fwd(io->x_atoms, B.Wr_a, nullptr, Na, kD, nullptr, 0, 0, 0, B.U, nullptr, precision, stream_));
    RC(fnb_proj_fwd(io->x_atoms, B.Wr_b, nullptr, Na, kD, nullptr, 0, 0, 0, B.V, nullptr, precision, stream_));
    RC(fnb_proj_fwd(io->edge_feat, B.Wr_e, P->br, Ea, kD, nullptr, 0, 0, 0, B.T, nullptr, precision, stream_));
    int64_t blocks = (Ea * 32 + 255) / 256;
    if (blocks > kNumSMs * 16) blocks = kNumSMs * 16;
    if (cudaError_t le = fnb_launch(k_bl_combine, dim3((int)blocks), dim3(256), 0, stream, B.U, B.V, B.T, io->edge_index, Ea)) return (int)le;
    FNB_CHECK_LAUNCH();
    RC(fnb_proj_fwd(B.T, B.W0pad_bl, B.b0pad_bl, Ea, kD, nullptr, 0, 0, 0, B.h0_bl, nullptr, precision, stream_));
  }
  // ---- tails of the per-atom / per-bond heads
  if (!skip_tails) {
    TailJobs J{};
    int64_t most = 0;
    auto add = [&](const float *h0, int64_t n, const fnb_mlp3_params &m, float *out) {
      if (n <= 0) return;
      TailJob &t = J.j[J.n++];
      t.h0 = h0; t.n = n; t.W1 = m.W1; t.b1 = m.b1; t.W2 = m.W2; t.b2 = m.b2; t.out = out;
      if (n > most) most = n;
    };
    add(B.h0_ba, Na, P->ba, io->bond_angle);
    add(B.h0_da, Ea, P->da, io->dihedral);
    if (want_bl) add(B.h0_bl, Ea, P->bl, io->bond_length);
    if (J.n) {
      int64_t gx = (most + 127) / 128;
      if (gx > kNumSMs * 8) gx = kNumSMs * 8;
      if (cudaError_t le = fnb_launch(k_mlp_tail_fwd2, dim3((unsigned)gx, J.n), dim3(128), 0, stream, J)) return (int)le;
      FNB_CHECK_LAUNCH();
    }
  }
  // skip_tails: the caller (fnb_pretrain_step) runs the backward program next on the same streams; the energy chain
  // stays on its stream (the backward continues it there and joins once, before the readout gradient) instead of
  // making the per-atom / per-bond tails wait ~40 us for a 1 024-row GEMM (gpurun_out/r4n_device_profile.log)
  if (two && G > 0 && !skip_tails) {
    RC((int)cudaEventRecord(aux.join, sB));
    RC((int)cudaStreamWaitEvent(stream, aux.join, 0));
  }
  return 0;
}

// defer_join != 0: the weight gradients still running on the auxiliary streams are NOT joined into the caller's
// stream at return: fnb_pretrain_step joins the weight-gradient stream through the encoder backward that follows
// (which ends by waiting for that in-order stream) and the energy head's stream through aux.h_done.
int fnb_pretrain_heads_backward_impl(const fnb_pretrain_head_params *P, const fnb_pretrain_head_grads *D,
                                     const fnb_pretrain_head_io *io, int precision, void *workspace,
                                     size_t workspace_bytes, void *bwd_workspace, size_t bwd_workspace_bytes,
                                     void *scratch, void *stream_, int defer_join, const fnb_mse_term *fused,
                                     float *loss_out) {
  RC(check_io(P, io));
  if (!D || !workspace || !bwd_workspace || !scratch) return FNB_ERR_NULL;
  // fused != NULL: [0] bond angle, [1] dihedral, [2] energy targets and weights; the tails then compute
  // g = 2 w / n (pred - target) themselves and loss_out receives sum_t w_t mean((pred_t - target_t)^2)
  if (!fused && (!io->g_bond_angle || !io->g_dihedral || !io->g_energy)) return FNB_ERR_NULL;
  if (fused && (!loss_out || !fused[0].target || !fused[1].target || !fused[2].target)) return FNB_ERR_NULL;
  if (!io->g_atoms || !io->g_frags || !io->g_edge) return FNB_ERR_NULL;
  if (!io->batch32 || !io->frag_batch32) return FNB_ERR_NULL;
  const fnb_mlp3_grads *gm[3] = {&D->ba, &D->da, &D->fc};
  for (int i = 0; i < 3; ++i)
    if (!gm[i]->W0 || !gm[i]->b0 || !gm[i]->W1 || !gm[i]->b1 || !gm[i]->W2 || !gm[i]->b2) return FNB_ERR_NULL;
  const int64_t Na = io->n_atoms, Ea = io->n_edges, G = io->n_graphs;
  FwdBufs B;
  BwdBufs W;
  if (fwd_layout(Na, Ea, G, (char *)workspace, &B) > workspace_bytes) return FNB_ERR_WORKSPACE;
  if (bwd_layout(Na, Ea, G, (char *)bwd_workspace, &W) > bwd_workspace_bytes) return FNB_ERR_WORKSPACE;
  cudaStream_t stream = (cudaStream_t)stream_;

  FnbAux aux{};
  const bool two = fnb_aux_streams(&aux) == 0;
  cudaStream_t sB = two ? aux.hstream : stream;
  void *sB_ = (void *)sB;
  void *scratchB = two ? (void *)W.scratch2 : scratch;
  int ctas_ba = 0, ctas_da = 0, ctas_fc = 0;
  RC(opt_in_smem());
  // ---- energy head on the auxiliary stream (latency-bound ~1e3-row work that hides under the other heads): readout,
  // first layer, tail forward and backward (with the loss in the training step), input gradient and the fragments'
  // readout backward in one kernel, then the weight gradient of the first layer
  if (G > 0) {
    if (two) {
      RC((int)cudaEventRecord(aux.fork, stream));
      RC((int)cudaStreamWaitEvent(sB, aux.fork, 0));
      RC((int)cudaMemsetAsync(W.scratch2, 0, kScratchCounters * sizeof(float), sB));
    }
    EnergyArgs e = energy_args(P, io, B.readout);
    if (fused) {
      e.target = fused[2].target;
      e.loss_coef = fused[2].weight / (float)G;
    } else {
      e.gout = io->g_energy;
    }
    e.dh0 = W.dh0_fc; e.d_readout = W.d_readout; e.g_frags = io->g_frags; e.rec = W.rec_fc;
    ctas_fc = tail_grid(G, EH_ROWS);
    if (cudaError_t le = fnb_launch(k_energy_head, dim3(ctas_fc), dim3(EH_THREADS), kEnergySmem, sB, e)) return (int)le;
    FNB_CHECK_LAUNCH();
    if (two) RC((int)cudaEventRecord(aux.join, sB));
    RC(fnb_proj_bwd_dw(B.readout, W.dh0_fc, G, 2 * kD, D->fc.W0, nullptr, precision, scratchB, sB_));
    if (two) RC((int)cudaEventRecord(defer_join ? aux.h_done : aux.wjoin, sB));
  } else {
    RC((int)cudaMemsetAsync(D->fc.W0, 0, sizeof(float) * kD * 2 * kD, stream));
    if (two && defer_join) RC((int)cudaEventRecord(aux.h_done, stream));
  }
  // ---- tails of the per-atom / per-bond heads: dh0 + per-CTA records of their tail gradients
  {
    TailJobs J{};
    auto add = [&](const float *h0, int64_t n, const fnb_mlp3_params &m, const float *gout, float *dh0, float *rec) {
      TailJob &t = J.j[J.n++];
      t.h0 = h0; t.n = n; t.W1 = m.W1; t.b1 = m.b1; t.W2 = m.W2; t.b2 = m.b2; t.gout = gout; t.dh0 = dh0; t.rec = rec;
    };
    ctas_ba = tail_grid(Na, 128);
    ctas_da = tail_grid(Ea, 128);
    add(B.h0_ba, Na, P->ba, io->g_bond_angle, W.dh0_ba, W.rec_ba);
    add(B.h0_da, Ea, P->da, io->g_dihedral, W.dh0_da, W.rec_da);
    if (fused) {
      J.j[0].target = fused[0].target; J.j[0].loss_coef = Na > 0 ? fused[0].weight / (float)Na : 0.f;
      J.j[1].target = fused[1].target; J.j[1].loss_coef = Ea > 0 ? fused[1].weight / (float)Ea : 0.f;
    }
    const int gx = ctas_ba > ctas_da ? ctas_ba : ctas_da;
    // a job with fewer tiles than gx: its surplus CTAs return at once and write no record, so the record count of a
    // job is min(gx, tiles of the job) = its own tail_grid
    if (cudaError_t le = fnb_launch(k_mlp_tail_bwd2, dim3(gx, 2), dim3(128), kTailBwd2Smem, stream, J)) return (int)le;
    FNB_CHECK_LAUNCH();
  }
  // ---- first layers: dX on the caller's stream (it feeds the encoder backward), dW on the weight-gradient stream
  cudaStream_t sW = two ? aux.wstream : stream;
  void *sW_ = (void *)sW;
  void *scratchW = two ? (void *)W.scratch3 : scratch;
  if (two) {
    RC((int)cudaEventRecord(aux.ready[0], stream));     // dh0 of both heads is complete
    RC((int)cudaStreamWaitEvent(sW, aux.ready[0], 0));
    RC((int)cudaMemsetAsync(W.scratch3, 0, kScratchCounters * sizeof(float), sW));
  }
  if (Na > 0) {
    RC(fnb_proj_bwd_dx(B.W0pad_ba, B.W0padT_ba, W.dh0_ba, Na, kD, W.dx_ba, precision, scratch, stream_));
    RC(fnb_proj_bwd_dw(io->x_atoms, W.dh0_ba, Na, kD, W.dWpad_ba, nullptr, precision, scratchW, sW_));
  } else {
    RC((int)cudaMemsetAsync(W.dWpad_ba, 0, sizeof(float) * kPadMat, sW));
  }
  if (Ea > 0) {
    RC(fnb_proj_bwd_dx(B.W0pad_da, B.W0padT_da, W.dh0_da, Ea, kD, io->g_edge, precision, scratch, stream_));
    RC(fnb_proj_bwd_dw(io->edge_feat, W.dh0_da, Ea, kD, W.dWpad_da, nullptr, precision, scratchW, sW_));
  } else {
    RC((int)cudaMemsetAsync(W.dWpad_da, 0, sizeof(float) * kPadMat, sW));
  }
  {  // the 64-row slices of the padded first-layer gradients, on the stream that produced them
    SumBuilder cp;
    cp.add(W.dWpad_ba, 1, 0, 0, 64 * kD, D->ba.W0);
    cp.add(W.dWpad_da, 1, 0, 0, 64 * kD, D->da.W0);
    RC(cp.launch(sW));
  }
  if (G > 0) {
    if (two) RC((int)cudaStreamWaitEvent(stream, aux.join, 0));
    // readout backward (pretrain_heads.py:93-96): every atom receives its molecule's gradient row on top of the
    // bond-angle head's gradient
    RC(fnb_segment_gather(W.d_readout, 2 * kD, io->batch32, Na, W.dx_ba, io->g_atoms, stream_));
  }
  // ---- parameter gradients of the tails and the 64-row slices of the padded first-layer gradients
  SumBuilder sb;
  sb.add_tail(W.rec_ba, ctas_ba, 64, 32, D->ba.W1, D->ba.b1, D->ba.W2, D->ba.b2, D->ba.b0);
  sb.add_tail(W.rec_da, ctas_da, 64, 32, D->da.W1, D->da.b1, D->da.W2, D->da.b2, D->da.b0);
  sb.add_tail(W.rec_fc, ctas_fc, 128, 64, D->fc.W1, D->fc.b1, D->fc.W2, D->fc.b2, D->fc.b0);
  if (fused) {
    sb.add(W.rec_ba, ctas_ba, kRecSmall, 64 * 32 + 2 * 32 + 1 + 64, 1, W.loss_parts + 0);
    sb.add(W.rec_da, ctas_da, kRecSmall, 64 * 32 + 2 * 32 + 1 + 64, 1, W.loss_parts + 1);
    sb.add(W.rec_fc, ctas_fc, kRecWide, 128 * 64 + 2 * 64 + 1 + 128, 1, W.loss_parts + 2);
  }
  // (on the weight-gradient stream: the encoder backward that follows on the caller's stream needs none of this; the
  // tails' records are complete at aux.ready[0], which that stream has waited for, the energy head's at aux.join)
  if (two && G > 0) RC((int)cudaStreamWaitEvent(sW, aux.join, 0));
  RC(sb.launch(sW));
  if (fused) {
    if (cudaError_t le = fnb_launch(k_loss_total, dim3(1), dim3(32), 0, sW, (const float *)W.loss_parts, 3, loss_out))
      return (int)le;
    FNB_CHECK_LAUNCH();
  }
  if (two) RC((int)cudaEventRecord(aux.done[0], sW));
  if (two && !defer_join) {
    if (G > 0) RC((int)cudaStreamWaitEvent(stream, aux.wjoin, 0));   // energy head's first-layer weight gradient
    RC((int)cudaStreamWaitEvent(stream, aux.done[0], 0));            // first-layer weight gradients of the other heads
  }
  return 0;
}

extern "C" int fnb_pretrain_heads_backward(const fnb_pretrain_head_params *P, const fnb_pretrain_head_grads *D,
                                           const fnb_pretrain_head_io *io, int precision, void *workspace,
                                           size_t workspace_bytes, void *bwd_workspace, size_t bwd_workspace_bytes,
                                           void *scratch, void *stream_) {
  return fnb_pretrain_heads_backward_impl(P, D, io, precision, workspace, workspace_bytes, bwd_workspace,
                                          bwd_workspace_bytes, scratch, stream_, 0, nullptr, nullptr);
}

// ------------------------------------------------------------------------------------------------------------------------
// Loss of the pretraining loop (pretrain_utils.py:22-26): a weighted sum of mean-squared errors,
//   loss = sum_t w_t / n_t * sum_i (pred_t[i] - target_t[i])^2,   grad_t[i] = 2 w_t / n_t (pred_t[i] - target_t[i])
// in one launch (the reference's effective weights are dihedral 2, angle 1, energy 1 because loss_lngth is overwritten).
namespace {
struct MseArgs {
  const float *pred[4], *target[4];
  float *grad[4];
  int64_t n[4], begin[5];
  float w[4];
  int n_terms;
  float *loss;
  float *scratch;
};
__global__ void __launch_bounds__(256) k_mse_sum(MseArgs a) {
  pdl_wait();
  __shared__ float s_part[8];
  __shared__ float s_rec[4], s_fin[4];
  const int64_t total = a.begin[a.n_terms];
  float acc = 0.f;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int t = 0;
    while (t + 1 < a.n_terms && i >= a.begin[t + 1]) ++t;
    const int64_t k = i - a.begin[t];
    const float d = __ldg(a.pred[t] + k) - __ldg(a.target[t] + k);
    const float c = a.w[t] / (float)a.n[t];
    acc = fmaf(c * d, d, acc);
    if (a.grad[t]) a.grad[t][k] = 2.f * c * d;
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 4) {
    float s = 0.f;
    if (threadIdx.x == 0)
      for (int w = 0; w < 8; ++w) s += s_part[w];
    s_rec[threadIdx.x] = s;
  }
  __syncthreads();
  if (!cta_finish<4>(s_rec, s_fin, a.scratch)) return;
  if (threadIdx.x == 0) a.loss[0] = s_fin[0];
}
}  // namespace

extern "C" int fnb_mse_sum_loss(const fnb_mse_term *terms, int n_terms, float *loss, void *scratch, void *stream) {
  if (!terms || !loss || !scratch) return FNB_ERR_NULL;
  if (n_terms < 1 || n_terms > 4) return FNB_ERR_SIZE;
  MseArgs a{};
  a.n_terms = n_terms;
  a.loss = loss;
  a.scratch = reinterpret_cast<float *>(scratch);
  int64_t total = 0;
  for (int t = 0; t < n_terms; ++t) {
    if (terms[t].n <= 0) return FNB_ERR_SIZE;
    if (!terms[t].pred || !terms[t].target) return FNB_ERR_NULL;
    a.pred[t] = terms[t].pred; a.target[t] = terms[t].target; a.grad[t] = terms[t].grad; a.n[t] = terms[t].n;
    a.w[t] = terms[t].weight;
    a.begin[t] = total;
    total += terms[t].n;
  }
  a.begin[n_terms] = total;
  int64_t blocks = (total + 255) / 256;
  if (blocks > kNumSMs * 2) blocks = kNumSMs * 2;
  if (cudaError_t le = fnb_launch(k_mse_sum, dim3((int)blocks), dim3(256), 0, (cudaStream_t)stream, a)) return (int)le;
  FNB_CHECK_LAUNCH();
  return 0;
}
