// Data-parallel gradient exchange fused with the optimizer: ONE kernel per step that reads every rank's gradient buffer
// over NVLink / NVSwitch peer memory, averages in a fixed rank order and applies Adam to the local parameters.
//
// Reference: Lightning Fabric DDP (fragnet/train/finetune/finetune_gat2_pl.py:230, utils_pl.py:88) = NCCL all-reduce of
// the gradients (mean) followed by torch.optim.Adam.step.  The live gradient of the GAT2 pretraining model is ~1.4 MB:
// latency-bound, not link-bound (DESIGN.md section 7) -- ncclAllReduce + the 1/W scale + the Adam launch cost ~55 us of
// a 1.3 ms step at 8 GPUs, most of it protocol and launch latency.  Here the exchange is the optimizer's own read:
//   1. flag barrier over peer memory (every rank has finished its backward: release store of the step number into
//      every peer's flag row, acquire spin on the own row);
//   2. g[i] = (1/W) * sum_{r = 0..W-1} g_r[i]  with 16-byte peer loads, r ascending on every rank => bitwise identical
//      parameters everywhere (what an all-reduce guarantees) and run-to-run deterministic; Adam on p, m, v in place;
//   3. second flag barrier by the last CTA (nobody may overwrite its gradient buffer while a peer still reads it).
// The gradient buffers and the flag rows live in symmetric memory (torch.distributed._symmetric_memory: cudaMalloc'd,
// peer-mapped at rendezvous); the library only sees raw device pointers (fnb_peer_set).
// fnb_allreduce_adam_runs is the same kernel with per-run Adam step counts: a small table of runs that tile the flat
// buffer, each with its own bias corrections (torch.optim.Adam keeps one step count per parameter; a resumed run with
// gradual unfreezing has parameters at different counts).  The finetuning step uses it too: its gradient is ~7.8 MB
// for the e1pt4 head against ~1.4 MB for pretraining, and every rank reads all W buffers (W x 7.8 MB per rank and step).
#include "common.cuh"

namespace {

__device__ __forceinline__ void st_release_sys(unsigned *p, unsigned v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned *p) {
  unsigned v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// peer (or own) gradient: system-coherent, not cached in L1
__device__ __forceinline__ float4 ld_peer4(const float *p) {
  float4 v;
  asm volatile("ld.relaxed.sys.global.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p)
               : "memory");
  return v;
}
// Bounded spin: a rank that never arrives traps this kernel (launch failure) instead of hanging the GPU for good.
__device__ __forceinline__ void wait_flag(const unsigned *p, unsigned epoch) {
  for (unsigned long long spins = 0; (int)(ld_acquire_sys(p) - epoch) < 0; ++spins)
    if (spins > (1ull << 31)) __trap();
}

struct AdamArgs {
  float *p, *m, *v;
  int64_t n;             // floats, multiple of 4 (flat buffers are 256-byte aligned per tensor)
  float beta1, beta2, eps, weight_decay, step_size, inv_sqrt_bc2, inv_world;
  unsigned epoch;
  unsigned *done;        // device-local arrival counter of this kernel's CTAs (zero between launches)
};

// The exchange and the update; coef(i4, step_size, inv_sqrt_bc2) gives the bias corrections of the 4 floats at 4 * i4
// (an Adam run boundary never splits them).
template <class Coef>
__device__ __forceinline__ void allreduce_adam(const fnb_peer_set &ps, const AdamArgs &a, Coef coef) {
  const int W = ps.world, me = ps.rank;
  // ---- 1. every rank's gradient is complete
  if (blockIdx.x == 0 && threadIdx.x < W) {
    __threadfence_system();
    st_release_sys(reinterpret_cast<unsigned *>(ps.flags[threadIdx.x]) + me, a.epoch);
  }
  if (threadIdx.x < W) wait_flag(reinterpret_cast<const unsigned *>(ps.flags[me]) + threadIdx.x, a.epoch);
  __syncthreads();
  // ---- 2. mean gradient in rank order + Adam (torch.optim.Adam, no amsgrad)
  const int64_t n4 = a.n >> 2;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 8
    for (int r = 0; r < W; ++r) {
      const float4 x = ld_peer4(reinterpret_cast<const float *>(ps.grads[r]) + 4 * i);
      g.x += x.x; g.y += x.y; g.z += x.z; g.w += x.w;
    }
    float step_size, inv_sqrt_bc2;
    coef(i, step_size, inv_sqrt_bc2);
    float4 p = ld4(a.p + 4 * i), m = ld4(a.m + 4 * i), v = ld4(a.v + 4 * i);
    float *gp = &g.x, *pp = &p.x, *mp = &m.x, *vp = &v.x;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float gk = gp[k] * a.inv_world;
      if (a.weight_decay != 0.f) gk = fmaf(a.weight_decay, pp[k], gk);
      mp[k] = fmaf(a.beta1, mp[k], (1.f - a.beta1) * gk);
      vp[k] = fmaf(a.beta2, vp[k], (1.f - a.beta2) * gk * gk);
      pp[k] -= step_size * mp[k] / (sqrtf(vp[k]) * inv_sqrt_bc2 + a.eps);
    }
    st4(a.p + 4 * i, p); st4(a.m + 4 * i, m); st4(a.v + 4 * i, v);
  }
  // ---- 3. all ranks are done reading: only then may anyone's next backward overwrite its gradient buffer
  __shared__ int s_last;
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    s_last = atomicAdd(a.done, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!s_last) return;
  if (threadIdx.x == 0) *a.done = 0;
  if (threadIdx.x < W) {
    __threadfence_system();
    st_release_sys(reinterpret_cast<unsigned *>(ps.flags[threadIdx.x]) + W + me, a.epoch);
    wait_flag(reinterpret_cast<const unsigned *>(ps.flags[me]) + W + threadIdx.x, a.epoch);
  }
}

__global__ void __launch_bounds__(256) k_allreduce_adam(fnb_peer_set ps, AdamArgs a) {
  allreduce_adam(ps, a, [&](int64_t, float &step_size, float &inv_sqrt_bc2) {
    step_size = a.step_size;
    inv_sqrt_bc2 = a.inv_sqrt_bc2;
  });
}

// Per-run bias corrections: run r covers the float4 groups [end4[r-1], end4[r]) (end4[-1] = 0) and tiles the buffer.
struct AdamRunTable {
  int64_t end4[FNB_MAX_ADAM_RUNS];
  float step_size[FNB_MAX_ADAM_RUNS], inv_sqrt_bc2[FNB_MAX_ADAM_RUNS];
};

// A thread's float4 groups ascend, so its run index only moves forward.  __grid_constant__: the table is read from the
// parameter bank with a dynamic index, not copied to local memory.
__global__ void __launch_bounds__(256) k_allreduce_adam_runs(fnb_peer_set ps, AdamArgs a,
                                                             const __grid_constant__ AdamRunTable rt) {
  int run = 0;
  allreduce_adam(ps, a, [&](int64_t i4, float &step_size, float &inv_sqrt_bc2) {
    while (i4 >= rt.end4[run]) ++run;
    step_size = rt.step_size[run];
    inv_sqrt_bc2 = rt.inv_sqrt_bc2[run];
  });
}

// Argument checks and launch arguments shared by both entry points (bias corrections left to the caller); blocks = 0:
// nothing to do (n == 0).
int adam_args(const fnb_peer_set *peers, float *param, float *exp_avg, float *exp_avg_sq, int64_t n, float beta1,
              float beta2, float eps, float weight_decay, int64_t step, uint32_t epoch, void *done_counter,
              AdamArgs &a, int &blocks) {
  blocks = 0;
  if (!peers || !param || !exp_avg || !exp_avg_sq || !done_counter) return FNB_ERR_NULL;
  if (n < 0 || (n & 3) || step < 1 || peers->world < 1 || peers->world > FNB_MAX_PEERS || peers->rank < 0 ||
      peers->rank >= peers->world)
    return FNB_ERR_SIZE;
  if (n == 0) return 0;
  for (int r = 0; r < peers->world; ++r) {
    if (!peers->grads[r] || !peers->flags[r]) return FNB_ERR_NULL;
    if (!fnb_aligned16(peers->grads[r])) return FNB_ERR_ALIGN;
  }
  if (!fnb_aligned16(param) || !fnb_aligned16(exp_avg) || !fnb_aligned16(exp_avg_sq)) return FNB_ERR_ALIGN;
  a.p = param; a.m = exp_avg; a.v = exp_avg_sq; a.n = n; a.beta1 = beta1; a.beta2 = beta2; a.eps = eps;
  a.weight_decay = weight_decay; a.step_size = a.inv_sqrt_bc2 = 0.f;
  a.inv_world = 1.f / (float)peers->world; a.epoch = epoch; a.done = reinterpret_cast<unsigned *>(done_counter);
  int64_t b = ((n >> 2) + 255) / 256;
  if (b > kNumSMs) b = kNumSMs;           // every CTA spins on the flags: keep them all resident
  if (b < 1) b = 1;
  blocks = (int)b;
  return 0;
}

void bias_corrections(float lr, float beta1, float beta2, int64_t step, float &step_size, float &inv_sqrt_bc2) {
  const double bc1 = 1.0 - pow((double)beta1, (double)step), bc2 = 1.0 - pow((double)beta2, (double)step);
  step_size = (float)(lr / bc1);
  inv_sqrt_bc2 = (float)(1.0 / sqrt(bc2));
}

}  // namespace

extern "C" int fnb_allreduce_adam_step(const fnb_peer_set *peers, float *param, float *exp_avg, float *exp_avg_sq,
                                       int64_t n, float lr, float beta1, float beta2, float eps, float weight_decay,
                                       int64_t step, uint32_t epoch, void *done_counter, void *stream) {
  AdamArgs a;
  int blocks;
  if (int rc = adam_args(peers, param, exp_avg, exp_avg_sq, n, beta1, beta2, eps, weight_decay, step, epoch,
                         done_counter, a, blocks))
    return rc;
  if (blocks == 0) return 0;
  bias_corrections(lr, beta1, beta2, step, a.step_size, a.inv_sqrt_bc2);
  k_allreduce_adam<<<blocks, 256, 0, (cudaStream_t)stream>>>(*peers, a);
  FNB_CHECK_LAUNCH();
  return 0;
}

extern "C" int fnb_allreduce_adam_runs(const fnb_peer_set *peers, float *param, float *exp_avg, float *exp_avg_sq,
                                       int64_t n, const fnb_adam_run *runs, int n_runs, float lr, float beta1,
                                       float beta2, float eps, float weight_decay, uint32_t epoch, void *done_counter,
                                       void *stream) {
  AdamArgs a;
  int blocks;
  if (!runs) return FNB_ERR_NULL;
  if (int rc = adam_args(peers, param, exp_avg, exp_avg_sq, n, beta1, beta2, eps, weight_decay, 1, epoch,
                         done_counter, a, blocks))
    return rc;
  if (blocks == 0) return 0;
  if (n_runs < 1 || n_runs > FNB_MAX_ADAM_RUNS) return FNB_ERR_SIZE;
  AdamRunTable rt;
  for (int r = 0; r < n_runs; ++r) {
    const fnb_adam_run &x = runs[r];
    if ((x.first & 3) || (x.end & 3)) return FNB_ERR_ALIGN;
    if (x.first != (r ? runs[r - 1].end : 0) || x.end <= x.first || x.step < 1) return FNB_ERR_SIZE;
    rt.end4[r] = x.end >> 2;
    bias_corrections(lr, beta1, beta2, x.step, rt.step_size[r], rt.inv_sqrt_bc2[r]);
  }
  if (runs[n_runs - 1].end != n) return FNB_ERR_SIZE;
  for (int r = n_runs; r < FNB_MAX_ADAM_RUNS; ++r) {      // never read: the last run ends at n
    rt.end4[r] = INT64_MAX;
    rt.step_size[r] = rt.inv_sqrt_bc2[r] = 0.f;
  }
  k_allreduce_adam_runs<<<blocks, 256, 0, (cudaStream_t)stream>>>(*peers, a, rt);
  FNB_CHECK_LAUNCH();
  return 0;
}
