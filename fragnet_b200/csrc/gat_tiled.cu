// Node-tiled fused GAT2 attention kernels (forward, destination-side backward, source-side backward) and the
// by-source attention sums.
//
// Reference math (fragnet/model/gat/gat2.py:146-169 bond graph, :196-224 atom graph, :250-272 fragment-connection
// graph, :286-316 fragment graph; SURVEY.md App. A):
//   z[e,h] = S_t[t_e,h] + S_e[e,h] + S_s[s_e,h],  l = LeakyReLU_0.2(z),  p = softmax over the edges of t_e,
//   out[t] = sum_e p[e,h] * h[s_e,h,:]          (index_select, cat, mul, sum, scatter_softmax, scatter_add upstream)
//
// Why tiles.  The first version ran one warp per destination node with the segment's edges spread over lanes;
// `ncu --set full` (profiles/r1b_ncu_full.md) showed it issue/latency bound: 73-80 registers (37 % occupancy), ~7 of
// 32 lanes busy in the logit phase, 40 shuffles + 8 expf per node on the short scoreboard, DRAM 6-17 % busy.  Here a
// CTA owns T_NPC consecutive destination nodes = ONE contiguous range of CSR slots, and each phase uses the natural
// parallel axis out of shared memory:
//   phase 1  one thread per edge slot      : col/row/S gathers + edge term -> logits              (coalesced, no idle lanes)
//   phase 2  one thread per (node, head)   : max, sum, normalise in shared memory                 (no shuffles)
//   phase 3  one warp per node             : 512-byte row gathers of h[s] weighted by p, 4 in flight per warp
// Nodes whose in-degree exceeds the tile capacity (fragment-connection graphs of large salts can reach hundreds;
// SURVEY.md fact 9) take a warp-serial path inside the same kernel, so any degree is handled.
// The tiny edge-embedding algebra (App. A.5), the inter-layer ReLU(Dropout(.)) (gat2.py:414-418), the output masks
// (gat2.py:173-176) and the consumer graph's edge term ride in the prologue/epilogue, and parameter-gradient partials
// are reduced by the last CTA to finish (common.cuh: cta_finish) -- no floating-point atomics, no extra launches.
#include "common.cuh"

namespace {

constexpr int T_NPC = 64;        // max destination (or source) nodes per tile; the launcher picks npc <= T_NPC
constexpr int T_THREADS = 256;
constexpr int T_WARPS = T_THREADS / 32;
constexpr int FWD_CAP = 1024;    // edge slots staged per sub-tile (forward)
constexpr int BWD_CAP = 768;     // edge slots staged per sub-tile (backward kernels stage two float4 per slot)
constexpr int kDeepDegree = 24;  // mean in-degree from which the DEEP instantiations pay

// Largest le in (lb, nn] whose slots fit `cap`; returns lb when node lb alone exceeds it (hub path).
__device__ __forceinline__ int subtile_end(const int *s_rowptr, int lb, int nn, int cap) {
  const int base = s_rowptr[lb];
  if (s_rowptr[nn] - base <= cap) return nn;
  int le = lb;
  while (le < nn && s_rowptr[le + 1] - base <= cap) ++le;
  return le;
}

// ================================================================================================
// Forward
struct FwdT {
  const int *rowptr, *col, *row, *eid;
  const float *h, *S, *edge_attr;          // edge_attr: slot-ordered attributes (AFFINE) or the [n_real,4] table
  const float *We, *be, *alpha_e;          // AFFINE: embedding weight [32,in], bias [32], alpha + off_e
  int alpha_e_stride;
  int n_real, n_nodes;
  float *out, *y, *p_saved;
  PostAct post;
  int mask_lo, mask_hi;
  const float *next_alpha;
  int next_stride;
  float *next_Se;
  int npc;
  int deep;       // mean in-degree >= kDeepDegree: the DEEP instantiation
};

template <int MODE>
__device__ __forceinline__ float4 edge_term_t(const FwdT &a, int slot, const float *coef) {
  float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
  if (MODE == FNB_EDGE_AFFINE1) {
    const float c = __ldg(a.edge_attr + slot);
    r.x = fmaf(c, coef[0], coef[4]);
    r.y = fmaf(c, coef[1], coef[5]);
    r.z = fmaf(c, coef[2], coef[6]);
    r.w = fmaf(c, coef[3], coef[7]);
  } else if (MODE == FNB_EDGE_AFFINE6) {
    const float2 *ap = reinterpret_cast<const float2 *>(a.edge_attr + (int64_t)slot * 6);
    const float2 a0 = __ldg(ap), a1 = __ldg(ap + 1), a2 = __ldg(ap + 2);
    const float v[6] = {a0.x, a0.y, a1.x, a1.y, a2.x, a2.y};
    float acc[4];
#pragma unroll
    for (int hh = 0; hh < 4; ++hh) {
      float s = coef[24 + hh];
#pragma unroll
      for (int k = 0; k < 6; ++k) s = fmaf(v[k], coef[hh * 6 + k], s);
      acc[hh] = s;
    }
    r = make_float4(acc[0], acc[1], acc[2], acc[3]);
  } else if (MODE == FNB_EDGE_TABLE) {
    const int e = __ldg(a.eid + slot);
    if (e < a.n_real) r = ldg4(a.edge_attr + (int64_t)e * 4);
  }
  return r;
}

template <int MODE>
__device__ __forceinline__ float4 edge_logit(const FwdT &a, int slot, int t, int s, const float *coef) {
  const float4 St = ldg4(a.S + (int64_t)t * 8);
  const float4 Ss = ldg4(a.S + (int64_t)s * 8 + 4);
  const float4 Se = edge_term_t<MODE>(a, slot, coef);
  return make_float4(leaky(St.x + Se.x + Ss.x), leaky(St.y + Se.y + Ss.y), leaky(St.z + Se.z + Ss.z),
                     leaky(St.w + Se.w + Ss.w));
}

// coef[h*in + k] = sum_j We[j,k] alpha_e[h,j];  coef[4*in + h] = sum_j be[j] alpha_e[h,j]   (App. A.5)
template <int IN>
__device__ __forceinline__ void edge_coef_prologue(const float *We, const float *be, const float *alpha_e, int stride,
                                                   float *coef) {
  const int o = threadIdx.x;
  if (o >= 4 * IN + 4) return;
  float s = 0.f;
  if (o < 4 * IN) {
    const int hh = o / IN, k = o % IN;
    for (int j = 0; j < kHd; ++j) s = fmaf(__ldg(We + j * IN + k), __ldg(alpha_e + hh * stride + j), s);
  } else {
    const int hh = o - 4 * IN;
    for (int j = 0; j < kHd; ++j) s = fmaf(__ldg(be + j), __ldg(alpha_e + hh * stride + j), s);
  }
  coef[o] = s;
}

// Row epilogue shared by the tile and hub paths: mask, pre-/post-activation stores, consumer edge term.
__device__ __forceinline__ void fwd_store_row(const FwdT &a, int t, float4 acc, const float *s_na) {
  const int lane = threadIdx.x & 31;
  if (t >= a.mask_lo && t < a.mask_hi) acc = make_float4(0.f, 0.f, 0.f, 0.f);
  if (a.out) st4(a.out + (int64_t)t * kD + lane * 4, acc);
  if (a.y) st4(a.y + (int64_t)t * kD + lane * 4, post_act(a.post, acc, (uint64_t)t * 32 + lane));
  if (a.next_alpha) {
    const float se = warp_sum4(dot4(acc, ld4(s_na + lane * 4)), dot4(acc, ld4(s_na + 128 + lane * 4)),
                               dot4(acc, ld4(s_na + 256 + lane * 4)), dot4(acc, ld4(s_na + 384 + lane * 4)));
    if ((lane & 7) == 0) a.next_Se[(int64_t)t * 4 + (lane >> 3)] = se;
  }
}

// In-degree above the tile capacity: warp 0 streams the segment three times (max, sum, aggregate).
template <int MODE>
__device__ void fwd_hub(const FwdT &a, int t, int beg, int end, const float *coef, const float *s_na) {
  const int lane = threadIdx.x & 31, head = lane >> 3;
  float m[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
  for (int base = beg; base < end; base += 32) {
    const int slot = base + lane;
    if (slot < end) {
      const float4 l = edge_logit<MODE>(a, slot, t, __ldg(a.col + slot), coef);
      m[0] = fmaxf(m[0], l.x); m[1] = fmaxf(m[1], l.y); m[2] = fmaxf(m[2], l.z); m[3] = fmaxf(m[3], l.w);
    }
  }
  float den[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int hh = 0; hh < 4; ++hh) m[hh] = warp_max(m[hh]);
  for (int base = beg; base < end; base += 32) {
    const int slot = base + lane;
    if (slot < end) {
      const float4 l = edge_logit<MODE>(a, slot, t, __ldg(a.col + slot), coef);
      den[0] += expf(l.x - m[0]); den[1] += expf(l.y - m[1]); den[2] += expf(l.z - m[2]); den[3] += expf(l.w - m[3]);
    }
  }
#pragma unroll
  for (int hh = 0; hh < 4; ++hh) den[hh] = warp_sum(den[hh]);
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int base = beg; base < end; base += 32) {
    const int slot = base + lane;
    const int cnt = min(32, end - base);
    int s = 0;
    float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
    if (slot < end) {
      s = __ldg(a.col + slot);
      const float4 l = edge_logit<MODE>(a, slot, t, s, coef);
      p = make_float4(expf(l.x - m[0]) / den[0], expf(l.y - m[1]) / den[1], expf(l.z - m[2]) / den[2],
                      expf(l.w - m[3]) / den[3]);
      if (a.p_saved)
        st4(a.p_saved + (int64_t)slot * 4, make_float4(l.x > 0.f ? p.x : -p.x, l.y > 0.f ? p.y : -p.y,
                                                      l.z > 0.f ? p.z : -p.z, l.w > 0.f ? p.w : -p.w));
    }
    for (int j = 0; j < cnt; ++j) {
      const int sj = __shfl_sync(kFull, s, j);
      const float4 pj = make_float4(__shfl_sync(kFull, p.x, j), __shfl_sync(kFull, p.y, j), __shfl_sync(kFull, p.z, j),
                                    __shfl_sync(kFull, p.w, j));
      const float w = pick(pj, head);
      const float4 v = ldg4(a.h + (int64_t)sj * kD + lane * 4);
      acc.x = fmaf(w, v.x, acc.x); acc.y = fmaf(w, v.y, acc.y); acc.z = fmaf(w, v.z, acc.z); acc.w = fmaf(w, v.w, acc.w);
    }
  }
  fwd_store_row(a, t, acc, s_na);
}

// DEEP: the instantiation for graphs with a high mean in-degree (fragment-connection graphs of multi-component salts,
// ~60 edges per node: profiles/r3o_ncu_full_stress.md): 8 row gathers in flight per warp instead of 4 (fewer
// latency round trips per node; 64 registers, 4 CTAs per SM) and a warp-parallel softmax phase (8 lanes per
// (node, head) with shuffle reductions instead of one thread walking the whole segment while 3/4 of the CTA waits).
// WIDE: the same code compiled for 5 CTAs per SM (48 registers, no spills) instead of 6 (40 registers, 12 bytes
// spilled).  Measured on the bond graph: batch 1 024 (843 tiles = one wave at 6 per SM) 38.6 us at 6 per SM vs 43.5 us
// at 5; batch 4 096 (3 359 tiles) 127.6 us vs 119.7 us -- so graphs with more tiles than one 6-per-SM wave take WIDE.
template <int MODE, bool DEEP = false, bool WIDE = false>
__global__ void __launch_bounds__(T_THREADS, DEEP ? 4 : (WIDE ? 5 : 6)) k_gat_fwd_tiled(FwdT a) {
  __shared__ int s_rowptr[T_NPC + 1];
  constexpr int CAP = DEEP ? 2 * FWD_CAP : FWD_CAP;   // DEEP: longer sub-tiles, fewer phase barriers per node
  __shared__ int s_src[CAP];
  __shared__ __align__(16) float s_l[CAP * 4];
  __shared__ float s_coef[28];
  __shared__ __align__(16) float s_na[4 * kD];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, head = lane >> 3;
  pdl_wait();
  if (MODE == FNB_EDGE_AFFINE1) edge_coef_prologue<1>(a.We, a.be, a.alpha_e, a.alpha_e_stride, s_coef);
  if (MODE == FNB_EDGE_AFFINE6) edge_coef_prologue<6>(a.We, a.be, a.alpha_e, a.alpha_e_stride, s_coef);
  if (a.next_alpha)  // consumer graph's edge slice, 4 heads x 128 columns
    for (int i = tid; i < 4 * kD; i += T_THREADS) s_na[i] = __ldg(a.next_alpha + (int64_t)(i >> 7) * a.next_stride + (i & 127));

  const int n_tiles = (a.n_nodes + a.npc - 1) / a.npc;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int n0 = tile * a.npc, nn = min(a.npc, a.n_nodes - n0);
    __syncthreads();  // readers of the previous tile are done; also publishes s_coef
    if (tid <= nn) s_rowptr[tid] = __ldg(a.rowptr + n0 + tid);
    __syncthreads();
    int lb = 0;
    while (lb < nn) {
      const int le = subtile_end(s_rowptr, lb, nn, CAP);
      if (le == lb) {  // hub node (CTA-uniform branch)
        if (warp == 0) fwd_hub<MODE>(a, n0 + lb, s_rowptr[lb], s_rowptr[lb + 1], s_coef, s_na);
        ++lb;
        continue;
      }
      const int e0 = s_rowptr[lb], cnt = s_rowptr[le] - e0;
      // ---- phase 1: logits, one thread per slot
      for (int i = tid; i < cnt; i += T_THREADS) {
        const int slot = e0 + i;
        const int s = __ldg(a.col + slot), t = __ldg(a.row + slot);
        st4(s_l + i * 4, edge_logit<MODE>(a, slot, t, s, s_coef));
        s_src[i] = s;
      }
      __syncthreads();
      // ---- phase 2: softmax per (node, head)
      if (DEEP) {   // one warp per node, 8 lanes per head, edges strided over the 8 lanes
        const int sub = lane & 7;
        for (int n = lb + warp; n < le; n += T_WARPS) {
          const int b = s_rowptr[n] - e0, e = s_rowptr[n + 1] - e0;
          float m = -INFINITY;
          for (int j = b + sub; j < e; j += 8) m = fmaxf(m, s_l[j * 4 + head]);
          m = fmaxf(m, __shfl_xor_sync(kFull, m, 1));
          m = fmaxf(m, __shfl_xor_sync(kFull, m, 2));
          m = fmaxf(m, __shfl_xor_sync(kFull, m, 4));
          float den = 0.f;
          for (int j = b + sub; j < e; j += 8) {
            const float l = s_l[j * 4 + head];
            const float ex = expf(l - m);
            den += ex;
            s_l[j * 4 + head] = l > 0.f ? ex : -ex;
          }
          den = head_sum(den);
          const float inv = 1.f / den;
          for (int j = b + sub; j < e; j += 8) s_l[j * 4 + head] *= inv;
        }
      } else {
      for (int q = tid; q < (le - lb) * 4; q += T_THREADS) {
        const int n = lb + (q >> 2), hh = q & 3;
        const int b = s_rowptr[n] - e0, e = s_rowptr[n + 1] - e0;
        float m = -INFINITY;
        for (int j = b; j < e; ++j) m = fmaxf(m, s_l[j * 4 + hh]);
        float den = 0.f;
        for (int j = b; j < e; ++j) {   // one exp per edge; the sign bit keeps (z > 0) for LeakyReLU's derivative
          const float l = s_l[j * 4 + hh];
          const float ex = expf(l - m);
          den += ex;
          s_l[j * 4 + hh] = l > 0.f ? ex : -ex;
        }
        const float inv = 1.f / den;
        for (int j = b; j < e; ++j) s_l[j * 4 + hh] *= inv;
      }
      }
      __syncthreads();
      // ---- phase 3: save p (coalesced), then one warp per node aggregates source rows
      if (a.p_saved)
        for (int i = tid; i < cnt; i += T_THREADS) st4(a.p_saved + (int64_t)(e0 + i) * 4, ld4(s_l + i * 4));
      for (int n = lb + warp; n < le; n += T_WARPS) {
        const int b = s_rowptr[n] - e0, e = s_rowptr[n + 1] - e0;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        int j = b;
        if (DEEP) {
          for (; j + 8 <= e; j += 8) {
            float4 v[8];
            float pj[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
              v[u] = ldg4(a.h + (int64_t)s_src[j + u] * kD + lane * 4);
              pj[u] = fabsf(s_l[(j + u) * 4 + head]);
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
              acc.x = fmaf(pj[u], v[u].x, acc.x);
              acc.y = fmaf(pj[u], v[u].y, acc.y);
              acc.z = fmaf(pj[u], v[u].z, acc.z);
              acc.w = fmaf(pj[u], v[u].w, acc.w);
            }
          }
        }
        for (; j + 4 <= e; j += 4) {
          float4 v[4];
          float pj[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            v[u] = ldg4(a.h + (int64_t)s_src[j + u] * kD + lane * 4);
            pj[u] = fabsf(s_l[(j + u) * 4 + head]);
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            acc.x = fmaf(pj[u], v[u].x, acc.x);
            acc.y = fmaf(pj[u], v[u].y, acc.y);
            acc.z = fmaf(pj[u], v[u].z, acc.z);
            acc.w = fmaf(pj[u], v[u].w, acc.w);
          }
        }
        for (; j < e; ++j) {
          const float4 v = ldg4(a.h + (int64_t)s_src[j] * kD + lane * 4);
          const float pj = fabsf(s_l[j * 4 + head]);
          acc.x = fmaf(pj, v.x, acc.x);
          acc.y = fmaf(pj, v.y, acc.y);
          acc.z = fmaf(pj, v.z, acc.z);
          acc.w = fmaf(pj, v.w, acc.w);
        }
        fwd_store_row(a, n0 + n, acc, s_na);
      }
      lb = le;
      if (lb < nn) __syncthreads();  // next sub-tile overwrites the staging arrays
    }
  }
  pdl_launch_dependents();
}

// ================================================================================================
// Backward, destination side: dz[slot,h], dSt[t,h], gradients of the affine edge-term constants.
//   dp[e,h] = <g[t_e,h,:], h[s_e,h,:]>,  dl = p (dp - sum_seg p dp),  dz = dl * (z > 0 ? 1 : 0.2)
struct DstT {
  const int *rowptr, *col;
  const float *h, *dout, *p_saved, *edge_attr;
  float *dz, *dSt;
  int n_nodes;
  float *scratch;
  const float *We, *be, *alpha_e;
  int alpha_e_stride;
  float *dWe, *dbe, *d_alpha_e;
  int npc;
  // FUSE: the incoming gradient is assembled here instead of by a separate pass over the rows (see dst_grad_row)
  const float *f_dz;       // [E_up,4] dz of the consumer graph whose edge e is this graph's node e, or NULL
  const int *f_slot;       // consumer graph's slot_of_eid
  const float *f_alpha;    // consumer head vector, edge slice: [4, f_stride] (128 columns used)
  int f_stride;
  const float *f_base, *f_dy, *f_y;
  float f_scale;
  const float *f_pool;     // [n_seg,128] gradient of the pooled rows (atom -> fragment sum pooling), or NULL
  const int *f_seg;        // [N] segment of every row
  float *g_out;            // [N,128] assembled gradient, read by the source pass
};

template <int MODE> struct CoefT { static constexpr int NC = 1, PARTS = 1, IN = 1; };
template <> struct CoefT<FNB_EDGE_AFFINE1> { static constexpr int NC = 8, PARTS = 32, IN = 1; };
template <> struct CoefT<FNB_EDGE_AFFINE6> { static constexpr int NC = 28, PARTS = 9, IN = 6; };

__device__ __forceinline__ float dz_of(float p, float dp, float delta) {
  return fabsf(p) * (dp - delta) * (signbit(p) ? kNegSlope : 1.f);
}

// Gradient arriving at row t of this graph's output.  FUSE: the row is assembled on the fly,
//   g[t,:] = sum_h dz_up[slot_up[t],h] alpha_up[h,:]  (+ g_base[t,:])  (+ dy[t,:] (y[t,:] > 0) scale)  (+ pool[seg[t],:])
// i.e. the edge-term backward of the consumer graph (gat2.py:203-208: this graph's output rows are the consumer's edge
// vectors) plus the ReLU(Dropout) backward of gat2.py:414-418, in the summation order of k_edge_table_bwd_tiled, and
// written once for the source pass -- a whole pass over [N,128] leaves the critical path of the backward.
template <bool FUSE>
__device__ __forceinline__ float4 dst_grad_row(const DstT &a, int t, const float *s_ae) {
  const int lane = threadIdx.x & 31;
  const int64_t o = (int64_t)t * kD + lane * 4;
  if (!FUSE) return ldg4(a.dout + o);
  float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
  if (a.f_dz) {
    const float4 dz = ldg4(a.f_dz + (int64_t)__ldg(a.f_slot + t) * 4);
    const float4 ae0 = ld4(s_ae + lane * 4), ae1 = ld4(s_ae + 128 + lane * 4), ae2 = ld4(s_ae + 256 + lane * 4),
                 ae3 = ld4(s_ae + 384 + lane * 4);
    g.x = dz.x * ae0.x + dz.y * ae1.x + dz.z * ae2.x + dz.w * ae3.x;
    g.y = dz.x * ae0.y + dz.y * ae1.y + dz.z * ae2.y + dz.w * ae3.y;
    g.z = dz.x * ae0.z + dz.y * ae1.z + dz.z * ae2.z + dz.w * ae3.z;
    g.w = dz.x * ae0.w + dz.y * ae1.w + dz.z * ae2.w + dz.w * ae3.w;
  }
  if (a.f_base) {
    const float4 b = ldg4(a.f_base + o);
    g.x += b.x; g.y += b.y; g.z += b.z; g.w += b.w;
  }
  if (a.f_dy) {
    const float4 d = ldg4(a.f_dy + o);
    if (a.f_y) {
      const float4 y = ldg4(a.f_y + o);
      g.x += y.x > 0.f ? d.x * a.f_scale : 0.f;
      g.y += y.y > 0.f ? d.y * a.f_scale : 0.f;
      g.z += y.z > 0.f ? d.z * a.f_scale : 0.f;
      g.w += y.w > 0.f ? d.w * a.f_scale : 0.f;
    } else {
      g.x += d.x; g.y += d.y; g.z += d.z; g.w += d.w;
    }
  }
  if (a.f_pool) {   // pooling backward (gat2.py:234): every member row receives its fragment's gradient
    const float4 q = ldg4(a.f_pool + (int64_t)__ldg(a.f_seg + t) * kD + lane * 4);
    g.x += q.x; g.y += q.y; g.z += q.z; g.w += q.w;
  }
  st4(a.g_out + o, g);
  return g;
}

// Hub node on the destination side: warp 0, edges one at a time (dp parked in dz between the two passes).
__device__ void dst_hub(const DstT &a, int t, int beg, int end, const float4 g) {
  const int lane = threadIdx.x & 31, head = lane >> 3;
  float delta = 0.f;  // this lane's head
  for (int slot = beg; slot < end; ++slot) {
    const float4 v = ldg4(a.h + (int64_t)__ldg(a.col + slot) * kD + lane * 4);
    const float d = head_sum(dot4(g, v));
    const float p = __ldg(a.p_saved + (int64_t)slot * 4 + head);
    delta = fmaf(fabsf(p), d, delta);
    if ((lane & 7) == 0) a.dz[(int64_t)slot * 4 + head] = d;
  }
  __syncwarp();
  float dst = 0.f;
  if ((lane & 7) == 0) {
    for (int slot = beg; slot < end; ++slot) {
      const float p = __ldg(a.p_saved + (int64_t)slot * 4 + head);
      const float v = dz_of(p, a.dz[(int64_t)slot * 4 + head], delta);
      a.dz[(int64_t)slot * 4 + head] = v;
      dst += v;
    }
    a.dSt[(int64_t)t * 4 + head] = dst;
  }
}

// DEEP (mean in-degree >= 24): only the softmax-backward phase changes (one warp per node, 8 lanes per head) -- with
// ~60 edges per node a thread per (node, head) leaves 3/4 of the CTA waiting at the barrier.  Deeper gathers at lower
// occupancy were measured slower here (the per-edge dot + head reduction keeps the warps busy).
template <int MODE, bool FUSE, bool DEEP = false>
__global__ void __launch_bounds__(T_THREADS, 6) k_gat_bwd_dst_tiled(DstT a) {
  constexpr int NC = CoefT<MODE>::NC, PARTS = CoefT<MODE>::PARTS, IN = CoefT<MODE>::IN;
  __shared__ int s_rowptr[T_NPC + 1];
  __shared__ int s_src[BWD_CAP];
  __shared__ __align__(16) float s_p[BWD_CAP * 4];
  __shared__ __align__(16) float s_dp[BWD_CAP * 4];
  __shared__ float s_red[PARTS * NC];
  __shared__ float s_rec[32], s_fin[32];
  __shared__ __align__(16) float s_ae[FUSE ? 4 * kD : 4];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, head = lane >> 3;
  // coefficient-gradient lane: coefficient c, slots part, part + PARTS, ...
  const bool coef_thread = NC > 1 && tid < NC * PARTS;
  const int c = tid % NC, part = tid / NC;
  const int c_head = (NC == 8) ? (c & 3) : (c < 24 ? c / 6 : c - 24);
  const int c_k = (NC == 8) ? (c < 4 ? 0 : -1) : (c < 24 ? c % 6 : -1);  // -1: bias term (attribute = 1)
  float cacc = 0.f;
  if (FUSE && a.f_dz)   // parameters, not produced by the preceding launch: staged before the dependency wait
    for (int i = tid; i < 4 * kD; i += T_THREADS) s_ae[i] = __ldg(a.f_alpha + (int64_t)(i >> 7) * a.f_stride + (i & 127));
  pdl_wait();

  const int n_tiles = (a.n_nodes + a.npc - 1) / a.npc;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int n0 = tile * a.npc, nn = min(a.npc, a.n_nodes - n0);
    __syncthreads();
    if (tid <= nn) s_rowptr[tid] = __ldg(a.rowptr + n0 + tid);
    __syncthreads();
    int lb = 0;
    while (lb < nn) {
      const int le = subtile_end(s_rowptr, lb, nn, BWD_CAP);
      if (le == lb) {
        const int beg = s_rowptr[lb], end = s_rowptr[lb + 1];
        if (warp == 0) dst_hub(a, n0 + lb, beg, end, dst_grad_row<FUSE>(a, n0 + lb, s_ae));
        if (NC > 1) {
          __syncthreads();  // warp 0's dz is visible to the block
          if (coef_thread)
            for (int slot = beg + part; slot < end; slot += PARTS) {
              const float x = c_k < 0 ? 1.f : __ldg(a.edge_attr + (int64_t)slot * IN + c_k);
              cacc = fmaf(a.dz[(int64_t)slot * 4 + c_head], x, cacc);
            }
        }
        ++lb;
        continue;
      }
      const int e0 = s_rowptr[lb], cnt = s_rowptr[le] - e0;
      // ---- phase A0: stage sources and probabilities (coalesced)
      for (int i = tid; i < cnt; i += T_THREADS) {
        s_src[i] = __ldg(a.col + e0 + i);
        st4(s_p + i * 4, ldg4(a.p_saved + (int64_t)(e0 + i) * 4));
      }
      __syncthreads();
      // ---- phase A: dp per edge, one warp per node
      for (int n = lb + warp; n < le; n += T_WARPS) {
        const int b = s_rowptr[n] - e0, e = s_rowptr[n + 1] - e0;
        const float4 g = dst_grad_row<FUSE>(a, n0 + n, s_ae);
        int j = b;
        for (; j + 4 <= e; j += 4) {
          float4 v[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) v[u] = ldg4(a.h + (int64_t)s_src[j + u] * kD + lane * 4);
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const float d = head_sum(dot4(g, v[u]));
            if ((lane & 7) == 0) s_dp[(j + u) * 4 + head] = d;
          }
        }
        for (; j < e; ++j) {
          const float4 v = ldg4(a.h + (int64_t)s_src[j] * kD + lane * 4);
          const float d = head_sum(dot4(g, v));
          if ((lane & 7) == 0) s_dp[j * 4 + head] = d;
        }
      }
      __syncthreads();
      // ---- phase B: softmax backward per (node, head)
      if (DEEP) {
        const int sub = lane & 7;
        for (int n = lb + warp; n < le; n += T_WARPS) {
          const int b = s_rowptr[n] - e0, e = s_rowptr[n + 1] - e0;
          float delta = 0.f;
          for (int j = b + sub; j < e; j += 8) delta = fmaf(fabsf(s_p[j * 4 + head]), s_dp[j * 4 + head], delta);
          delta = head_sum(delta);
          float dst = 0.f;
          for (int j = b + sub; j < e; j += 8) {
            const float v = dz_of(s_p[j * 4 + head], s_dp[j * 4 + head], delta);
            s_dp[j * 4 + head] = v;
            dst += v;
          }
          dst = head_sum(dst);
          if (sub == 0) a.dSt[(int64_t)(n0 + n) * 4 + head] = dst;
        }
      } else
      for (int q = tid; q < (le - lb) * 4; q += T_THREADS) {
        const int n = lb + (q >> 2), hh = q & 3;
        const int b = s_rowptr[n] - e0, e = s_rowptr[n + 1] - e0;
        float delta = 0.f;
        for (int j = b; j < e; ++j) delta = fmaf(fabsf(s_p[j * 4 + hh]), s_dp[j * 4 + hh], delta);
        float dst = 0.f;
        for (int j = b; j < e; ++j) {
          const float v = dz_of(s_p[j * 4 + hh], s_dp[j * 4 + hh], delta);
          s_dp[j * 4 + hh] = v;
          dst += v;
        }
        a.dSt[(int64_t)(n0 + n) * 4 + hh] = dst;
      }
      __syncthreads();
      // ---- phase C: dz out (coalesced) and the edge-term constants
      for (int i = tid; i < cnt; i += T_THREADS) st4(a.dz + (int64_t)(e0 + i) * 4, ld4(s_dp + i * 4));
      if (coef_thread)
        for (int i = part; i < cnt; i += PARTS) {
          const float x = c_k < 0 ? 1.f : __ldg(a.edge_attr + (int64_t)(e0 + i) * IN + c_k);
          cacc = fmaf(s_dp[i * 4 + c_head], x, cacc);
        }
      lb = le;
      if (lb < nn) __syncthreads();
    }
  }

  pdl_launch_dependents();
  if (NC > 1) {
    // CTA record of the coefficient gradients, then the cross-CTA tree; the finishing CTA turns d_coef into the
    // gradients of the embedding and of the edge slice of the head vector (App. A.5).
    __syncthreads();
    if (coef_thread) s_red[part * NC + c] = cacc;
    __syncthreads();
    if (tid < 32) {
      float s = 0.f;
      if (tid < NC)
        for (int k = 0; k < PARTS; ++k) s += s_red[k * NC + tid];
      s_rec[tid] = s;
    }
    __syncthreads();
    if (!cta_finish<32>(s_rec, s_fin, a.scratch)) return;
    const float *dcoef = s_fin;
    const int n_w = kHd * IN;
    for (int o = tid; o < n_w + kHd + kH * kHd; o += T_THREADS) {
      if (o < n_w) {  // dWe[j,k] = sum_h d_coef[h*in+k] alpha_e[h,j]
        const int j = o / IN, k = o % IN;
        float s = 0.f;
        for (int hh = 0; hh < kH; ++hh) s = fmaf(dcoef[hh * IN + k], a.alpha_e[hh * a.alpha_e_stride + j], s);
        a.dWe[o] = s;
      } else if (o < n_w + kHd) {  // dbe[j] = sum_h d_coef[4in+h] alpha_e[h,j]
        const int j = o - n_w;
        float s = 0.f;
        for (int hh = 0; hh < kH; ++hh) s = fmaf(dcoef[4 * IN + hh], a.alpha_e[hh * a.alpha_e_stride + j], s);
        a.dbe[j] = s;
      } else {  // d alpha_e[h,j] = sum_k d_coef[h*in+k] We[j,k] + d_coef[4in+h] be[j]
        const int r = o - n_w - kHd, hh = r / kHd, j = r % kHd;
        float s = dcoef[4 * IN + hh] * a.be[j];
        for (int k = 0; k < IN; ++k) s = fmaf(dcoef[hh * IN + k], a.We[j * IN + k], s);
        a.d_alpha_e[hh * a.alpha_e_stride + j] = s;
      }
    }
  }
}

// ================================================================================================
// Backward, source side (reverse CSR): dh[s] = sum_{e: s_e=s} p g[t_e] + dSt[s] alpha_t + dSs[s] alpha_s,
// dSs[s] = sum dz, d alpha_t = sum_n dSt[n,h] h[n,h,:], d alpha_s likewise, d_bias = column sums of dh.
struct SrcT {
  const int *rrowptr, *rslot, *rdst;
  const float *h, *dout, *p_saved, *dz, *dSt, *alpha;
  int alpha_stride, off_t, off_s;
  float *dh, *d_alpha, *d_bias;
  float *scratch;
  int n_nodes;
  int npc;
};

template <bool DEEP>
__global__ void __launch_bounds__(T_THREADS, DEEP ? 3 : 4) k_gat_bwd_src_tiled(SrcT a) {
  __shared__ int s_rowptr[T_NPC + 1];
  constexpr int CAP = DEEP ? 1024 : BWD_CAP;
  __shared__ int s_t[CAP];
  __shared__ __align__(16) float s_p[CAP * 4];   // reused as the 8 x 384 per-warp records at the end
  __shared__ __align__(16) float s_dz[CAP * 4];  // reused as CTA record [384] + final [384]
  __shared__ __align__(16) float s_dSs[T_NPC * 4];
  static_assert(BWD_CAP * 4 >= T_WARPS * 384, "per-warp records must fit the staging array");
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, head = lane >> 3;
  pdl_wait();
  const float4 at = ldg4(a.alpha + (int64_t)head * a.alpha_stride + a.off_t + (lane & 7) * 4);
  const float4 as = ldg4(a.alpha + (int64_t)head * a.alpha_stride + a.off_s + (lane & 7) * 4);
  float pa[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  float4 colsum = make_float4(0.f, 0.f, 0.f, 0.f);

  // (gt, hr: dSt and the node's own row, loaded by the caller BEFORE its gather loop so that their latency hides
  // under the gathers instead of adding a second round trip per node)
  auto finish_row = [&](int s, float4 acc, float gs, float gt, float4 hr) {
    acc.x += gt * at.x + gs * as.x;
    acc.y += gt * at.y + gs * as.y;
    acc.z += gt * at.z + gs * as.z;
    acc.w += gt * at.w + gs * as.w;
    st4(a.dh + (int64_t)s * kD + lane * 4, acc);
    colsum.x += acc.x; colsum.y += acc.y; colsum.z += acc.z; colsum.w += acc.w;
    pa[0] = fmaf(gt, hr.x, pa[0]); pa[1] = fmaf(gt, hr.y, pa[1]); pa[2] = fmaf(gt, hr.z, pa[2]); pa[3] = fmaf(gt, hr.w, pa[3]);
    pa[4] = fmaf(gs, hr.x, pa[4]); pa[5] = fmaf(gs, hr.y, pa[5]); pa[6] = fmaf(gs, hr.z, pa[6]); pa[7] = fmaf(gs, hr.w, pa[7]);
  };

  const int n_tiles = (a.n_nodes + a.npc - 1) / a.npc;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int n0 = tile * a.npc, nn = min(a.npc, a.n_nodes - n0);
    __syncthreads();
    if (tid <= nn) s_rowptr[tid] = __ldg(a.rrowptr + n0 + tid);
    __syncthreads();
    int lb = 0;
    while (lb < nn) {
      const int le = subtile_end(s_rowptr, lb, nn, CAP);
      if (le == lb) {  // hub source node: warp 0, reverse slots one at a time
        if (warp == 0) {
          const int beg = s_rowptr[lb], end = s_rowptr[lb + 1];
          float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
          float gs = 0.f;
          for (int r = beg; r < end; ++r) {
            const int slot = __ldg(a.rslot + r);
            const float p = fabsf(__ldg(a.p_saved + (int64_t)slot * 4 + head));
            gs += __ldg(a.dz + (int64_t)slot * 4 + head);
            const float4 v = ldg4(a.dout + (int64_t)__ldg(a.rdst + r) * kD + lane * 4);
            acc.x = fmaf(p, v.x, acc.x); acc.y = fmaf(p, v.y, acc.y); acc.z = fmaf(p, v.z, acc.z); acc.w = fmaf(p, v.w, acc.w);
          }
          finish_row(n0 + lb, acc, gs, __ldg(a.dSt + (int64_t)(n0 + lb) * 4 + head),
                     ldg4(a.h + (int64_t)(n0 + lb) * kD + lane * 4));
        }
        ++lb;
        continue;
      }
      const int r0 = s_rowptr[lb], cnt = s_rowptr[le] - r0;
      // ---- phase 1: stage p, dz (16-byte gathers through the reverse permutation) and destinations
      for (int i = tid; i < cnt; i += T_THREADS) {
        const int slot = __ldg(a.rslot + r0 + i);
        s_t[i] = __ldg(a.rdst + r0 + i);
        const float4 p = ldg4(a.p_saved + (int64_t)slot * 4);
        st4(s_p + i * 4, make_float4(fabsf(p.x), fabsf(p.y), fabsf(p.z), fabsf(p.w)));
        st4(s_dz + i * 4, ldg4(a.dz + (int64_t)slot * 4));
      }
      __syncthreads();
      // ---- phase 2: dSs per (node, head)
      if (DEEP) {
        const int sub = lane & 7;
        for (int n = lb + warp; n < le; n += T_WARPS) {
          const int b = s_rowptr[n] - r0, e = s_rowptr[n + 1] - r0;
          float sdz = 0.f;
          for (int j = b + sub; j < e; j += 8) sdz += s_dz[j * 4 + head];
          sdz = head_sum(sdz);
          if (sub == 0) s_dSs[(n - lb) * 4 + head] = sdz;
        }
      } else {
      for (int q = tid; q < (le - lb) * 4; q += T_THREADS) {
        const int n = lb + (q >> 2), hh = q & 3;
        const int b = s_rowptr[n] - r0, e = s_rowptr[n + 1] - r0;
        float s = 0.f;
        for (int j = b; j < e; ++j) s += s_dz[j * 4 + hh];
        s_dSs[(n - lb) * 4 + hh] = s;
      }
      }
      __syncthreads();
      // ---- phase 3: one warp per source node gathers the destination gradients
      for (int n = lb + warp; n < le; n += T_WARPS) {
        const int b = s_rowptr[n] - r0, e = s_rowptr[n + 1] - r0;
        const float gt = __ldg(a.dSt + (int64_t)(n0 + n) * 4 + head);
        const float4 hr = ldg4(a.h + (int64_t)(n0 + n) * kD + lane * 4);
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        int j = b;
        if (DEEP) {
          for (; j + 8 <= e; j += 8) {
            float4 v[8];
            float pj[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
              v[u] = ldg4(a.dout + (int64_t)s_t[j + u] * kD + lane * 4);
              pj[u] = s_p[(j + u) * 4 + head];
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
              acc.x = fmaf(pj[u], v[u].x, acc.x);
              acc.y = fmaf(pj[u], v[u].y, acc.y);
              acc.z = fmaf(pj[u], v[u].z, acc.z);
              acc.w = fmaf(pj[u], v[u].w, acc.w);
            }
          }
        }
        for (; j + 4 <= e; j += 4) {
          float4 v[4];
          float pj[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            v[u] = ldg4(a.dout + (int64_t)s_t[j + u] * kD + lane * 4);
            pj[u] = s_p[(j + u) * 4 + head];
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            acc.x = fmaf(pj[u], v[u].x, acc.x);
            acc.y = fmaf(pj[u], v[u].y, acc.y);
            acc.z = fmaf(pj[u], v[u].z, acc.z);
            acc.w = fmaf(pj[u], v[u].w, acc.w);
          }
        }
        for (; j < e; ++j) {
          const float4 v = ldg4(a.dout + (int64_t)s_t[j] * kD + lane * 4);
          const float pj = s_p[j * 4 + head];
          acc.x = fmaf(pj, v.x, acc.x);
          acc.y = fmaf(pj, v.y, acc.y);
          acc.z = fmaf(pj, v.z, acc.z);
          acc.w = fmaf(pj, v.w, acc.w);
        }
        finish_row(n0 + n, acc, s_dSs[(n - lb) * 4 + head], gt, hr);
      }
      lb = le;
      if (lb < nn) __syncthreads();
    }
  }

  // CTA record: [0,128) d alpha_t[4,32] (index head*32 + col = lane*4 + i), [128,256) d alpha_s, [256,384) colsum(dh)
  pdl_launch_dependents();
  __syncthreads();
  float *s_w = s_p;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    s_w[warp * 384 + lane * 4 + i] = pa[i];
    s_w[warp * 384 + 128 + lane * 4 + i] = pa[4 + i];
  }
  st4(s_w + warp * 384 + 256 + lane * 4, colsum);
  __syncthreads();
  float *s_rec = s_dz, *s_fin = s_dz + 384;
  for (int j = tid; j < 384; j += T_THREADS) {
    float sum = 0.f;
#pragma unroll
    for (int w = 0; w < T_WARPS; ++w) sum += s_w[w * 384 + j];
    s_rec[j] = sum;
  }
  __syncthreads();
  if (!cta_finish<384>(s_rec, s_fin, a.scratch)) return;
  for (int j = tid; j < 384; j += T_THREADS) {
    const float v = s_fin[j];
    if (j < 128) a.d_alpha[(j >> 5) * a.alpha_stride + a.off_t + (j & 31)] = v;
    else if (j < 256) a.d_alpha[((j - 128) >> 5) * a.alpha_stride + a.off_s + (j & 31)] = v;
    else if (a.d_bias) a.d_bias[j - 256] = v;
  }
}

// ================================================================================================
// Edge-term backward for TABLE mode (atom graph <- bond features, fragment graph <- fragment-connection features):
//   g_feat[e,:] = g_in[e,:] + sum_h dz[slot_of_eid[e],h] alpha_e[h,:],   d alpha_e[h,:] = sum_e dz[e,h] feat[e,:]
// where g_in is either a plain gradient (g_base) or the ReLU(Dropout) backward of the gradient that arrived at the
// post-activation copy of feat:  g_in = dy * (y > 0) * scale   (gat2.py:414-418), fused here to save a pass.
struct TableT {
  const float *dz;
  const int *slot_of_eid;
  const float *feat, *alpha;
  int alpha_stride, off_e;
  const float *g_base, *dy, *y;
  float scale;
  float *g_feat, *d_alpha;
  float *scratch;
  int n_real;
};

__global__ void __launch_bounds__(T_THREADS, 5) k_edge_table_bwd_tiled(TableT a) {
  __shared__ __align__(16) float s_w[T_WARPS * 512];
  __shared__ __align__(16) float s_rec[512];
  __shared__ __align__(16) float s_fin[512];
  __shared__ __align__(16) float s_ae[4 * kD];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  pdl_wait();
  for (int i = threadIdx.x; i < 4 * kD; i += T_THREADS)
    s_ae[i] = __ldg(a.alpha + (int64_t)(i >> 7) * a.alpha_stride + a.off_e + (i & 127));
  __syncthreads();
  float4 acc[4];
#pragma unroll
  for (int hh = 0; hh < 4; ++hh) acc[hh] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int e = blockIdx.x * T_WARPS + warp; e < a.n_real; e += gridDim.x * T_WARPS) {
    const float4 dz = ldg4(a.dz + (int64_t)__ldg(a.slot_of_eid + e) * 4);
    const float4 f = ldg4(a.feat + (int64_t)e * kD + lane * 4);
    const float4 ae0 = ld4(s_ae + lane * 4), ae1 = ld4(s_ae + 128 + lane * 4), ae2 = ld4(s_ae + 256 + lane * 4),
                 ae3 = ld4(s_ae + 384 + lane * 4);
    if (a.g_feat) {   // NULL: only the head-vector gradient (the row gradient is assembled by the consumer's destination pass)
      float4 g;
      g.x = dz.x * ae0.x + dz.y * ae1.x + dz.z * ae2.x + dz.w * ae3.x;
      g.y = dz.x * ae0.y + dz.y * ae1.y + dz.z * ae2.y + dz.w * ae3.y;
      g.z = dz.x * ae0.z + dz.y * ae1.z + dz.z * ae2.z + dz.w * ae3.z;
      g.w = dz.x * ae0.w + dz.y * ae1.w + dz.z * ae2.w + dz.w * ae3.w;
      if (a.g_base) {
        const float4 o = ld4(a.g_base + (int64_t)e * kD + lane * 4);
        g.x += o.x; g.y += o.y; g.z += o.z; g.w += o.w;
      }
      if (a.dy) {
        const float4 d = ldg4(a.dy + (int64_t)e * kD + lane * 4), o = ldg4(a.y + (int64_t)e * kD + lane * 4);
        g.x += o.x > 0.f ? d.x * a.scale : 0.f;
        g.y += o.y > 0.f ? d.y * a.scale : 0.f;
        g.z += o.z > 0.f ? d.z * a.scale : 0.f;
        g.w += o.w > 0.f ? d.w * a.scale : 0.f;
      }
      st4(a.g_feat + (int64_t)e * kD + lane * 4, g);
    }
    const float d4[4] = {dz.x, dz.y, dz.z, dz.w};
#pragma unroll
    for (int hh = 0; hh < 4; ++hh) {
      acc[hh].x = fmaf(d4[hh], f.x, acc[hh].x);
      acc[hh].y = fmaf(d4[hh], f.y, acc[hh].y);
      acc[hh].z = fmaf(d4[hh], f.z, acc[hh].z);
      acc[hh].w = fmaf(d4[hh], f.w, acc[hh].w);
    }
  }
  pdl_launch_dependents();
#pragma unroll
  for (int hh = 0; hh < 4; ++hh) st4(s_w + warp * 512 + hh * 128 + lane * 4, acc[hh]);
  __syncthreads();
  for (int j = threadIdx.x; j < 512; j += T_THREADS) {
    float sum = 0.f;
#pragma unroll
    for (int w = 0; w < T_WARPS; ++w) sum += s_w[w * 512 + j];
    s_rec[j] = sum;
  }
  __syncthreads();
  if (!cta_finish<512>(s_rec, s_fin, a.scratch)) return;
  for (int j = threadIdx.x; j < 512; j += T_THREADS) a.d_alpha[(j >> 7) * a.alpha_stride + a.off_e + (j & 127)] = s_fin[j];
}

// Nodes per tile: 64 when that still yields >= 2 tiles per SM, otherwise halve (down to 8 = one node per warp) so that
// small graphs (fragment / fragment-connection graphs have 5-10x fewer nodes than the bond graph) fill the machine
// (measured sweep: profiles/r1f_kbench_npc*.log).
inline int pick_npc(int64_t n_nodes) {
  for (int npc = T_NPC; npc > 8; npc >>= 1)
    if ((n_nodes + npc - 1) / npc >= (int64_t)kNumSMs * 2) return npc;
  return 8;
}

inline int tile_grid(int64_t n_nodes, int npc, int ctas_per_sm) {
  int64_t tiles = (n_nodes + npc - 1) / npc;
  const int64_t cap = (int64_t)kNumSMs * ctas_per_sm;
  if (tiles > cap) tiles = cap;
  if (tiles < 1) tiles = 1;
  return (int)tiles;
}

// The cross-CTA reductions (cta_finish) keep one record per CTA in the caller's scratch.  Largest grids: the
// destination pass (32-float record) and the source pass (384) tile_grid(., ., <= 6), the edge-table backward (512)
// kNumSMs * 4.
static_assert(kScratchFloats >= finish_scratch_floats(32, kNumSMs * 6), "scratch must hold the destination-pass records");
static_assert(kScratchFloats >= finish_scratch_floats(384, kNumSMs * 6), "scratch must hold the source-pass records");
static_assert(kScratchFloats >= finish_scratch_floats(512, kNumSMs * 4), "scratch must hold the edge-table records");

template <int MODE>
int launch_fwd(const FwdT &a, cudaStream_t stream) {
  if (a.deep) {
    const cudaError_t le = fnb_launch(k_gat_fwd_tiled<MODE, true>, dim3(tile_grid(a.n_nodes, a.npc, 4)), dim3(T_THREADS), 0, stream, a);
    if (le != cudaSuccess) return (int)le;
  } else if (((int64_t)a.n_nodes + a.npc - 1) / a.npc > (int64_t)kNumSMs * 6) {
    const cudaError_t le = fnb_launch(k_gat_fwd_tiled<MODE, false, true>, dim3(tile_grid(a.n_nodes, a.npc, 5)), dim3(T_THREADS), 0, stream, a);
    if (le != cudaSuccess) return (int)le;
  } else {
    const cudaError_t le = fnb_launch(k_gat_fwd_tiled<MODE>, dim3(tile_grid(a.n_nodes, a.npc, 6)), dim3(T_THREADS), 0, stream, a);
    if (le != cudaSuccess) return (int)le;
  }
  FNB_CHECK_LAUNCH();
  return 0;
}

inline bool deep_graph(const fnb_graph *g) {
  return g->n_nodes > 0 && g->n_edges >= (int64_t)kDeepDegree * g->n_nodes;
}

inline bool graph_ok(const fnb_graph *g) {
  return g && g->n_nodes >= 0 && g->n_edges >= 0 && g->n_nodes < INT32_MAX && g->n_edges < INT32_MAX;
}

// w[n,:] = sum of |p| over the reverse-CSR slots of source n.
__global__ void k_attn_by_source(const int *__restrict__ rrowptr, const int *__restrict__ rslot,
                                 const float *__restrict__ p_saved, int64_t n_nodes, float *__restrict__ w) {
  for (int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; n < n_nodes; n += (int64_t)gridDim.x * blockDim.x) {
    const int beg = rrowptr[n], end = rrowptr[n + 1];
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int r = beg; r < end; ++r) {
      const float4 p = ldg4(p_saved + (int64_t)rslot[r] * 4);
      acc.x += fabsf(p.x);
      acc.y += fabsf(p.y);
      acc.z += fabsf(p.z);
      acc.w += fabsf(p.w);
    }
    st4(w + n * 4, acc);
  }
}

}  // namespace

extern "C" int fnb_gat_fwd_tiled(const fnb_graph *g, const fnb_gat_fwd_args *f, void *stream_) {
  if (!graph_ok(g) || !f) return g && f ? FNB_ERR_SIZE : FNB_ERR_NULL;
  if (g->n_nodes == 0) return 0;
  if (!g->rowptr || !f->h || !f->S || (!f->out && !f->y) || (g->n_edges > 0 && (!g->col || !g->row)))
    return FNB_ERR_NULL;
  if (!fnb_aligned16(f->h) || !fnb_aligned16(f->S) || !fnb_aligned16(f->out) || !fnb_aligned16(f->y) ||
      !fnb_aligned16(f->p_saved))
    return FNB_ERR_ALIGN;
  if (f->next_alpha_e && (!f->next_Se || (f->next_alpha_stride & 3) || !fnb_aligned16(f->next_alpha_e)))
    return FNB_ERR_ALIGN;
  if (f->y && !(f->post.p >= 0.f && f->post.p < 1.f)) return FNB_ERR_SIZE;
  FwdT a;
  a.rowptr = g->rowptr; a.col = g->col; a.row = g->row; a.eid = g->eid;
  a.h = f->h; a.S = f->S; a.edge_attr = nullptr; a.We = f->We; a.be = f->be; a.alpha_e = f->alpha_e;
  a.alpha_e_stride = f->alpha_stride; a.n_real = (int)g->n_real_edges; a.n_nodes = (int)g->n_nodes;
  a.out = f->out; a.y = f->y; a.p_saved = f->p_saved;
  a.post.p = f->post.p; a.post.scale = 1.f / (1.f - f->post.p); a.post.training = f->post.training;
  a.post.relu = f->post.relu; a.post.seed = f->post.seed; a.post.offset = f->post.offset;
  a.mask_lo = (int)f->mask_lo; a.mask_hi = (int)f->mask_hi;
  a.next_alpha = f->next_alpha_e; a.next_stride = f->next_alpha_stride; a.next_Se = f->next_Se;
  a.npc = pick_npc(g->n_nodes);
  a.deep = deep_graph(g) ? 1 : 0;
  cudaStream_t stream = (cudaStream_t)stream_;
  // slot-ordered inputs are read only at slots: a graph without edges (or, for the table, without real edges) may
  // pass NULL for them, as empty buffers are
  const bool slots = g->n_edges > 0;
  switch (f->edge_mode) {
    case FNB_EDGE_NONE:
      return launch_fwd<FNB_EDGE_NONE>(a, stream);
    case FNB_EDGE_AFFINE1:
      if ((slots && !g->edge_attr) || !f->We || !f->be || !f->alpha_e) return FNB_ERR_NULL;
      a.edge_attr = g->edge_attr;
      return launch_fwd<FNB_EDGE_AFFINE1>(a, stream);
    case FNB_EDGE_AFFINE6:
      if ((slots && !g->edge_attr) || !f->We || !f->be || !f->alpha_e) return FNB_ERR_NULL;
      if (reinterpret_cast<uintptr_t>(g->edge_attr) & 7u) return FNB_ERR_ALIGN;
      a.edge_attr = g->edge_attr;
      return launch_fwd<FNB_EDGE_AFFINE6>(a, stream);
    case FNB_EDGE_TABLE:
      if ((g->n_real_edges > 0 && !f->edge_table) || (slots && !g->eid)) return FNB_ERR_NULL;
      if (!fnb_aligned16(f->edge_table)) return FNB_ERR_ALIGN;
      a.edge_attr = f->edge_table;
      return launch_fwd<FNB_EDGE_TABLE>(a, stream);
    default:
      return FNB_ERR_MODE;
  }
}

extern "C" int fnb_gat_bwd_tiled(const fnb_graph *g, const fnb_gat_bwd_args *b, void *stream_) {
  return fnb_gat_bwd_tiled_fused(g, b, nullptr, nullptr, nullptr, stream_);
}

extern "C" int fnb_gat_bwd_tiled_marked(const fnb_graph *g, const fnb_gat_bwd_args *b, void *between_passes, void *stream_) {
  return fnb_gat_bwd_tiled_fused(g, b, nullptr, (cudaEvent_t)between_passes, nullptr, stream_);
}

int fnb_gat_bwd_tiled_fused(const fnb_graph *g, const fnb_gat_bwd_args *b, const FnbDstFuse *fz, cudaEvent_t after_dst,
                            cudaEvent_t before_src, void *stream_) {
  if (!graph_ok(g) || !b) return g && b ? FNB_ERR_SIZE : FNB_ERR_NULL;
  if (g->n_nodes == 0) return 0;
  if (!g->rowptr || !g->rrowptr || !b->h || !b->dout || !b->dSt || !b->dh || !b->alpha || !b->d_alpha || !b->scratch ||
      (g->n_edges > 0 && (!g->col || !g->rslot || !g->rdst || !b->p_saved || !b->dz)))
    return FNB_ERR_NULL;
  if (fz) {
    if ((fz->dz_up && (!fz->slot_of_eid || !fz->alpha_up)) || (fz->y && !fz->dy) || (fz->pool && !fz->seg_of))
      return FNB_ERR_NULL;
    if ((fz->alpha_up_stride & 3) || !fnb_aligned16(fz->alpha_up) || !fnb_aligned16(fz->dz_up) ||
        !fnb_aligned16(fz->g_base) || !fnb_aligned16(fz->dy) || !fnb_aligned16(fz->y) || !fnb_aligned16(fz->pool))
      return FNB_ERR_ALIGN;
  }
  if ((b->alpha_stride & 3) || (b->off_t & 3) || (b->off_s & 3) || (b->off_e & 3) || !fnb_aligned16(b->alpha) ||
      !fnb_aligned16(b->h) || !fnb_aligned16(b->dout) || !fnb_aligned16(b->dh) || !fnb_aligned16(b->dz) ||
      !fnb_aligned16(b->p_saved) || !fnb_aligned16(b->dSt) || !fnb_aligned16(b->scratch))
    return FNB_ERR_ALIGN;
  cudaStream_t stream = (cudaStream_t)stream_;
  DstT d;
  d.rowptr = g->rowptr; d.col = g->col; d.h = b->h; d.dout = b->dout; d.p_saved = b->p_saved;
  d.edge_attr = g->edge_attr; d.dz = b->dz; d.dSt = b->dSt; d.n_nodes = (int)g->n_nodes; d.scratch = (float *)b->scratch;
  d.We = b->We; d.be = b->be; d.alpha_e = b->alpha + b->off_e; d.alpha_e_stride = b->alpha_stride;
  d.dWe = b->dWe; d.dbe = b->dbe; d.d_alpha_e = b->d_alpha + b->off_e;
  d.npc = pick_npc(g->n_nodes);
  d.f_dz = nullptr; d.f_slot = nullptr; d.f_alpha = nullptr; d.f_stride = 0; d.f_base = d.f_dy = d.f_y = nullptr;
  d.f_scale = 1.f; d.g_out = nullptr; d.f_pool = nullptr; d.f_seg = nullptr;
  if (fz) {   // the incoming gradient is assembled into b->dout by the destination pass
    d.f_dz = fz->dz_up; d.f_slot = fz->slot_of_eid; d.f_alpha = fz->alpha_up; d.f_stride = fz->alpha_up_stride;
    d.f_base = fz->g_base; d.f_dy = fz->dy; d.f_y = fz->y; d.f_scale = fz->scale;
    d.f_pool = fz->pool; d.f_seg = fz->seg_of;
    d.g_out = const_cast<float *>(b->dout);
  }
  const int grid = tile_grid(g->n_nodes, d.npc, 6);
  const bool affine = b->edge_mode == FNB_EDGE_AFFINE1 || b->edge_mode == FNB_EDGE_AFFINE6;
  if (affine && ((g->n_edges > 0 && !g->edge_attr) || !b->We || !b->be || !b->dWe || !b->dbe)) return FNB_ERR_NULL;
  const bool fuse = fz != nullptr, deep = deep_graph(g);
  if (b->edge_mode != FNB_EDGE_AFFINE1 && b->edge_mode != FNB_EDGE_AFFINE6 && b->edge_mode != FNB_EDGE_NONE &&
      b->edge_mode != FNB_EDGE_TABLE)
    return FNB_ERR_MODE;
  if (b->edge_mode == FNB_EDGE_AFFINE6 && (reinterpret_cast<uintptr_t>(g->edge_attr) & 7u)) return FNB_ERR_ALIGN;
#define FNB_LAUNCH_DST(MODE)                                                                                         \
  do {                                                                                                               \
    cudaError_t le;                                                                                                  \
    if (deep)                                                                                                        \
      le = fuse ? fnb_launch(k_gat_bwd_dst_tiled<MODE, true, true>, dim3(grid), dim3(T_THREADS), 0, stream, d)       \
                : fnb_launch(k_gat_bwd_dst_tiled<MODE, false, true>, dim3(grid), dim3(T_THREADS), 0, stream, d);     \
    else                                                                                                             \
      le = fuse ? fnb_launch(k_gat_bwd_dst_tiled<MODE, true>, dim3(grid), dim3(T_THREADS), 0, stream, d)             \
                : fnb_launch(k_gat_bwd_dst_tiled<MODE, false>, dim3(grid), dim3(T_THREADS), 0, stream, d);           \
    if (le != cudaSuccess) return (int)le;                                                                           \
  } while (0)
  if (b->edge_mode == FNB_EDGE_AFFINE1) {
    FNB_LAUNCH_DST(FNB_EDGE_AFFINE1);
  } else if (b->edge_mode == FNB_EDGE_AFFINE6) {
    if (reinterpret_cast<uintptr_t>(g->edge_attr) & 7u) return FNB_ERR_ALIGN;
    FNB_LAUNCH_DST(FNB_EDGE_AFFINE6);
  } else if (b->edge_mode == FNB_EDGE_NONE || b->edge_mode == FNB_EDGE_TABLE) {
    FNB_LAUNCH_DST(FNB_EDGE_NONE);
  } else {
    return FNB_ERR_MODE;
  }
#undef FNB_LAUNCH_DST
  FNB_CHECK_LAUNCH();
  if (after_dst)   // consumers of the destination pass's inputs (the consumer graph's dz) may be overwritten from here on
    if (cudaError_t ee = cudaEventRecord(after_dst, stream)) return (int)ee;
  if (before_src)  // readers of the buffer the source pass overwrites (args->dh), on another stream
    if (cudaError_t ee = cudaStreamWaitEvent(stream, before_src, 0)) return (int)ee;
  SrcT s;
  s.rrowptr = g->rrowptr; s.rslot = g->rslot; s.rdst = g->rdst; s.h = b->h; s.dout = b->dout; s.p_saved = b->p_saved;
  s.dz = b->dz; s.dSt = b->dSt; s.alpha = b->alpha; s.alpha_stride = b->alpha_stride; s.off_t = b->off_t;
  s.off_s = b->off_s; s.dh = b->dh; s.d_alpha = b->d_alpha; s.d_bias = b->d_bias; s.scratch = (float *)b->scratch;
  s.n_nodes = (int)g->n_nodes;
  s.npc = d.npc;
  if (deep) {
    if (cudaError_t le = fnb_launch(k_gat_bwd_src_tiled<true>, dim3(tile_grid(g->n_nodes, d.npc, 3)), dim3(T_THREADS), 0, stream, s)) return (int)le;
  } else {
    if (cudaError_t le = fnb_launch(k_gat_bwd_src_tiled<false>, dim3(grid), dim3(T_THREADS), 0, stream, s)) return (int)le;
  }
  FNB_CHECK_LAUNCH();
  return 0;
}

extern "C" int fnb_edge_table_bwd_fused(const fnb_graph *g, const float *dz, const float *feat, const float *alpha,
                                        int alpha_stride, int off_e, const float *g_base, const float *dy,
                                        const float *y, float post_scale, float *g_feat, float *d_alpha,
                                        void *scratch, void *stream_) {
  if (!graph_ok(g)) return g ? FNB_ERR_SIZE : FNB_ERR_NULL;
  if (!alpha || !d_alpha || !scratch) return FNB_ERR_NULL;
  if (g->n_real_edges > 0 && (!dz || !g->slot_of_eid || !feat)) return FNB_ERR_NULL;
  if ((dy == nullptr) != (y == nullptr)) return FNB_ERR_NULL;
  if ((alpha_stride & 3) || (off_e & 3) || !fnb_aligned16(alpha) || !fnb_aligned16(feat) || !fnb_aligned16(g_feat) ||
      !fnb_aligned16(dz) || !fnb_aligned16(g_base) || !fnb_aligned16(dy) || !fnb_aligned16(y) ||
      !fnb_aligned16(scratch))
    return FNB_ERR_ALIGN;
  TableT a;
  a.dz = dz; a.slot_of_eid = g->slot_of_eid; a.feat = feat; a.alpha = alpha; a.alpha_stride = alpha_stride;
  a.off_e = off_e; a.g_base = g_base; a.dy = dy; a.y = y; a.scale = post_scale; a.g_feat = g_feat; a.d_alpha = d_alpha;
  a.scratch = (float *)scratch; a.n_real = (int)g->n_real_edges;
  int64_t blocks = (g->n_real_edges + T_WARPS - 1) / T_WARPS;
  if (blocks > kNumSMs * 4) blocks = kNumSMs * 4;
  if (blocks < 1) blocks = 1;
  if (cudaError_t le = fnb_launch(k_edge_table_bwd_tiled, dim3((int)blocks), dim3(T_THREADS), 0, (cudaStream_t)stream_, a)) return (int)le;
  FNB_CHECK_LAUNCH();
  return 0;
}

extern "C" int fnb_attn_by_source(const int32_t *rrowptr, const int32_t *rslot, const float *p_saved, int64_t n_nodes,
                                  float *w, void *stream) {
  if (n_nodes < 0) return FNB_ERR_SIZE;
  if (n_nodes == 0) return 0;
  if (!rrowptr || !w) return FNB_ERR_NULL;   // rslot, p_saved: read only at the slots rrowptr lists (none: may be NULL)
  int64_t blocks = (n_nodes + 255) / 256;
  if (blocks > kNumSMs * 8) blocks = kNumSMs * 8;
  k_attn_by_source<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(rrowptr, rslot, p_saved, n_nodes, w);
  FNB_CHECK_LAUNCH();
  return 0;
}
