// On-device collate: destination-sorted CSR and reverse (source-sorted) CSR of a batched edge list.
//
// What this replaces in the reference: torch_scatter groups edges implicitly on every call
// (scatter_softmax / scatter_add, fragnet/model/gat/gat2.py:153-165, 210-219, 257-268, 303-312) and
// torch_geometric's add_self_loops (gat2.py:179) re-concatenates the edge list in every layer.
// Here the grouping is done ONCE per batch and reused by all layers, forward and backward.
//
// Bit-exactness contract: slots of one destination (source) are ordered by edge id, i.e. the
// result equals a stable sort of the edge list by destination (source).  The pipeline is a
// counting sort -- histogram (integer atomics: counts are order independent), exclusive scan,
// atomic slot claim -- followed by a per-slot rank-by-counting pass that orders each segment by
// edge id, which removes the only non-determinism (the claim order).
#include "common.cuh"

namespace {

constexpr int kScanBlock = 1024;
constexpr int kScanItems = 4;
constexpr int kScanTile = kScanBlock * kScanItems;

__device__ __forceinline__ void edge_nodes(const int64_t *dst, const int64_t *src, int64_t n_real, int64_t e,
                                           int64_t &d, int64_t &s) {
  if (e < n_real) {
    d = dst[e];
    s = src ? src[e] : e;
  } else {  // appended self loop (add_self_loops, gat2.py:179)
    d = s = e - n_real;
  }
}

__global__ void k_histogram(const int64_t *__restrict__ dst, const int64_t *__restrict__ src, int64_t n_real,
                            int64_t n_total, int64_t n_nodes, int64_t n_src_nodes, int *__restrict__ cnt_dst,
                            int *__restrict__ cnt_src, int *__restrict__ status) {
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < n_total; e += (int64_t)gridDim.x * blockDim.x) {
    int64_t d, s;
    edge_nodes(dst, src, n_real, e, d, s);
    if (d < 0 || d >= n_nodes || s < 0 || s >= n_src_nodes) {
      if (status) atomicExch(status, 1);
      continue;
    }
    atomicAdd(&cnt_dst[d], 1);
    if (cnt_src) atomicAdd(&cnt_src[s], 1);
  }
}

// Exclusive scan, three launches (tile sums, scan of tile sums, apply); blockIdx.y selects the array.
struct ScanArrays {
  const int *in[2];
  int *out[2];
  int *tile_sums[2];
  int64_t n[2];
};

__device__ __forceinline__ int block_exclusive_scan(int v, int *total) {
  __shared__ int warp_tot[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int t = __shfl_up_sync(kFull, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) warp_tot[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    int w = warp_tot[lane];
    int winc = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int t = __shfl_up_sync(kFull, winc, o);
      if (lane >= o) winc += t;
    }
    warp_tot[lane] = winc - w;  // exclusive prefix of warp totals
    if (lane == 31) *total = winc;
  }
  __syncthreads();
  int res = warp_tot[warp] + inc - v;
  __syncthreads();
  return res;
}

__global__ void __launch_bounds__(kScanBlock) k_scan_tiles(ScanArrays a) {
  const int which = blockIdx.y;
  const int64_t n = a.n[which];
  const int64_t base = (int64_t)blockIdx.x * kScanTile + (int64_t)threadIdx.x * kScanItems;
  if ((int64_t)blockIdx.x * kScanTile >= n) return;
  int v[kScanItems], sum = 0;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) {
    v[i] = (base + i < n) ? a.in[which][base + i] : 0;
    sum += v[i];
  }
  __shared__ int total;
  int excl = block_exclusive_scan(sum, &total);
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) {
    if (base + i < n) a.out[which][base + i] = excl;
    excl += v[i];
  }
  if (threadIdx.x == 0) a.tile_sums[which][blockIdx.x] = total;
}

// One block per array: exclusive scan of the tile sums in place; writes the grand total to out[n].
__global__ void __launch_bounds__(kScanBlock) k_scan_tile_sums(ScanArrays a, int n_tiles0, int n_tiles1) {
  const int which = blockIdx.x;
  const int n_tiles = which == 0 ? n_tiles0 : n_tiles1;
  int *ts = a.tile_sums[which];
  __shared__ int total;
  int carry = 0;
  for (int base = 0; base < n_tiles; base += kScanBlock) {
    int i = base + threadIdx.x;
    int v = i < n_tiles ? ts[i] : 0;
    int excl = block_exclusive_scan(v, &total);
    if (i < n_tiles) ts[i] = carry + excl;
    carry += total;
    __syncthreads();
  }
  if (threadIdx.x == 0) a.out[which][a.n[which]] = carry;
}

__global__ void __launch_bounds__(kScanBlock) k_scan_apply(ScanArrays a) {
  const int which = blockIdx.y;
  const int64_t n = a.n[which];
  const int add = a.tile_sums[which][blockIdx.x];
  const int64_t base = (int64_t)blockIdx.x * kScanTile + (int64_t)threadIdx.x * kScanItems;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i)
    if (base + i < n) a.out[which][base + i] += add;
}

// Claim a slot inside the destination / source segment (arbitrary order; fixed by k_rank below).
__global__ void k_claim(const int64_t *__restrict__ dst, const int64_t *__restrict__ src, int64_t n_real,
                        int64_t n_total, int64_t n_nodes, int64_t n_src_nodes, const int *__restrict__ rowptr,
                        const int *__restrict__ rrowptr, int *__restrict__ cnt_dst, int *__restrict__ cnt_src,
                        int *__restrict__ tmp_eid, int *__restrict__ tmp_reid) {
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < n_total; e += (int64_t)gridDim.x * blockDim.x) {
    int64_t d, s;
    edge_nodes(dst, src, n_real, e, d, s);
    if (d < 0 || d >= n_nodes || s < 0 || s >= n_src_nodes) continue;
    int k = atomicSub(&cnt_dst[d], 1) - 1;
    tmp_eid[rowptr[d] + k] = (int)e;
    if (cnt_src) {
      int kr = atomicSub(&cnt_src[s], 1) - 1;
      tmp_reid[rrowptr[s] + kr] = (int)e;
    }
  }
}

// One thread per claimed slot: rank of its edge id among the ids of its segment -> final slot.
__global__ void k_rank_forward(const int64_t *__restrict__ dst, const int64_t *__restrict__ src, int64_t n_real,
                               int64_t n_total, const int *__restrict__ rowptr, const int *__restrict__ tmp_eid,
                               int *__restrict__ col, int *__restrict__ row, int *__restrict__ eid,
                               int *__restrict__ slot_of_eid) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n_total; i += (int64_t)gridDim.x * blockDim.x) {
    const int e = tmp_eid[i];
    if (e < 0 || e >= n_total) continue;  // only reachable after an out-of-range index (status != 0)
    int64_t d, s;
    edge_nodes(dst, src, n_real, e, d, s);
    const int beg = rowptr[d], end = rowptr[d + 1];
    int rank = 0;
    for (int j = beg; j < end; ++j) rank += (tmp_eid[j] < e);
    const int slot = beg + rank;
    if (col) col[slot] = (int)s;
    if (row) row[slot] = (int)d;
    if (eid) eid[slot] = e;
    if (slot_of_eid) slot_of_eid[e] = slot;
  }
}

__global__ void k_rank_reverse(const int64_t *__restrict__ dst, const int64_t *__restrict__ src, int64_t n_real,
                               int64_t n_total, const int *__restrict__ rrowptr, const int *__restrict__ tmp_reid,
                               const int *__restrict__ slot_of_eid, int *__restrict__ rslot, int *__restrict__ rdst) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n_total; i += (int64_t)gridDim.x * blockDim.x) {
    const int e = tmp_reid[i];
    if (e < 0 || e >= n_total) continue;
    int64_t d, s;
    edge_nodes(dst, src, n_real, e, d, s);
    const int beg = rrowptr[s], end = rrowptr[s + 1];
    int rank = 0;
    for (int j = beg; j < end; ++j) rank += (tmp_reid[j] < e);
    rslot[beg + rank] = slot_of_eid[e];
    rdst[beg + rank] = (int)d;
  }
}

__global__ void k_gather_rows(const float *__restrict__ in, const int *__restrict__ index, int64_t n_rows, int width,
                              float *__restrict__ out) {
  const int64_t total = n_rows * width;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / width;
    const int c = (int)(i - r * width);
    out[i] = in[(int64_t)index[r] * width + c];
  }
}

__global__ void k_segment_offsets(const int64_t *__restrict__ ids, int64_t n, int64_t n_segments,
                                  int *__restrict__ offsets) {
  for (int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; g <= n_segments;
       g += (int64_t)gridDim.x * blockDim.x) {
    int64_t lo = 0, hi = n;  // first i with ids[i] >= g
    while (lo < hi) {
      int64_t mid = (lo + hi) >> 1;
      if (ids[mid] < g) lo = mid + 1; else hi = mid;
    }
    offsets[g] = (int)lo;
  }
}

__global__ void k_narrow(const int64_t *__restrict__ in, int64_t n, int *__restrict__ out) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = (int)in[i];
}

inline int grid_for(int64_t n, int block) {
  int64_t g = (n + block - 1) / block;
  const int64_t cap = (int64_t)kNumSMs * 16;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

inline size_t align_up(size_t x) { return (x + 255) & ~(size_t)255; }

}  // namespace

extern "C" size_t fnb_csr_workspace_bytes(int64_t n_nodes, int64_t n_edges_total) {
  if (n_nodes < 0 || n_edges_total < 0) return 0;
  const size_t n_tiles = (size_t)(n_nodes + kScanTile - 1) / kScanTile + 1;
  return 2 * align_up((size_t)n_nodes * 4) + 2 * align_up((size_t)n_edges_total * 4) + 2 * align_up(n_tiles * 4) + 256;
}

extern "C" int fnb_csr_build(const int64_t *dst, const int64_t *src, int64_t n_edges, int64_t n_nodes,
                             int append_self_loops, int32_t *rowptr, int32_t *col, int32_t *row, int32_t *eid,
                             int32_t *slot_of_eid, int32_t *rrowptr, int32_t *rslot, int32_t *rdst, void *workspace,
                             size_t workspace_bytes, int32_t *status, void *stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (n_edges < 0 || n_nodes < 0) return FNB_ERR_SIZE;
  const int64_t n_total = n_edges + (append_self_loops ? n_nodes : 0);
  if (n_total >= (int64_t)INT32_MAX || n_nodes >= (int64_t)INT32_MAX) return FNB_ERR_SIZE;
  if (!rowptr || !workspace || (n_edges > 0 && !dst)) return FNB_ERR_NULL;
  const bool reverse = rrowptr != nullptr;
  if (reverse && (!rslot || !rdst || !slot_of_eid)) return FNB_ERR_NULL;
  if (workspace_bytes < fnb_csr_workspace_bytes(n_nodes, n_total)) return FNB_ERR_WORKSPACE;
  // With src == NULL the "source" index space is the edge list itself (membership lists); a reverse
  // CSR makes no sense there.
  if (!src && reverse && n_edges > 0) return FNB_ERR_MODE;
  const int64_t n_src_nodes = src ? n_nodes : n_total;

  char *ws = (char *)workspace;
  int *cnt_dst = (int *)ws;  ws += align_up((size_t)n_nodes * 4);
  int *cnt_src = (int *)ws;  ws += align_up((size_t)n_nodes * 4);
  int *tmp_eid = (int *)ws;  ws += align_up((size_t)n_total * 4);
  int *tmp_reid = (int *)ws; ws += align_up((size_t)n_total * 4);
  const int n_tiles = (int)((n_nodes + kScanTile - 1) / kScanTile);
  int *tiles0 = (int *)ws;   ws += align_up(((size_t)n_tiles + 1) * 4);
  int *tiles1 = (int *)ws;

  cudaError_t err;
  if (n_nodes > 0) {
    err = cudaMemsetAsync(cnt_dst, 0, (size_t)n_nodes * 4, stream);
    if (err != cudaSuccess) return (int)err;
    if (reverse) {
      err = cudaMemsetAsync(cnt_src, 0, (size_t)n_nodes * 4, stream);
      if (err != cudaSuccess) return (int)err;
    }
  }
  if (n_total > 0) {
    k_histogram<<<grid_for(n_total, 256), 256, 0, stream>>>(dst, src, n_edges, n_total, n_nodes, n_src_nodes, cnt_dst,
                                                            reverse ? cnt_src : nullptr, status);
    FNB_CHECK_LAUNCH();
  }
  ScanArrays a;
  a.in[0] = cnt_dst; a.out[0] = rowptr; a.tile_sums[0] = tiles0; a.n[0] = n_nodes;
  a.in[1] = cnt_src; a.out[1] = rrowptr; a.tile_sums[1] = tiles1; a.n[1] = n_nodes;
  const int n_arrays = reverse ? 2 : 1;
  if (n_tiles > 0) {
    k_scan_tiles<<<dim3(n_tiles, n_arrays), kScanBlock, 0, stream>>>(a);
    FNB_CHECK_LAUNCH();
  }
  k_scan_tile_sums<<<n_arrays, kScanBlock, 0, stream>>>(a, n_tiles, n_tiles);
  FNB_CHECK_LAUNCH();
  if (n_tiles > 0) {
    k_scan_apply<<<dim3(n_tiles, n_arrays), kScanBlock, 0, stream>>>(a);
    FNB_CHECK_LAUNCH();
  }
  if (n_total > 0) {
    k_claim<<<grid_for(n_total, 256), 256, 0, stream>>>(dst, src, n_edges, n_total, n_nodes, n_src_nodes, rowptr,
                                                        rrowptr, cnt_dst, reverse ? cnt_src : nullptr, tmp_eid,
                                                        tmp_reid);
    FNB_CHECK_LAUNCH();
    k_rank_forward<<<grid_for(n_total, 256), 256, 0, stream>>>(dst, src, n_edges, n_total, rowptr, tmp_eid, col, row, eid,
                                                               slot_of_eid);
    FNB_CHECK_LAUNCH();
    if (reverse) {
      k_rank_reverse<<<grid_for(n_total, 256), 256, 0, stream>>>(dst, src, n_edges, n_total, rrowptr, tmp_reid,
                                                                 slot_of_eid, rslot, rdst);
      FNB_CHECK_LAUNCH();
    }
  }
  return 0;
}

extern "C" int fnb_gather_rows(const float *in, const int32_t *index, int64_t n_rows, int width, float *out,
                               void *stream) {
  if (n_rows < 0 || width <= 0) return FNB_ERR_SIZE;
  if (n_rows == 0) return 0;
  if (!in || !index || !out) return FNB_ERR_NULL;
  k_gather_rows<<<grid_for(n_rows * width, 256), 256, 0, (cudaStream_t)stream>>>(in, index, n_rows, width, out);
  FNB_CHECK_LAUNCH();
  return 0;
}

extern "C" int fnb_segment_offsets(const int64_t *sorted_ids, int64_t n, int64_t n_segments, int32_t *offsets,
                                   void *stream) {
  if (n < 0 || n_segments < 0 || n >= (int64_t)INT32_MAX) return FNB_ERR_SIZE;
  if (!offsets || (n > 0 && !sorted_ids)) return FNB_ERR_NULL;
  k_segment_offsets<<<grid_for(n_segments + 1, 256), 256, 0, (cudaStream_t)stream>>>(sorted_ids, n, n_segments,
                                                                                    offsets);
  FNB_CHECK_LAUNCH();
  return 0;
}

extern "C" int fnb_narrow_index(const int64_t *in, int64_t n, int32_t *out, void *stream) {
  if (n < 0) return FNB_ERR_SIZE;
  if (n == 0) return 0;
  if (!in || !out) return FNB_ERR_NULL;
  k_narrow<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(in, n, out);
  FNB_CHECK_LAUNCH();
  return 0;
}
