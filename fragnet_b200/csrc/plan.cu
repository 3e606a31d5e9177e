// On-device collate of a whole batch in ONE call: the five CSR plans (bond, atom + self loops, fragment-connection,
// fragment, atom->fragment membership), their reverse CSRs, the slot-ordered edge attributes and the readout offsets.
//
// What this replaces in the reference: torch_scatter groups edges implicitly on EVERY scatter_softmax / scatter_add
// call (fragnet/model/gat/gat2.py:153-165, 210-219, 234, 257-268, 303-312, 820-821), torch_geometric's add_self_loops
// (gat2.py:179) re-concatenates the edge list in every layer.  Here the grouping is done once per batch and shared
// by all layers, forward and backward.  One counting sort runs over the CONCATENATION of the five edge lists, so a
// batch costs 9 launches in total:
//   memset, histogram, 3-launch exclusive scan, slot claim, rank (forward), rank (reverse), aux (narrowing, offsets).
// fnb_csr_build runs the same sort (counting_sort below) over one caller's graph, with the other four graphs empty.
// Bit-exactness contract (tested against torch.sort(stable=True)): slots of one destination (source) are ordered by
// edge id; the only non-deterministic step (the atomic slot claim) is followed by a rank-by-counting pass.
// Also here: the small standalone index helpers fnb_gather_rows, fnb_segment_offsets and fnb_narrow_index.
#include "common.cuh"

namespace {

constexpr int PG = 5;  // bond, atom, fbond, frag, pool

struct GDesc {
  const int64_t *dst, *src;  // src == nullptr: src[e] = e (membership list)
  int n_real, n_total, n_nodes, n_src_nodes;
  int node_base;  // first counter of this graph in the concatenated count / scan arrays
  int edge_base;  // first edge of this graph in the concatenated edge space (host-side prefix of n_total)
  int reverse;
  int *rowptr, *col, *row, *eid, *slot_of_eid, *rrowptr, *rslot, *rdst;
  const float *attr_in;
  float *attr_out;
  int attr_w;
};

struct PlanArgs {
  GDesc g[PG];
  int e_total, n_total;
  int *cnt_dst, *cnt_src;   // [n_total]
  int *x_dst, *x_src;       // [n_total + 1] exclusive scans of the counters (global over the concatenation)
  int *tmp_eid, *tmp_reid;  // [e_total]
  int *status;
};

__device__ __forceinline__ int graph_of_edge(const PlanArgs &a, int e) {
  int g = 0;
#pragma unroll
  for (int i = 1; i < PG; ++i) g += (e >= a.g[i].edge_base);
  return g;
}
__device__ __forceinline__ int graph_of_node(const PlanArgs &a, int n) {
  int g = 0;
#pragma unroll
  for (int i = 1; i < PG; ++i) g += (n >= a.g[i].node_base);
  return g;
}
__device__ __forceinline__ bool edge_nodes_of(const GDesc &G, int e, int &d, int &s) {
  int64_t dd, ss;
  if (e < G.n_real) {
    dd = G.dst[e];
    ss = G.src ? G.src[e] : (int64_t)e;
  } else {  // appended self loop (add_self_loops, gat2.py:179)
    dd = ss = e - G.n_real;
  }
  d = (int)dd;
  s = (int)ss;
  return dd >= 0 && dd < G.n_nodes && ss >= 0 && ss < G.n_src_nodes;
}

__global__ void k_plan_histogram(PlanArgs a) {
  pdl_wait();
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < a.e_total; i += gridDim.x * blockDim.x) {
    const int gi = graph_of_edge(a, i);
    const GDesc &G = a.g[gi];
    int d, s;
    if (!edge_nodes_of(G, i - G.edge_base, d, s)) {
      atomicExch(a.status, 1);
      continue;
    }
    atomicAdd(&a.cnt_dst[G.node_base + d], 1);
    if (G.reverse) atomicAdd(&a.cnt_src[G.node_base + s], 1);
  }
}

// ---- exclusive scan over one or two arrays (blockIdx.y), three launches
constexpr int kScanBlock = 1024, kScanItems = 4, kScanTile = kScanBlock * kScanItems;
struct ScanArrays2 {
  const int *in[2];
  int *out[2];
  int *tile_sums[2];
  int n;
};
__device__ __forceinline__ int block_excl_scan(int v, int *total) {
  __shared__ int warp_tot[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(kFull, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) warp_tot[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    const int w = warp_tot[lane];
    int winc = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(kFull, winc, o);
      if (lane >= o) winc += t;
    }
    warp_tot[lane] = winc - w;
    if (lane == 31) *total = winc;
  }
  __syncthreads();
  const int res = warp_tot[warp] + inc - v;
  __syncthreads();
  return res;
}
__global__ void __launch_bounds__(kScanBlock) k_plan_scan_tiles(ScanArrays2 a) {
  pdl_wait();
  const int which = blockIdx.y;
  const int base = blockIdx.x * kScanTile + threadIdx.x * kScanItems;
  int v[kScanItems], sum = 0;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) {
    v[i] = (base + i < a.n) ? a.in[which][base + i] : 0;
    sum += v[i];
  }
  __shared__ int total;
  int excl = block_excl_scan(sum, &total);
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) {
    if (base + i < a.n) a.out[which][base + i] = excl;
    excl += v[i];
  }
  if (threadIdx.x == 0) a.tile_sums[which][blockIdx.x] = total;
}
__global__ void __launch_bounds__(kScanBlock) k_plan_scan_sums(ScanArrays2 a, int n_tiles) {
  pdl_wait();
  const int which = blockIdx.x;
  int *ts = a.tile_sums[which];
  __shared__ int total;
  int carry = 0;
  for (int base = 0; base < n_tiles; base += kScanBlock) {
    const int i = base + threadIdx.x;
    const int v = i < n_tiles ? ts[i] : 0;
    const int excl = block_excl_scan(v, &total);
    if (i < n_tiles) ts[i] = carry + excl;
    carry += total;
    __syncthreads();
  }
  if (threadIdx.x == 0) a.out[which][a.n] = carry;
}
__global__ void __launch_bounds__(kScanBlock) k_plan_scan_apply(ScanArrays2 a) {
  pdl_wait();
  const int which = blockIdx.y;
  const int add = a.tile_sums[which][blockIdx.x];
  const int base = blockIdx.x * kScanTile + threadIdx.x * kScanItems;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i)
    if (base + i < a.n) a.out[which][base + i] += add;
}

// Claim a position inside the destination / source segment (arbitrary order; fixed by the rank kernels).
__global__ void k_plan_claim(PlanArgs a) {
  pdl_wait();
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < a.e_total; i += gridDim.x * blockDim.x) {
    const int gi = graph_of_edge(a, i);
    const GDesc &G = a.g[gi];
    const int e = i - G.edge_base;
    int d, s;
    if (!edge_nodes_of(G, e, d, s)) continue;
    const int k = atomicSub(&a.cnt_dst[G.node_base + d], 1) - 1;
    a.tmp_eid[a.x_dst[G.node_base + d] + k] = e;
    if (G.reverse) {
      const int kr = atomicSub(&a.cnt_src[G.node_base + s], 1) - 1;
      a.tmp_reid[a.x_src[G.node_base + s] + kr] = e;
    }
  }
}

// One thread per claimed position: rank of its edge id inside its segment -> final slot; also the row pointers.
__global__ void k_plan_rank_forward(PlanArgs a) {
  pdl_wait();
  const int stride = gridDim.x * blockDim.x, t0 = blockIdx.x * blockDim.x + threadIdx.x;
  for (int i = t0; i < a.e_total; i += stride) {
    int gi = 0;
#pragma unroll
    for (int k = 1; k < PG; ++k) gi += (i >= a.x_dst[a.g[k].node_base]);
    const GDesc &G = a.g[gi];
    const int e = a.tmp_eid[i];
    if (e < 0 || e >= G.n_total) continue;  // only reachable after an out-of-range index (status != 0)
    int d, s;
    if (!edge_nodes_of(G, e, d, s)) continue;
    const int beg = a.x_dst[G.node_base + d], end = a.x_dst[G.node_base + d + 1];
    int rank = 0;
    for (int j = beg; j < end; ++j) rank += (a.tmp_eid[j] < e);
    const int slot = beg - a.x_dst[G.node_base] + rank;
    if (G.col) G.col[slot] = s;
    if (G.row) G.row[slot] = d;
    if (G.eid) G.eid[slot] = e;
    if (G.slot_of_eid) G.slot_of_eid[e] = slot;
    if (G.attr_out && e < G.n_real)
      for (int k = 0; k < G.attr_w; ++k) G.attr_out[(int64_t)slot * G.attr_w + k] = G.attr_in[(int64_t)e * G.attr_w + k];
  }
  for (int j = t0; j < a.n_total; j += stride) {
    const GDesc &G = a.g[graph_of_node(a, j)];
    const int n = j - G.node_base;
    const int b0 = a.x_dst[G.node_base];
    G.rowptr[n] = a.x_dst[j] - b0;
    if (n == G.n_nodes - 1) G.rowptr[n + 1] = a.x_dst[j + 1] - b0;
    if (G.reverse) {
      const int r0 = a.x_src[G.node_base];
      G.rrowptr[n] = a.x_src[j] - r0;
      if (n == G.n_nodes - 1) G.rrowptr[n + 1] = a.x_src[j + 1] - r0;
    }
  }
  // graphs without nodes still get rowptr[0] = 0
  if (t0 < PG && a.g[t0].n_nodes == 0) {
    a.g[t0].rowptr[0] = 0;
    if (a.g[t0].reverse) a.g[t0].rrowptr[0] = 0;
  }
}

__global__ void k_plan_rank_reverse(PlanArgs a) {
  pdl_wait();
  const int n_rev = a.x_src[a.n_total];  // edges of the graphs that have a reverse CSR
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_rev; i += gridDim.x * blockDim.x) {
    int gi = 0;
#pragma unroll
    for (int k = 1; k < PG; ++k) gi += (i >= a.x_src[a.g[k].node_base]);
    const GDesc &G = a.g[gi];
    if (!G.reverse) continue;
    const int e = a.tmp_reid[i];
    if (e < 0 || e >= G.n_total) continue;
    int d, s;
    if (!edge_nodes_of(G, e, d, s)) continue;
    const int beg = a.x_src[G.node_base + s], end = a.x_src[G.node_base + s + 1];
    int rank = 0;
    for (int j = beg; j < end; ++j) rank += (a.tmp_reid[j] < e);
    const int r = beg - a.x_src[G.node_base] + rank;
    G.rslot[r] = G.slot_of_eid[e];
    G.rdst[r] = d;
  }
}

struct AuxArgs {
  const int64_t *a2f, *batch, *frag_batch;
  int *a2f32, *batch32, *frag_batch32, *atom_ptr, *frag_ptr;
  int n_atoms, n_frags, n_graphs;
};
// First position i in [0, n) with ids[i] >= key (ids sorted ascending); I is the index type of the caller's loop.
template <class I>
__device__ __forceinline__ I lower_bound64(const int64_t *ids, I n, int64_t key) {
  I lo = 0, hi = n;
  while (lo < hi) {
    const I mid = (lo + hi) >> 1;
    if (ids[mid] < key) lo = mid + 1; else hi = mid;
  }
  return lo;
}
// int64 -> int32 narrowing of atom_to_frag_ids / batch / frag_batch, and the molecule boundaries of the sorted
// batch vectors (data.py:896-901) for the readout (gat2.py:820-821).
__global__ void k_plan_aux(AuxArgs a) {
  pdl_wait();
  const int stride = gridDim.x * blockDim.x, t0 = blockIdx.x * blockDim.x + threadIdx.x;
  for (int i = t0; i < a.n_atoms; i += stride) {
    a.a2f32[i] = (int)a.a2f[i];
    if (a.batch) a.batch32[i] = (int)a.batch[i];
  }
  if (a.frag_batch)
    for (int i = t0; i < a.n_frags; i += stride) a.frag_batch32[i] = (int)a.frag_batch[i];
  if (a.batch && a.frag_batch)
    for (int g = t0; g <= a.n_graphs; g += stride) {
      a.atom_ptr[g] = lower_bound64(a.batch, a.n_atoms, g);
      a.frag_ptr[g] = lower_bound64(a.frag_batch, a.n_frags, g);
    }
}

// ---- standalone index helpers (fnb_gather_rows, fnb_segment_offsets, fnb_narrow_index)
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
       g += (int64_t)gridDim.x * blockDim.x)
    offsets[g] = (int)lower_bound64(ids, n, g);
}

__global__ void k_narrow(const int64_t *__restrict__ in, int64_t n, int *__restrict__ out) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = (int)in[i];
}

template <class T>
T *take(char *base, size_t &off, size_t n) {
  off = (off + 255) & ~(size_t)255;
  T *p = base ? reinterpret_cast<T *>(base + off) : nullptr;
  off += n * sizeof(T);
  return p;
}

// Temporaries of one counting sort over n_nodes counters and n_edges edges (all graphs of a PlanArgs together).
struct SortTemps {
  int *cnt_dst, *cnt_src, *x_dst, *x_src, *tmp_eid, *tmp_reid, *tiles0, *tiles1;
  size_t cnt_bytes;   // cnt_dst and cnt_src are adjacent: one memset
};

SortTemps take_sort_temps(char *base, size_t &off, int64_t n_nodes, int64_t n_edges) {
  SortTemps t;
  t.cnt_dst = take<int>(base, off, n_nodes);
  t.cnt_src = take<int>(base, off, n_nodes);
  t.cnt_bytes = base ? (size_t)(reinterpret_cast<char *>(t.cnt_src) - reinterpret_cast<char *>(t.cnt_dst)) +
                           (size_t)n_nodes * 4
                     : 0;
  t.x_dst = take<int>(base, off, n_nodes + 1);
  t.x_src = take<int>(base, off, n_nodes + 1);
  t.tmp_eid = take<int>(base, off, n_edges);
  t.tmp_reid = take<int>(base, off, n_edges);
  const int64_t n_tiles = (n_nodes + kScanTile - 1) / kScanTile;
  t.tiles0 = take<int>(base, off, n_tiles + 1);
  t.tiles1 = take<int>(base, off, n_tiles + 1);
  return t;
}

struct PlanLayout {
  // outputs
  int *rowptr[PG], *col[PG], *row[PG], *eid[PG], *slot_of_eid[PG], *rrowptr[PG], *rslot[PG], *rdst[PG];
  float *attr_bond, *attr_fbond;
  int *a2f32, *batch32, *frag_batch32, *atom_ptr, *frag_ptr, *status;
  SortTemps t;
  size_t total;
};

struct Sz { int n_nodes[PG], n_total[PG], reverse[PG]; int e_total, n_total_nodes; };

Sz sizes(const fnb_batch_inputs *in) {
  Sz z;
  const int64_t nn[PG] = {in->n_bonds, in->n_atoms, in->n_fbond_nodes, in->n_frags, in->n_frags};
  const int64_t ne[PG] = {in->n_bond_edges, in->n_bonds + in->n_atoms, in->n_fbond_edges, in->n_fbond_nodes, in->n_atoms};
  const int rev[PG] = {1, 1, 1, 1, 0};
  z.e_total = 0; z.n_total_nodes = 0;
  for (int i = 0; i < PG; ++i) {
    z.n_nodes[i] = (int)nn[i]; z.n_total[i] = (int)ne[i]; z.reverse[i] = rev[i];
    z.e_total += (int)ne[i]; z.n_total_nodes += (int)nn[i];
  }
  return z;
}

PlanLayout plan_layout(const fnb_batch_inputs *in, char *base) {
  const Sz z = sizes(in);
  PlanLayout L{};
  size_t off = 0;
  for (int i = 0; i < PG; ++i) {
    L.rowptr[i] = take<int>(base, off, (size_t)z.n_nodes[i] + 1);
    L.col[i] = take<int>(base, off, z.n_total[i]);
    if (i < 4) {
      L.row[i] = take<int>(base, off, z.n_total[i]);
      L.eid[i] = take<int>(base, off, z.n_total[i]);
      L.slot_of_eid[i] = take<int>(base, off, z.n_total[i]);
      L.rrowptr[i] = take<int>(base, off, (size_t)z.n_nodes[i] + 1);
      L.rslot[i] = take<int>(base, off, z.n_total[i]);
      L.rdst[i] = take<int>(base, off, z.n_total[i]);
    }
  }
  L.attr_bond = take<float>(base, off, in->n_bond_edges);
  L.attr_fbond = take<float>(base, off, (size_t)in->n_fbond_edges * 6);
  L.a2f32 = take<int>(base, off, in->n_atoms);
  L.batch32 = take<int>(base, off, in->n_atoms);
  L.frag_batch32 = take<int>(base, off, in->n_frags);
  L.atom_ptr = take<int>(base, off, (size_t)in->n_graphs + 1);
  L.frag_ptr = take<int>(base, off, (size_t)in->n_graphs + 1);
  L.status = take<int>(base, off, 1);    // index error
  L.t = take_sort_temps(base, off, z.n_total_nodes, z.e_total);
  L.total = (off + 255) & ~(size_t)255;
  return L;
}

// fnb_csr_build's workspace: the sort temporaries and two spare words -- rowptr[0] of the four empty graphs, and the
// status word when the caller passes none.
struct CsrLayout {
  SortTemps t;
  int *spare;
  size_t total;
};

CsrLayout csr_layout(int64_t n_nodes, int64_t n_edges_total, char *base) {
  CsrLayout L;
  size_t off = 0;
  L.t = take_sort_temps(base, off, n_nodes, n_edges_total);
  L.spare = take<int>(base, off, 2);
  L.total = off;
  return L;
}

bool inputs_ok(const fnb_batch_inputs *in) {
  if (!in) return false;
  const int64_t v[] = {in->n_atoms, in->n_frags, in->n_bonds, in->n_bond_edges, in->n_fbond_nodes, in->n_fbond_edges,
                       in->n_graphs};
  int64_t sum = 0;
  for (int64_t x : v) {
    if (x < 0 || x >= (int64_t)INT32_MAX) return false;
    sum += x;
  }
  return sum + in->n_atoms + in->n_bonds < (int64_t)INT32_MAX;   // concatenated edge space stays in int32
}

inline int grid_for(int64_t n) {
  int64_t g = (n + 255) / 256;
  if (g > kNumSMs * 16) g = kNumSMs * 16;
  if (g < 1) g = 1;
  return (int)g;
}

// The k_plan_* kernels index edges and nodes with int and stride by up to one grid_for() grid (kNumSMs * 16 blocks of
// 256 threads): a sort of at most this many edges or nodes keeps every index plus one stride inside int32.
constexpr int64_t kMaxSortItems = (int64_t)INT32_MAX - (int64_t)kNumSMs * 16 * 256;

// The plan struct over a laid-out arena (pure function of the inputs' sizes).
void fill_plan(const fnb_batch_inputs *in, const PlanLayout &L, const Sz &z, fnb_batch_plan *out) {
  const int n_real[PG] = {(int)in->n_bond_edges, (int)in->n_bonds, (int)in->n_fbond_edges, (int)in->n_fbond_nodes,
                          (int)in->n_atoms};
  fnb_graph *gs[4] = {&out->bond, &out->atom, &out->fbond, &out->frag};
  for (int i = 0; i < 4; ++i) {
    fnb_graph &g = *gs[i];
    g.n_nodes = z.n_nodes[i]; g.n_edges = z.n_total[i]; g.n_real_edges = n_real[i];
    g.rowptr = L.rowptr[i]; g.col = L.col[i]; g.row = L.row[i]; g.eid = L.eid[i]; g.slot_of_eid = L.slot_of_eid[i];
    g.rrowptr = L.rrowptr[i]; g.rslot = L.rslot[i]; g.rdst = L.rdst[i]; g.edge_attr = nullptr;
  }
  out->bond.edge_attr = L.attr_bond;
  out->fbond.edge_attr = L.attr_fbond;
  out->pool_rowptr = L.rowptr[4]; out->pool_col = L.col[4]; out->a2f = L.a2f32;
  out->n_atoms = in->n_atoms; out->n_frags = in->n_frags;
  out->mol_atom_ptr = in->batch ? L.atom_ptr : nullptr; out->mol_frag_ptr = in->batch ? L.frag_ptr : nullptr;
  out->batch32 = in->batch ? L.batch32 : nullptr; out->frag_batch32 = in->batch ? L.frag_batch32 : nullptr;
  out->n_graphs = in->batch ? in->n_graphs : 0;
  out->status = L.status;
}

// The counting sort of the graphs described by `a` (its graphs, e_total, n_total and status), with the temporaries `t`:
// zero the counters, histogram, 3-launch exclusive scan, slot claim, forward rank, forward_ready (optional), reverse
// rank.  Every launch is in stream order on `stream`.
int counting_sort(PlanArgs a, const SortTemps &t, cudaStream_t stream, cudaEvent_t forward_ready) {
  a.cnt_dst = t.cnt_dst; a.cnt_src = t.cnt_src; a.x_dst = t.x_dst; a.x_src = t.x_src;
  a.tmp_eid = t.tmp_eid; a.tmp_reid = t.tmp_reid;
  const int n_tiles = (a.n_total + kScanTile - 1) / kScanTile;
  if (a.n_total > 0) {
    const cudaError_t err = cudaMemsetAsync(t.cnt_dst, 0, t.cnt_bytes, stream);
    if (err != cudaSuccess) return (int)err;
  }
  if (a.e_total > 0) {
    if (cudaError_t le = fnb_launch(k_plan_histogram, dim3(grid_for(a.e_total)), dim3(256), 0, stream, a)) return (int)le;
    FNB_CHECK_LAUNCH();
  }
  ScanArrays2 sc;
  sc.in[0] = t.cnt_dst; sc.out[0] = t.x_dst; sc.tile_sums[0] = t.tiles0;
  sc.in[1] = t.cnt_src; sc.out[1] = t.x_src; sc.tile_sums[1] = t.tiles1;
  sc.n = a.n_total;
  if (n_tiles > 0) {
    if (cudaError_t le = fnb_launch(k_plan_scan_tiles, dim3(n_tiles, 2), dim3(kScanBlock), 0, stream, sc)) return (int)le;
    FNB_CHECK_LAUNCH();
  }
  if (cudaError_t le = fnb_launch(k_plan_scan_sums, dim3(2), dim3(kScanBlock), 0, stream, sc, n_tiles)) return (int)le;
  FNB_CHECK_LAUNCH();
  if (n_tiles > 0) {
    if (cudaError_t le = fnb_launch(k_plan_scan_apply, dim3(n_tiles, 2), dim3(kScanBlock), 0, stream, sc)) return (int)le;
    FNB_CHECK_LAUNCH();
  }
  if (a.e_total > 0) {
    if (cudaError_t le = fnb_launch(k_plan_claim, dim3(grid_for(a.e_total)), dim3(256), 0, stream, a)) return (int)le;
    FNB_CHECK_LAUNCH();
  }
  if (cudaError_t le = fnb_launch(k_plan_rank_forward, dim3(grid_for(a.e_total > a.n_total ? a.e_total : a.n_total)),
                                  dim3(256), 0, stream, a))
    return (int)le;
  FNB_CHECK_LAUNCH();
  if (forward_ready) {
    const cudaError_t err = cudaEventRecord(forward_ready, stream);
    if (err != cudaSuccess) return (int)err;
  }
  if (a.e_total > 0) {
    if (cudaError_t le = fnb_launch(k_plan_rank_reverse, dim3(grid_for(a.e_total)), dim3(256), 0, stream, a)) return (int)le;
    FNB_CHECK_LAUNCH();
  }
  return 0;
}

}  // namespace

extern "C" size_t fnb_batch_plan_bytes(const fnb_batch_inputs *in) {
  if (!inputs_ok(in)) return 0;
  return plan_layout(in, nullptr).total;
}

int fnb_batch_plan_view(const fnb_batch_inputs *in, void *arena, size_t arena_bytes, fnb_batch_plan *out) {
  if (!in || !out || !arena) return FNB_ERR_NULL;
  if (!inputs_ok(in)) return FNB_ERR_SIZE;
  if (reinterpret_cast<uintptr_t>(arena) & 255u) return FNB_ERR_ALIGN;
  const PlanLayout L = plan_layout(in, (char *)arena);
  if (L.total > arena_bytes) return FNB_ERR_WORKSPACE;
  fill_plan(in, L, sizes(in), out);
  return 0;
}

extern "C" int fnb_batch_plan_build(const fnb_batch_inputs *in, void *arena, size_t arena_bytes, fnb_batch_plan *out,
                                    void *stream_) {
  return fnb_batch_plan_build_impl(in, arena, arena_bytes, out, stream_, nullptr);
}

// forward_ready (optional): recorded once everything the FORWARD attention kernels read is complete -- destination-
// sorted CSRs, slot-ordered edge attributes, the pooling CSR.  The reverse CSRs and the int32 /
// per-molecule arrays (backward, readout) follow; a step's first attention kernel starts ~20 us earlier by waiting
// for this event instead of for the whole plan.
int fnb_batch_plan_build_impl(const fnb_batch_inputs *in, void *arena, size_t arena_bytes, fnb_batch_plan *out,
                              void *stream_, cudaEvent_t forward_ready) {
  if (!in || !out || !arena) return FNB_ERR_NULL;
  if (!inputs_ok(in)) return FNB_ERR_SIZE;
  if (in->n_bonds > 0 && !in->edge_index) return FNB_ERR_NULL;
  if (in->n_fbond_nodes > 0 && !in->frag_index) return FNB_ERR_NULL;
  if (in->n_atoms > 0 && !in->atom_to_frag_ids) return FNB_ERR_NULL;
  if (in->n_bond_edges > 0 && (!in->edge_index_bonds_graph || !in->edge_attr_bonds)) return FNB_ERR_NULL;
  if (in->n_fbond_edges > 0 && (!in->edge_index_fbonds || !in->edge_attr_fbonds)) return FNB_ERR_NULL;
  if ((in->batch == nullptr) != (in->frag_batch == nullptr)) return FNB_ERR_NULL;
  if (reinterpret_cast<uintptr_t>(arena) & 255u) return FNB_ERR_ALIGN;
  const PlanLayout L = plan_layout(in, (char *)arena);
  if (L.total > arena_bytes) return FNB_ERR_WORKSPACE;
  const Sz z = sizes(in);
  cudaStream_t stream = (cudaStream_t)stream_;

  PlanArgs a{};
  // Row conventions (SURVEY.md fact 5): bond / fragment-connection graphs use row 0 of the edge list as the softmax
  // segment (gat2.py:138, :239); atom / fragment graphs use row 1 (gat2.py:187, :283); the atom graph gets its self
  // loops appended (gat2.py:179); the membership "graph" groups atoms by fragment (gat2.py:234).
  const int64_t *dsts[PG] = {in->edge_index_bonds_graph, in->edge_index ? in->edge_index + in->n_bonds : nullptr,
                             in->edge_index_fbonds, in->frag_index ? in->frag_index + in->n_fbond_nodes : nullptr,
                             in->atom_to_frag_ids};
  const int64_t *srcs[PG] = {in->edge_index_bonds_graph ? in->edge_index_bonds_graph + in->n_bond_edges : nullptr,
                             in->edge_index, in->edge_index_fbonds ? in->edge_index_fbonds + in->n_fbond_edges : nullptr,
                             in->frag_index, nullptr};
  const int n_real[PG] = {(int)in->n_bond_edges, (int)in->n_bonds, (int)in->n_fbond_edges, (int)in->n_fbond_nodes,
                          (int)in->n_atoms};
  int node_base = 0, edge_base = 0;
  for (int i = 0; i < PG; ++i) {
    GDesc &G = a.g[i];
    G.dst = dsts[i]; G.src = srcs[i]; G.n_real = n_real[i]; G.n_total = z.n_total[i]; G.n_nodes = z.n_nodes[i];
    G.n_src_nodes = i == 4 ? z.n_total[i] : z.n_nodes[i];
    G.node_base = node_base; G.edge_base = edge_base; G.reverse = z.reverse[i];
    G.rowptr = L.rowptr[i]; G.col = L.col[i]; G.row = L.row[i]; G.eid = L.eid[i]; G.slot_of_eid = L.slot_of_eid[i];
    G.rrowptr = L.rrowptr[i]; G.rslot = L.rslot[i]; G.rdst = L.rdst[i];
    G.attr_in = nullptr; G.attr_out = nullptr; G.attr_w = 0;
    node_base += z.n_nodes[i];
    edge_base += z.n_total[i];
  }
  a.g[0].attr_in = in->edge_attr_bonds; a.g[0].attr_out = L.attr_bond; a.g[0].attr_w = 1;
  a.g[2].attr_in = in->edge_attr_fbonds; a.g[2].attr_out = L.attr_fbond; a.g[2].attr_w = 6;
  a.e_total = z.e_total; a.n_total = z.n_total_nodes; a.status = L.status;

  const cudaError_t err = cudaMemsetAsync(L.status, 0, sizeof(int), stream);
  if (err != cudaSuccess) return (int)err;
  if (int rc = counting_sort(a, L.t, stream, forward_ready)) return rc;
  AuxArgs x;
  x.a2f = in->atom_to_frag_ids; x.batch = in->batch; x.frag_batch = in->frag_batch; x.a2f32 = L.a2f32;
  x.batch32 = L.batch32; x.frag_batch32 = L.frag_batch32; x.atom_ptr = L.atom_ptr; x.frag_ptr = L.frag_ptr;
  x.n_atoms = (int)in->n_atoms; x.n_frags = (int)in->n_frags; x.n_graphs = (int)in->n_graphs;
  if (cudaError_t le = fnb_launch(k_plan_aux, dim3(grid_for(in->n_atoms > in->n_graphs ? in->n_atoms : in->n_graphs + 1)), dim3(256), 0, stream, x))
    return (int)le;
  FNB_CHECK_LAUNCH();

  fill_plan(in, L, z, out);
  return 0;
}

extern "C" size_t fnb_csr_workspace_bytes(int64_t n_nodes, int64_t n_edges_total) {
  if (n_nodes < 0 || n_edges_total < 0) return 0;
  return csr_layout(n_nodes, n_edges_total, nullptr).total;
}

// One graph through the batch plan's counting sort: graph 0 of the PlanArgs is the caller's, graphs 1..4 are empty.
extern "C" int fnb_csr_build(const int64_t *dst, const int64_t *src, int64_t n_edges, int64_t n_nodes,
                             int append_self_loops, int32_t *rowptr, int32_t *col, int32_t *row, int32_t *eid,
                             int32_t *slot_of_eid, int32_t *rrowptr, int32_t *rslot, int32_t *rdst, void *workspace,
                             size_t workspace_bytes, int32_t *status, void *stream) {
  if (n_edges < 0 || n_nodes < 0) return FNB_ERR_SIZE;
  const int64_t n_total = n_edges + (append_self_loops ? n_nodes : 0);
  if (n_total > kMaxSortItems || n_nodes > kMaxSortItems) return FNB_ERR_SIZE;
  if (!rowptr || !workspace || (n_edges > 0 && !dst)) return FNB_ERR_NULL;
  const bool reverse = rrowptr != nullptr;
  if (reverse && n_total > 0 && (!rslot || !rdst || !slot_of_eid)) return FNB_ERR_NULL;
  if (workspace_bytes < fnb_csr_workspace_bytes(n_nodes, n_total)) return FNB_ERR_WORKSPACE;
  // With src == NULL the "source" index space is the edge list itself (membership lists); a reverse
  // CSR makes no sense there.
  if (!src && reverse && n_edges > 0) return FNB_ERR_MODE;

  const CsrLayout L = csr_layout(n_nodes, n_total, (char *)workspace);
  PlanArgs a{};
  GDesc &G = a.g[0];
  G.dst = dst; G.src = src; G.n_real = (int)n_edges; G.n_total = (int)n_total; G.n_nodes = (int)n_nodes;
  G.n_src_nodes = src ? (int)n_nodes : (int)n_total;
  G.reverse = reverse;
  G.rowptr = rowptr; G.col = col; G.row = row; G.eid = eid; G.slot_of_eid = slot_of_eid;
  G.rrowptr = rrowptr; G.rslot = rslot; G.rdst = rdst;
  for (int i = 1; i < PG; ++i) {     // empty graphs after the caller's; k_plan_rank_forward writes their rowptr[0]
    a.g[i].node_base = (int)n_nodes;
    a.g[i].edge_base = (int)n_total;
    a.g[i].rowptr = L.spare;
  }
  a.e_total = (int)n_total; a.n_total = (int)n_nodes;
  a.status = status ? status : L.spare + 1;    // the caller's status word is not zeroed here
  return counting_sort(a, L.t, (cudaStream_t)stream, nullptr);
}

extern "C" int fnb_gather_rows(const float *in, const int32_t *index, int64_t n_rows, int width, float *out,
                               void *stream) {
  if (n_rows < 0 || width <= 0) return FNB_ERR_SIZE;
  if (n_rows == 0) return 0;
  if (!in || !index || !out) return FNB_ERR_NULL;
  k_gather_rows<<<grid_for(n_rows * width), 256, 0, (cudaStream_t)stream>>>(in, index, n_rows, width, out);
  FNB_CHECK_LAUNCH();
  return 0;
}

extern "C" int fnb_segment_offsets(const int64_t *sorted_ids, int64_t n, int64_t n_segments, int32_t *offsets,
                                   void *stream) {
  if (n < 0 || n_segments < 0 || n >= (int64_t)INT32_MAX) return FNB_ERR_SIZE;
  if (!offsets || (n > 0 && !sorted_ids)) return FNB_ERR_NULL;
  k_segment_offsets<<<grid_for(n_segments + 1), 256, 0, (cudaStream_t)stream>>>(sorted_ids, n, n_segments, offsets);
  FNB_CHECK_LAUNCH();
  return 0;
}

extern "C" int fnb_narrow_index(const int64_t *in, int64_t n, int32_t *out, void *stream) {
  if (n < 0) return FNB_ERR_SIZE;
  if (n == 0) return 0;
  if (!in || !out) return FNB_ERR_NULL;
  k_narrow<<<grid_for(n), 256, 0, (cudaStream_t)stream>>>(in, n, out);
  FNB_CHECK_LAUNCH();
  return 0;
}
