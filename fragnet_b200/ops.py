"""Thin host wrappers over the C ABI: tensor -> pointer plumbing, CSR plans, scratch buffers.

PyTorch is used here only for device memory and streams; every computation is a call into
``libfragnet_b200.so``.  All wrappers launch on ``torch.cuda.current_stream()`` and never
synchronise.
"""
from __future__ import annotations

import ctypes as C
import weakref
from dataclasses import dataclass, field
from typing import Optional

import torch

from . import _abi
from ._abi import (EDGE_AFFINE1, EDGE_AFFINE6, EDGE_NONE, EDGE_TABLE,  # noqa: F401  (re-exported)
                   PRECISION_FP32, PRECISION_TF32, PRECISION_TF32X3)

D, H = 128, 4


def _lib():
    return _abi.load()


def _p(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _f32c(t: torch.Tensor) -> torch.Tensor:
    """fp32, contiguous view of ``t`` (copy only if needed)."""
    if t.dtype != torch.float32:
        t = t.float()
    return t if t.is_contiguous() else t.contiguous()


def require_cuda(device=None) -> torch.device:
    """The device kernels run on.  There is no CPU fallback."""
    if not torch.cuda.is_available():
        raise RuntimeError("fragnet_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    if device is not None and torch.device(device).type == "cuda":
        return torch.device(device)
    return torch.device("cuda", torch.cuda.current_device())


_scratch_cache = {}


def scratch(device: torch.device) -> torch.Tensor:
    """Per (device, stream) scratch of ``fnb_scratch_bytes()`` for partial sums."""
    key = (device.index, torch.cuda.current_stream(device).cuda_stream)
    buf = _scratch_cache.get(key)
    if buf is None:
        buf = torch.zeros(_lib().fnb_scratch_bytes(), dtype=torch.uint8, device=device)   # arrival counters start at 0
        _scratch_cache[key] = buf
    return buf


# ------------------------------------------------------------------------------------------------
# (a) CSR plans
@dataclass
class GraphCSR:
    """Destination-sorted CSR + reverse CSR of one batched graph (all int32, on device)."""
    n_nodes: int
    n_edges: int          # including appended self loops
    n_real: int           # edges present in the input edge list
    rowptr: torch.Tensor
    col: Optional[torch.Tensor]
    row: Optional[torch.Tensor]     # destination node of every slot
    eid: Optional[torch.Tensor]
    slot_of_eid: Optional[torch.Tensor]
    rrowptr: Optional[torch.Tensor] = None
    rslot: Optional[torch.Tensor] = None
    rdst: Optional[torch.Tensor] = None
    status: Optional[torch.Tensor] = None   # int32[1], non-zero if an index was out of range
    attr: Optional[torch.Tensor] = None     # per-edge attributes permuted into slot order
    _c: Optional[_abi.CGraph] = field(default=None, repr=False)

    def cstruct(self) -> _abi.CGraph:
        """``fnb_graph`` view of this plan (built on first use; set ``attr`` before that)."""
        if self._c is None:
            a = lambda t: None if t is None else t.data_ptr()
            self._c = _abi.CGraph(self.n_nodes, self.n_edges, self.n_real, a(self.rowptr), a(self.col), a(self.row),
                                  a(self.eid), a(self.slot_of_eid), a(self.rrowptr), a(self.rslot), a(self.rdst),
                                  a(self.attr))
        return self._c


def csr_build(dst: torch.Tensor, src: Optional[torch.Tensor], n_nodes: int, self_loops: bool = False,
              reverse: bool = True) -> GraphCSR:
    """``fnb_csr_build`` on int64 index vectors that live on a CUDA device."""
    assert dst.dtype == torch.int64 and dst.is_cuda and dst.is_contiguous()
    if src is not None:
        assert src.dtype == torch.int64 and src.is_contiguous() and src.shape == dst.shape
    dev = dst.device
    E = dst.numel()
    total = E + (n_nodes if self_loops else 0)
    i32 = dict(dtype=torch.int32, device=dev)
    rowptr = torch.empty(n_nodes + 1, **i32)
    col = torch.empty(total, **i32)
    row = torch.empty(total, **i32)
    eid = torch.empty(total, **i32)
    slot_of_eid = torch.empty(total, **i32)
    rrowptr = rslot = rdst = None
    if reverse:
        rrowptr = torch.empty(n_nodes + 1, **i32)
        rslot = torch.empty(total, **i32)
        rdst = torch.empty(total, **i32)
    lib = _lib()
    ws_bytes = lib.fnb_csr_workspace_bytes(n_nodes, total)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    status = torch.zeros(1, **i32)
    rc = lib.fnb_csr_build(_p(dst), _p(src), E, n_nodes, int(self_loops), _p(rowptr), _p(col), _p(row), _p(eid),
                           _p(slot_of_eid), _p(rrowptr), _p(rslot), _p(rdst), _p(ws), ws_bytes, _p(status), _stream())
    _abi.check(rc, "csr_build")
    return GraphCSR(n_nodes, total, E, rowptr, col, row, eid, slot_of_eid, rrowptr, rslot, rdst, status)


def gather_rows(src: torch.Tensor, index: torch.Tensor, n_rows: int) -> torch.Tensor:
    src = _f32c(src)
    width = src.shape[1] if src.dim() == 2 else 1
    out = torch.empty((n_rows, width), dtype=torch.float32, device=src.device)
    _abi.check(_lib().fnb_gather_rows(_p(src), _p(index), n_rows, width, _p(out), _stream()), "gather_rows")
    return out


def segment_offsets(sorted_ids: torch.Tensor, n_segments: int) -> torch.Tensor:
    out = torch.empty(n_segments + 1, dtype=torch.int32, device=sorted_ids.device)
    _abi.check(_lib().fnb_segment_offsets(_p(sorted_ids), sorted_ids.numel(), n_segments, _p(out), _stream()),
               "segment_offsets")
    return out


def narrow_index(ids: torch.Tensor) -> torch.Tensor:
    out = torch.empty(ids.numel(), dtype=torch.int32, device=ids.device)
    _abi.check(_lib().fnb_narrow_index(_p(ids), ids.numel(), _p(out), _stream()), "narrow_index")
    return out


class MoleculeCount:
    """Number of molecules of a batch = last entry of the sorted ``batch`` / ``frag_batch`` vectors + 1.  It is data
    dependent in the reference (scatter_add sizes its output ``index.max()+1``, gat2.py:820-821) and is the one
    value the host needs from the device per batch.  For device-resident vectors the 16-byte read-back is queued
    FIRST on the stream (before the collate and encoder launches) into pinned memory and only waited for when the
    readout needs it, by which time it has long completed -- the launch pipeline is never drained."""

    def __init__(self, batch_vec, frag_batch_vec):
        self._value, self._event, self._pinned = None, None, None
        vecs = [v for v in (batch_vec, frag_batch_vec) if v is not None and v.numel()]
        if not vecs:
            self._value = 0
        elif all(not v.is_cuda for v in vecs):
            self._value = max(int(v[-1]) for v in vecs) + 1
        else:
            self._pinned = torch.zeros(2, dtype=torch.int64).pin_memory()
            for i, v in enumerate(vecs):
                self._pinned[i:i + 1].copy_(v[-1:], non_blocking=True)
            self._event = torch.cuda.Event()
            self._event.record()

    def get(self) -> int:
        if self._value is None:
            self._event.synchronize()
            self._value = int(self._pinned.max()) + 1
        return self._value


class ReadoutPlan:
    def __init__(self, count, atom_ptr, frag_ptr, batch32, frag_batch32):
        self._count = count
        self.atom_ptr, self.frag_ptr = atom_ptr, frag_ptr          # int32 [>= G+1] molecule boundaries
        self.batch32, self.frag_batch32 = batch32, frag_batch32    # int32 [Na], [Nf]

    @property
    def n_graphs(self) -> int:
        return self._count.get() if isinstance(self._count, MoleculeCount) else int(self._count)


class LayerPlan:
    """Everything index-shaped that the GAT2 blocks of one batch share across layers, forward and backward, built by
    ONE ``fnb_batch_plan_build`` call into one arena: CSR / reverse CSR of the four graphs, the atom->fragment
    membership CSR, edge attributes permuted into slot order, int32 index copies and the readout offsets.
    ``bond / atom / fbond / frag / pool`` expose the same data as ``GraphCSR`` tensor views (tests, tools)."""

    def __init__(self, arena: torch.Tensor, c: _abi.CBatchPlan, keep: tuple, count: Optional[MoleculeCount] = None):
        self.arena, self.c, self.keep, self.count = arena, c, keep, count
        self.n_atoms, self.n_frags = int(c.n_atoms), int(c.n_frags)
        self._views = {}

    def cstruct(self) -> _abi.CBatchPlan:
        return self.c

    def _view(self, ptr, n, dtype=torch.int32):
        if not ptr:
            return None
        off = ptr - self.arena.data_ptr()
        return self.arena[off:off + 4 * n].view(dtype)

    def _graph(self, name) -> GraphCSR:
        if name not in self._views:
            if name == "pool":
                g = GraphCSR(self.n_frags, self.n_atoms, self.n_atoms, self._view(self.c.pool_rowptr, self.n_frags + 1),
                             self._view(self.c.pool_col, self.n_atoms), None, None, None)
            else:
                cg = getattr(self.c, name)
                n, e = int(cg.n_nodes), int(cg.n_edges)
                aw = {"bond": 1, "fbond": 6}.get(name, 0)
                attr = self._view(cg.edge_attr, e * aw, torch.float32) if aw else None
                g = GraphCSR(n, e, int(cg.n_real_edges), self._view(cg.rowptr, n + 1), self._view(cg.col, e),
                             self._view(cg.row, e), self._view(cg.eid, e), self._view(cg.slot_of_eid, e),
                             self._view(cg.rrowptr, n + 1), self._view(cg.rslot, e), self._view(cg.rdst, e),
                             self._view(self.c.status, 1), attr.view(e, aw) if aw > 1 else attr)
                g._c = cg
            self._views[name] = g
        return self._views[name]

    bond = property(lambda self: self._graph("bond"))
    atom = property(lambda self: self._graph("atom"))
    fbond = property(lambda self: self._graph("fbond"))
    frag = property(lambda self: self._graph("frag"))
    pool = property(lambda self: self._graph("pool"))

    @property
    def a2f32(self):
        return self._view(self.c.a2f, self.n_atoms)

    @property
    def status(self):
        return self._view(self.c.status, 1)

    @property
    def readout(self) -> Optional[ReadoutPlan]:
        if not self.c.mol_atom_ptr:
            return None
        cap = int(self.c.n_graphs)      # capacity of the offset arrays (an upper bound on the molecule count)
        return ReadoutPlan(self.count, self._view(self.c.mol_atom_ptr, cap + 1), self._view(self.c.mol_frag_ptr, cap + 1),
                           self._view(self.c.batch32, self.n_atoms), self._view(self.c.frag_batch32, self.n_frags))


def _idx(t: torch.Tensor, dev) -> torch.Tensor:
    t = t.to(device=dev, dtype=torch.int64)
    return t if t.is_contiguous() else t.contiguous()


def batch_inputs(edge_index, frag_index, atom_to_frag_ids, edge_index_bonds_graph, edge_attr_bonds, edge_index_fbonds,
                 edge_attr_fbonds, batch_vec, frag_batch_vec, n_atoms: int, n_frags: int, n_bond_nodes: int,
                 n_fbond_nodes: int, n_graphs: int, device, convert: bool = True):
    """``fnb_batch_inputs`` of one batch and the tensors it points into (keep them alive until the library has read
    them).  The library reads (``device``, contiguous) int64 indices and float32 edge attributes: ``convert`` converts a
    tensor that is not; without it the result is None instead (nothing is copied).  The batch vectors may be None."""
    if edge_index.shape[1] != n_bond_nodes or frag_index.shape[1] != n_fbond_nodes:
        raise ValueError("fragnet_b200: the bond graph needs one node per column of edge_index and the "
                         "fragment-connection graph one node per column of frag_index (gat2.py:179-185, 293-295); got "
                         f"{n_bond_nodes} vs {edge_index.shape[1]} and {n_fbond_nodes} vs {frag_index.shape[1]}")
    i64, f32 = torch.int64, torch.float32
    t = dict(edge_index=(edge_index, i64), frag_index=(frag_index, i64), atom_to_frag_ids=(atom_to_frag_ids, i64),
             edge_index_bonds_graph=(edge_index_bonds_graph, i64), edge_index_fbonds=(edge_index_fbonds, i64),
             batch=(batch_vec, i64), frag_batch=(frag_batch_vec, i64), edge_attr_bonds=(edge_attr_bonds, f32),
             edge_attr_fbonds=(edge_attr_fbonds, f32))
    for name, (x, dtype) in t.items():
        if x is not None and (x.device != device or x.dtype != dtype or not x.is_contiguous()):
            if not convert:
                return None
            x = x.to(device=device, dtype=dtype).contiguous()
        t[name] = x
    inp = _abi.CBatchInputs(**{name: _ptr(x) for name, x in t.items()}, n_atoms=n_atoms, n_frags=n_frags,
                            n_bonds=n_bond_nodes, n_bond_edges=t["edge_index_bonds_graph"].shape[1],
                            n_fbond_nodes=n_fbond_nodes, n_fbond_edges=t["edge_index_fbonds"].shape[1], n_graphs=n_graphs)
    return inp, tuple(t.values())


def build_layer_plan(edge_index, frag_index, atom_to_frag_ids, edge_index_bonds_graph, edge_attr_bonds,
                     edge_index_fbonds, edge_attr_fbonds, n_atoms: int, n_frags: int, n_bond_nodes: int,
                     n_fbond_nodes: int, device, batch_vec=None, frag_batch_vec=None) -> LayerPlan:
    """On-device collate (north-star kernel a) for one batch: one library call, 9 launches.

    Row conventions (SURVEY.md fact 5): bond / fragment-connection graphs use row 0 as the softmax
    segment (reference gat2.py:138, :239); atom / fragment graphs use row 1 (gat2.py:187, :283), and
    the atom graph gets its self loops appended (gat2.py:179)."""
    dev = require_cuda(device)
    # molecule count: read back lazily (MoleculeCount); the offset arrays are sized by the upper bound n_frags
    # (every molecule owns at least one fragment, fragments.py:230-234)
    have_batch = batch_vec is not None and frag_batch_vec is not None
    count = MoleculeCount(batch_vec, frag_batch_vec) if have_batch else None
    if not have_batch:
        batch_vec = frag_batch_vec = None
    inp, keep = batch_inputs(edge_index, frag_index, atom_to_frag_ids, edge_index_bonds_graph, edge_attr_bonds,
                             edge_index_fbonds, edge_attr_fbonds, batch_vec, frag_batch_vec, n_atoms, n_frags,
                             n_bond_nodes, n_fbond_nodes, n_frags if have_batch else 0, dev)
    lib = _lib()
    nbytes = lib.fnb_batch_plan_bytes(C.byref(inp))
    arena = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=dev)
    c = _abi.CBatchPlan()
    _abi.check(lib.fnb_batch_plan_build(C.byref(inp), _ptr(arena), arena.numel(), C.byref(c), _stream()),
               "batch_plan_build")
    return LayerPlan(arena, c, keep, count)


_plan_cache = []          # [(weakrefs, versions, sizes, device, plan)], most recent first
_PLAN_CACHE_SIZE = 4


def clear_plan_cache() -> None:
    """Forget cached plans (benchmarks call this every step so that the on-device collate is always timed)."""
    del _plan_cache[:]
    del _readout_cache[:]


def layer_plan_for(index_tensors: tuple, sizes: tuple, device, batch_vec=None, frag_batch_vec=None) -> LayerPlan:
    """Plan cache keyed by the IDENTITY of the caller's index tensors (weak references + version
    counters): the separate layer calls of the visualisation code share one plan, a new batch never hits a stale one."""
    key_tensors = tuple(index_tensors) + tuple(t for t in (batch_vec, frag_batch_vec) if t is not None)
    for refs, versions, szs, dev, plan in _plan_cache:
        if szs == sizes and dev == device and len(refs) == len(key_tensors) and \
                all(r() is t for r, t in zip(refs, key_tensors)) and \
                versions == tuple(t._version for t in key_tensors):
            return plan
    plan = build_layer_plan(*index_tensors, *sizes, device, batch_vec, frag_batch_vec)
    refs = tuple(weakref.ref(t) for t in key_tensors)
    _plan_cache.insert(0, (refs, tuple(t._version for t in key_tensors), sizes, device, plan))
    del _plan_cache[_PLAN_CACHE_SIZE:]
    return plan


_readout_cache = []


def readout_plan_for(batch_vec: torch.Tensor, frag_batch_vec: torch.Tensor, device) -> ReadoutPlan:
    """Molecule boundaries of the sorted ``batch`` / ``frag_batch`` vectors: taken from the batch plan the encoder
    built for the same tensors, else computed standalone."""
    for refs, _, _, dev, plan in _plan_cache:
        if dev == device and len(refs) >= 2 and refs[-2]() is batch_vec and refs[-1]() is frag_batch_vec and \
                plan.readout is not None:
            return plan.readout
    for refs, plan in _readout_cache:
        if refs[0]() is batch_vec and refs[1]() is frag_batch_vec:
            return plan
    dev = require_cuda(device)
    n_graphs = MoleculeCount(batch_vec, frag_batch_vec).get()
    b, fb = _idx(batch_vec, dev), _idx(frag_batch_vec, dev)
    plan = ReadoutPlan(n_graphs, segment_offsets(b, n_graphs), segment_offsets(fb, n_graphs),
                       narrow_index(b), narrow_index(fb))
    _readout_cache.insert(0, ((weakref.ref(batch_vec), weakref.ref(frag_batch_vec)), plan))
    del _readout_cache[_PLAN_CACHE_SIZE:]
    return plan


# ------------------------------------------------------------------------------------------------
# kernel wrappers (no autograd here; see autograd.py)
def proj_fwd(x, W, b, alpha=None, alpha_stride=0, off_t=0, off_s=0, want_S=True, precision=0):
    n, K = x.shape
    h = torch.empty((n, D), dtype=torch.float32, device=x.device)
    S = torch.empty((n, 8), dtype=torch.float32, device=x.device) if want_S else None
    _abi.check(_lib().fnb_proj_fwd(_p(x), _p(W), _p(b), n, K, _p(alpha), alpha_stride, off_t, off_s, _p(h), _p(S),
                                   precision, _stream()), "proj_fwd")
    return h, S


def proj_bwd(x, W, dh, need_dx: bool, precision=0, want_db=True):
    n, K = x.shape
    dx = torch.empty_like(x) if need_dx else None
    dW = torch.empty_like(W)
    db = torch.empty(D, dtype=torch.float32, device=x.device) if want_db else None
    _abi.check(_lib().fnb_proj_bwd(_p(x), _p(W), _p(dh), n, K, _p(dx), _p(dW), _p(db), precision,
                                   _p(scratch(x.device)), _stream()), "proj_bwd")
    return dx, dW, db


def node_scalars(h, alpha, alpha_stride, off_t, off_s):
    S = torch.empty((h.shape[0], 8), dtype=torch.float32, device=h.device)
    _abi.check(_lib().fnb_node_scalars(_p(h), h.shape[0], _p(alpha), alpha_stride, off_t, off_s, _p(S), _stream()),
               "node_scalars")
    return S


def attn_by_source(g: GraphCSR, p):
    w = torch.empty((g.n_nodes, H), dtype=torch.float32, device=p.device)
    _abi.check(_lib().fnb_attn_by_source(_p(g.rrowptr), _p(g.rslot), _p(p), g.n_nodes, _p(w), _stream()),
               "attn_by_source")
    return w


# ---- node-tiled attention kernels (gat_tiled.cu) ------------------------------------------------
def gat_fwd_tiled(g: GraphCSR, h, S, mode, *, table=None, We=None, be=None, alpha_e=None, alpha_stride=0,
                  save_p=True, want_out=True, post=None, mask=(-1, -1), next_alpha=None, next_alpha_stride=0):
    """``fnb_gat_fwd_tiled``.  ``post`` = (p, training, relu, seed, offset) additionally returns
    y = ReLU(Dropout(out)).  Returns (out | None, y | None, p_saved | None, next_Se | None)."""
    dev = h.device
    out = torch.empty((g.n_nodes, D), dtype=torch.float32, device=dev) if want_out else None
    y = torch.empty((g.n_nodes, D), dtype=torch.float32, device=dev) if post is not None else None
    p = torch.empty((g.n_edges, H), dtype=torch.float32, device=dev) if save_p else None
    nse = torch.empty((g.n_nodes, H), dtype=torch.float32, device=dev) if next_alpha is not None else None
    pa = _abi.CPostAct(*(post if post is not None else (0.0, 0, 0, 0, 0)))
    args = _abi.CGatFwdArgs(_ptr(h), _ptr(S), mode, _ptr(table), _ptr(We), _ptr(be), _ptr(alpha_e), alpha_stride,
                            _ptr(out), _ptr(y), pa, _ptr(p), mask[0], mask[1], _ptr(next_alpha), next_alpha_stride,
                            _ptr(nse))
    _abi.check(_lib().fnb_gat_fwd_tiled(C.byref(g.cstruct()), C.byref(args), _stream()), "gat_fwd_tiled")
    return out, y, p, nse


def gat_bwd_tiled(g: GraphCSR, h, dout, p, mode, alpha, alpha_stride, off_t, off_e, off_s, d_alpha, *, We=None,
                  be=None, want_bias_grad=False, mark=None, out=None):
    """``fnb_gat_bwd_tiled`` (destination pass + source pass).  Writes the off_t / off_s (and, for the affine modes,
    off_e) slices of ``d_alpha``.  Returns (dh, dz, d_bias | None, dWe | None, dbe | None).  ``mark``: a created
    ``torch.cuda.Event`` recorded between the two passes; ``out``: (dz, dSt, dh) buffers to reuse."""
    dev = h.device
    if out is not None:
        dz, dSt, dh = out
    else:
        dz = torch.empty((g.n_edges, H), dtype=torch.float32, device=dev)
        dSt = torch.empty((g.n_nodes, H), dtype=torch.float32, device=dev)
        dh = torch.empty((g.n_nodes, D), dtype=torch.float32, device=dev)
    db = torch.empty(D, dtype=torch.float32, device=dev) if want_bias_grad else None
    affine = mode in (EDGE_AFFINE1, EDGE_AFFINE6)
    dWe = torch.empty_like(We) if affine else None
    dbe = torch.empty_like(be) if affine else None
    args = _abi.CGatBwdArgs(_ptr(h), _ptr(dout), _ptr(p), mode, _ptr(We), _ptr(be), _ptr(alpha), alpha_stride, off_t,
                            off_e, off_s, _ptr(dz), _ptr(dSt), _ptr(dh), _ptr(d_alpha), _ptr(db), _ptr(dWe), _ptr(dbe),
                            _ptr(scratch(dev)))
    if mark is not None:
        _abi.check(_lib().fnb_gat_bwd_tiled_marked(C.byref(g.cstruct()), C.byref(args), C.c_void_p(mark.cuda_event),
                                                   _stream()), "gat_bwd_tiled_marked")
    else:
        _abi.check(_lib().fnb_gat_bwd_tiled(C.byref(g.cstruct()), C.byref(args), _stream()), "gat_bwd_tiled")
    return dh, dz, db, dWe, dbe


def edge_table_bwd_fused(g: GraphCSR, dz, feat, alpha, alpha_stride, off_e, d_alpha, *, g_base=None, dy=None, y=None,
                         post_scale=1.0):
    """``fnb_edge_table_bwd_fused``: edge-term backward of a TABLE graph with the ReLU(Dropout) backward of the
    gradient arriving at the post-activation copy of ``feat`` folded in."""
    g_feat = torch.empty((g.n_real, D), dtype=torch.float32, device=feat.device)
    _abi.check(_lib().fnb_edge_table_bwd_fused(C.byref(g.cstruct()), _p(dz), _p(feat), _p(alpha), alpha_stride, off_e,
                                               _p(g_base), _p(dy), _p(y), float(post_scale), _p(g_feat), _p(d_alpha),
                                               _p(scratch(feat.device)), _stream()), "edge_table_bwd_fused")
    return g_feat


def segment_sum(rowptr, col, n_segments, x, out=None, out_stride=D, alpha=None, alpha_stride=0, off_t=0, off_s=0):
    if out is None:
        out = torch.empty((n_segments, D), dtype=torch.float32, device=x.device)
    S = torch.empty((n_segments, 8), dtype=torch.float32, device=x.device) if alpha is not None else None
    _abi.check(_lib().fnb_segment_sum(_p(rowptr), _p(col), n_segments, _p(x), _p(out), out_stride, _p(alpha),
                                      alpha_stride, off_t, off_s, _p(S), _stream()), "segment_sum")
    return out, S


def segment_gather(g, g_stride, seg_of, n_rows, base=None):
    dx = torch.empty((n_rows, D), dtype=torch.float32, device=g.device)
    _abi.check(_lib().fnb_segment_gather(_p(g), g_stride, _p(seg_of), n_rows, _p(base), _p(dx), _stream()),
               "segment_gather")
    return dx


def _take_rng(n_counters: int) -> int:
    """Dropout masks are a function of (torch's seed, a counter).  The counter is the Philox offset of torch's own CUDA
    generator of the current device -- the stream torch's dropout kernels draw from -- advanced by what a call
    consumes: ``torch.manual_seed`` therefore restarts it, and re-seeding reproduces the masks exactly as it does for
    ``nn.Dropout``."""
    gen = torch.cuda.default_generators[torch.cuda.current_device()]
    off = int(gen.get_offset())
    gen.set_offset(off + (int(n_counters) + 3) // 4 * 4)        # torch keeps the offset a multiple of 4
    return off


def next_rng(n_elems: int):
    """(seed, offset) for one dropout call; the offset stream advances by the number of RNG
    counters the call consumes, so no two calls of a run share random numbers."""
    return torch.initial_seed() & 0xFFFFFFFFFFFFFFFF, _take_rng((n_elems + 3) // 4)


def reserve_rng(n_counters: int) -> int:
    """First counter of a block of ``n_counters`` RNG counters (whole-encoder calls reserve all their dropout sites
    at once: ``fnb_encoder_rng_span``)."""
    return _take_rng(n_counters)


def dropout_relu_fwd(x, p: float, training: bool, relu: bool, seed: int, offset: int):
    y = torch.empty_like(x)
    _abi.check(_lib().fnb_dropout_relu_fwd(_p(x), _p(y), x.numel(), float(p), int(training), int(relu), seed, offset,
                                           _stream()), "dropout_relu_fwd")
    return y


def dropout_relu_bwd(dy, y, p: float, training: bool):
    dx = torch.empty_like(y)
    _abi.check(_lib().fnb_dropout_relu_bwd(_p(dy), _p(y), _p(dx), y.numel(), float(p), int(training), _stream()),
               "dropout_relu_bwd")
    return dx
