"""Every route through the node-tiled attention kernels (gat_tiled.cu) against a float64 reference.

A launch of these kernels picks a tile size (pick_npc), an instantiation (plain, WIDE or DEEP) and a grid capped at a
few CTAs per SM; inside a tile, a node whose segment exceeds the staging capacity of a sub-tile takes a warp-serial hub
path, and the parameter gradients leave through the two-level cta_finish tree.  The graphs below are built from a
Python model of those choices, whose constants are parsed from the CUDA sources, so that each case lands on the route
it names -- and asserts that it did, from the model and from the kernel names and grids of a profiler trace -- and
follows the capacities if a later change moves them.

The reference is ``attention_ref``: the math of ``oracle.gat2_oracle.attention_block`` with every scatter sized to the
node count, so that nodes without incoming edges (real bond, fragment and fragment-connection graphs have them) get
the zero rows the kernels write.  On the GPU it runs in float64 on the device, with autograd for the gradients.
"""
import functools
import json
import os
import re
import tempfile
from dataclasses import dataclass

import pytest
import torch
import torch.nn.functional as F

from conftest import FP32_REL_TOL, rel_err
from oracle.shims import scatter_add, scatter_softmax

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "fragnet_b200", "csrc")
GRAD_TOL = 2e-5     # gradients: sums of O(100..1000) fp32 products in a different (fixed) order (test_gpu_tiled.py)
BIAS_TOL = 2e-4     # column sums of dh over every node


# ------------------------------------------------------------------------------------------------
# float64 reference
def attention_ref(h, dst, src, edge_vec, alpha, n_nodes, S=None):
    """One GAT2 attention block, as ``oracle.gat2_oracle.attention_block`` computes it, with every scatter given
    ``dim_size=n_nodes``: a node without incoming edges gets a zero output row.

    ``h`` [N,H,d], ``edge_vec`` [E,De], ``alpha`` [H, d+De+d].  With ``S`` [N,2H] the target and source terms of the
    logit are taken from ``S`` (the kernels' forward takes them as an input) and ``alpha`` is the edge slice [H,De].
    Returns (out [N,H*d], attention summed by source [N,H], pre-activation logits z [E,H]); z retains its gradient,
    which is what the kernels return as ``dz``."""
    n_heads, d = h.size(1), h.size(2)
    e_rep = edge_vec.repeat(n_heads, 1, 1).permute(1, 0, 2)
    if S is None:
        message = torch.cat([torch.index_select(h, 0, dst), e_rep, torch.index_select(h, 0, src)], dim=-1)
        z = torch.sum(message * alpha, dim=2)
    else:
        z = (torch.index_select(S[:, :n_heads], 0, dst) + torch.sum(e_rep * alpha, dim=2)
             + torch.index_select(S[:, n_heads:], 0, src))
    if z.requires_grad:
        z.retain_grad()
    logits = F.leaky_relu(z, 0.2)
    probs = scatter_softmax(logits, dst, dim=0, dim_size=n_nodes)
    weighted = probs[..., None] * torch.index_select(h, 0, src)
    summed = scatter_add(weighted, dst, dim=0, dim_size=n_nodes)
    by_source = scatter_add(probs, src, dim=0, dim_size=n_nodes)
    return summed.view(n_nodes, -1), by_source, z


# ------------------------------------------------------------------------------------------------
# route model: the launchers' choices of gat_tiled.cu, restated from constants parsed out of the sources
_CONST = re.compile(r"constexpr\s+int\s+(\w+)\s*=\s*(\d+)\s*;")
# the two capacities that are expressions inside the kernels; if either line changes, the model must be revisited
_FWD_CAP_LINE = re.compile(r"constexpr int CAP = DEEP \? (\d+) \* FWD_CAP : FWD_CAP;")
_SRC_CAP_LINE = re.compile(r"constexpr int CAP = DEEP \? (\d+) : BWD_CAP;")


def _read(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _constants(text, names):
    found = dict((k, int(v)) for k, v in _CONST.findall(text))
    missing = [n for n in names if n not in found]
    assert not missing, f"constants not found: {missing}"
    return {n: found[n] for n in names}


@dataclass(frozen=True)
class Routes:
    t_npc: int
    fwd_cap: int
    bwd_cap: int
    deep_degree: int
    fwd_deep_factor: int     # forward DEEP capacity = factor * FWD_CAP
    src_deep_cap: int
    n_sms: int
    finish_group: int
    # CTAs per SM of each grid (tile_grid's third argument in the launchers); the profiler trace checks the grids
    FWD_PER_SM, WIDE_PER_SM, DEEP_FWD_PER_SM, DST_PER_SM, SRC_PER_SM, DEEP_SRC_PER_SM = 6, 5, 4, 6, 6, 3

    @staticmethod
    @functools.lru_cache(maxsize=None)
    def parse():
        tiled = _read("gat_tiled.cu")
        c = _constants(tiled, ["T_NPC", "FWD_CAP", "BWD_CAP", "kDeepDegree"])
        k = _constants(_read("common.cuh"), ["kNumSMs", "kFinishGroup"])
        fwd = _FWD_CAP_LINE.findall(tiled)
        src = _SRC_CAP_LINE.findall(tiled)
        assert len(fwd) == 1 and len(src) == 1, "the forward / source-pass capacity lines of gat_tiled.cu changed"
        return Routes(c["T_NPC"], c["FWD_CAP"], c["BWD_CAP"], c["kDeepDegree"], int(fwd[0]), int(src[0]),
                      k["kNumSMs"], k["kFinishGroup"])

    def pick_npc(self, n):
        npc = self.t_npc
        while npc > 8:
            if -(-n // npc) >= self.n_sms * 2:
                return npc
            npc >>= 1
        return 8

    def tiles(self, n):
        return -(-n // self.pick_npc(n))

    def tile_grid(self, n, per_sm):
        return max(1, min(self.tiles(n), self.n_sms * per_sm))

    def deep(self, n, e):
        return n > 0 and e >= self.deep_degree * n

    def wide(self, n, e):
        return not self.deep(n, e) and self.tiles(n) > self.n_sms * self.FWD_PER_SM

    def caps(self, n, e):
        """Slots one sub-tile stages: (forward, destination pass, source pass)."""
        deep = self.deep(n, e)
        return (self.fwd_deep_factor * self.fwd_cap if deep else self.fwd_cap, self.bwd_cap,
                self.src_deep_cap if deep else self.bwd_cap)

    def grids(self, n, e):
        """(forward, destination pass, source pass) grid sizes."""
        fwd = self.DEEP_FWD_PER_SM if self.deep(n, e) else self.WIDE_PER_SM if self.wide(n, e) else self.FWD_PER_SM
        src = self.DEEP_SRC_PER_SM if self.deep(n, e) else self.SRC_PER_SM
        return self.tile_grid(n, fwd), self.tile_grid(n, self.DST_PER_SM), self.tile_grid(n, src)

    def subtiles(self, rowptr, cap):
        """The kernels' walk over tiles with subtile_end: ([(first node, end node, slots)] of the staged sub-tiles,
        [hub nodes])."""
        rp = rowptr.tolist() if torch.is_tensor(rowptr) else list(rowptr)
        n = len(rp) - 1
        npc = self.pick_npc(n)
        subs, hubs = [], []
        for n0 in range(0, n, npc):
            nn = min(npc, n - n0)
            lb = 0
            while lb < nn:
                base = rp[n0 + lb]
                if rp[n0 + nn] - base <= cap:
                    le = nn
                else:
                    le = lb
                    while le < nn and rp[n0 + le + 1] - base <= cap:
                        le += 1
                if le == lb:
                    hubs.append(n0 + lb)
                    lb += 1
                    continue
                subs.append((n0 + lb, n0 + le, rp[n0 + le] - base))
                lb = le
        return subs, hubs

    def first_n(self, pred, hi=1 << 18):
        """Smallest n from which pred(n) holds for every node count up to hi.  Not a bisection: tile counts fall each
        time pick_npc doubles the tile, so "more tiles than CTAs" holds on several ranges of n (the DEEP source pass
        loops over tiles from 3 553 to 4 720 nodes at npc 8, and again from 7 105, 14 209 and 28 417 nodes)."""
        assert pred(hi)
        n = hi
        while n > 1 and pred(n - 1):
            n -= 1
        return n

    def npc_thresholds(self):
        """{npc: smallest node count that picks it}, for every npc above 8."""
        out, npc = {}, self.t_npc
        while npc > 8:
            out[npc] = self.first_n(lambda n, v=npc: self.pick_npc(n) >= v)
            npc >>= 1
        return out

    def wide_threshold(self):
        return self.first_n(lambda n: self.wide(n, 0))

    def deep_fwd_loop_threshold(self):
        """Smallest node count whose DEEP forward has more tiles than CTAs."""
        return self.first_n(lambda n: self.tiles(n) > self.n_sms * self.DEEP_FWD_PER_SM)

    def deep_src_loop_threshold(self):
        return self.first_n(lambda n: self.tiles(n) > self.n_sms * self.DEEP_SRC_PER_SM)


def test_route_constants_parse():
    R = Routes.parse()
    assert (R.t_npc, R.fwd_cap, R.bwd_cap, R.deep_degree, R.n_sms, R.finish_group) == (64, 1024, 768, 24, 148, 32)
    assert R.caps(10, 0) == (1024, 768, 768)
    assert R.caps(10, 240) == (2048, 768, 1024)


def test_route_model_thresholds():
    R = Routes.parse()
    assert R.npc_thresholds() == {16: 4721, 32: 9441, 64: 18881}
    assert [R.pick_npc(n) for n in (1, 4720, 4721, 9440, 9441, 18880, 18881, 10 ** 6)] == [8, 8, 16, 16, 32, 32, 64, 64]
    assert R.wide_threshold() == 56833
    assert R.deep_fwd_loop_threshold() == 37889
    assert R.deep_src_loop_threshold() == 28417
    loops = lambda n: R.tiles(n) > R.n_sms * R.DEEP_SRC_PER_SM
    assert [loops(n) for n in (3552, 3553, 4720, 4721, 7104, 7105, 9440, 9441, 28416)] == [False, True, True, False,
                                                                                          False, True, True, False, False]
    assert not R.deep(500, 24 * 500 - 1) and R.deep(500, 24 * 500) and not R.deep(0, 0)
    assert R.grids(56833, 3 * 56833) == (740, 888, 888) and R.grids(56832, 0) == (888, 888, 888)
    assert R.grids(37889, 24 * 37889) == (592, 593, 444)
    # the sub-tile walk: a tile whose slots fill the capacity is one sub-tile, one slot more splits it, and a node
    # above the capacity on its own is a hub
    assert R.subtiles([0, 512, 1024], 1024) == ([(0, 2, 1024)], [])
    assert R.subtiles([0, 512, 1025], 1024) == ([(0, 1, 512), (1, 2, 513)], [])
    assert R.subtiles([0, 1, 1026, 1027], 1024) == ([(0, 1, 1), (2, 3, 1)], [1])


def _random_graph(n_nodes, n_edges, seed):
    g = torch.Generator().manual_seed(seed)
    dst = torch.randint(0, n_nodes, (n_edges,), generator=g)
    src = torch.randint(0, n_nodes, (n_edges,), generator=g)
    dst[:n_nodes] = torch.arange(n_nodes)
    return dst, src


@pytest.mark.parametrize("edge_dim", [0, 32])
def test_attention_ref_equals_oracle_block(edge_dim):
    from oracle import gat2_oracle as O
    n, E = 37, 300
    dst, src = _random_graph(n, E, 3)
    gen = torch.Generator().manual_seed(4)
    leaves = [torch.randn(*s, generator=gen, dtype=torch.float64).requires_grad_()
              for s in ((n, 4, 32), (E, edge_dim), (4, 64 + edge_dim))]
    gout, gw = torch.randn(n, 128, generator=gen, dtype=torch.float64), torch.randn(n, 4, generator=gen, dtype=torch.float64)
    grads = []
    for fn in (lambda *a: attention_ref(*a, n)[:2], O.attention_block):
        out, w = fn(leaves[0], dst, src, leaves[1], leaves[2])
        gr = torch.autograd.grad((out * gout).sum() + (w * gw).sum(), leaves)
        grads.append((out, w) + gr)
    for a, b in zip(*grads):
        assert torch.allclose(a, b, rtol=1e-13, atol=1e-13)


def test_attention_ref_nodes_without_edges():
    n = 12
    dst = torch.tensor([0, 0, 1, 3, 3, 3, 5, 2, 1])       # nodes 4 and 6..11 have no incoming edge
    src = torch.tensor([1, 2, 3, 0, 4, 5, 7, 9, 0])
    gen = torch.Generator().manual_seed(1)
    h = torch.randn(n, 4, 32, generator=gen, dtype=torch.float64)
    alpha = torch.randn(4, 64, generator=gen, dtype=torch.float64)
    out, w, z = attention_ref(h, dst, src, torch.zeros(9, 0, dtype=torch.float64), alpha, n)
    assert out.shape == (n, 128) and w.shape == (n, 4) and z.shape == (9, 4)
    no_in = torch.ones(n, dtype=torch.bool)
    no_in[dst] = False
    assert no_in.sum() == 7 and torch.equal(out[no_in], torch.zeros(7, 128, dtype=torch.float64))
    assert torch.allclose(w.sum(0), torch.full((4,), float(n - 7), dtype=torch.float64))   # each target's p sums to 1
    no_out = torch.ones(n, dtype=torch.bool)
    no_out[src] = False
    assert torch.equal(w[no_out], torch.zeros(int(no_out.sum()), 4, dtype=torch.float64))


# ------------------------------------------------------------------------------------------------
# graphs with prescribed in- and out-degrees
@dataclass
class Case:
    n: int
    dst: torch.Tensor      # int64 [E], input edge order
    src: torch.Tensor
    claims: dict           # description -> bool, evaluated from the route model when the case is built

    @property
    def E(self):
        return self.dst.numel()


def _balance(deg, total, free, gen):
    """Move the sum of ``deg`` to ``total`` one unit at a time on ``free`` nodes, keeping them >= 1."""
    deg = deg.clone()
    while (diff := total - int(deg.sum())) != 0:
        cand = (free & (deg > 1)) if diff < 0 else free
        idx = cand.nonzero().flatten()
        idx = idx[torch.randperm(idx.numel(), generator=gen)[:abs(diff)]]
        deg[idx] += 1 if diff > 0 else -1
    return deg


def _from_degrees(n, seed, base=(1, 5), in_fixed=None, out_fixed=None, total=None):
    """A graph of ``n`` nodes whose in- and out-degrees are ``base``-uniform except for the nodes of ``in_fixed`` /
    ``out_fixed`` ({node: degree}); the two degree sums are balanced (to ``total`` if given) on the other nodes, and
    sources are paired with destinations at random."""
    gen = torch.Generator().manual_seed(seed)
    degs = []
    for fixed in (in_fixed or {}, out_fixed or {}):
        deg = torch.randint(base[0], base[1] + 1, (n,), generator=gen)
        free = torch.ones(n, dtype=torch.bool)
        for node, d in fixed.items():
            deg[node] = d
            free[node] = False
        degs.append((deg, free))
    (din, fin), (dout, fout) = degs
    if total is not None:
        din = _balance(din, total, fin, gen)
    dout = _balance(dout, int(din.sum()), fout, gen)
    nodes = torch.arange(n)
    dst = torch.repeat_interleave(nodes, din)
    src = torch.repeat_interleave(nodes, dout)
    src = src[torch.randperm(src.numel(), generator=gen)]
    perm = torch.randperm(dst.numel(), generator=gen)
    return dst[perm].contiguous(), src[perm].contiguous()


def _rowptr(index, n):
    return torch.cat([torch.zeros(1, dtype=torch.long), torch.bincount(index, minlength=n).cumsum(0)])


def _route_facts(R, n, dst, src):
    """What the route model says a graph does in each kernel."""
    E = dst.numel()
    fcap, dcap, scap = R.caps(n, E)
    rp, rrp = _rowptr(dst, n), _rowptr(src, n)
    f = dict(deep=R.deep(n, E), wide=R.wide(n, E), npc=R.pick_npc(n), tiles=R.tiles(n), grids=R.grids(n, E),
             in_deg=torch.bincount(dst, minlength=n), out_deg=torch.bincount(src, minlength=n))
    f["fwd"], f["dst"], f["src"] = R.subtiles(rp, fcap), R.subtiles(rp, dcap), R.subtiles(rrp, scap)
    f["caps"] = (fcap, dcap, scap)
    return f


def _spread(total, k):
    """k degrees that sum to total, as even as possible, the larger ones last."""
    return [total // k + (1 if i >= k - total % k else 0) for i in range(k)]


def _case_no_edges_nodes(R):
    n = 200
    npc = R.pick_npc(n)
    t0 = 8 * npc                                   # a whole tile of nodes without an incoming edge
    zero_in = [5, 17, 33] + list(range(t0, t0 + npc)) + list(range(n - 5, n))
    zero_out = [3, 40, 41, 100, n - 1]
    dst, src = _from_degrees(n, 21, (1, 6), {v: 0 for v in zero_in}, {v: 0 for v in zero_out})
    f = _route_facts(R, n, dst, src)
    ind, outd = f["in_deg"], f["out_deg"]
    claims = {"one node per warp (npc 8)": f["npc"] == 8,
              "an interior node without incoming edges": bool((ind[1:t0] == 0).any()),
              "a whole tile without incoming edges": bool((ind[t0:t0 + npc] == 0).all()) and t0 % npc == 0,
              "trailing nodes without incoming edges": int(ind[-1]) == 0,
              "sources without outgoing edges": bool((outd == 0).any()),
              "no hub": not f["fwd"][1] and not f["dst"][1] and not f["src"][1]}
    return Case(n, dst, src, claims)


def _case_edgeless(R):
    n = 50
    e = torch.zeros(0, dtype=torch.long)
    return Case(n, e, e.clone(), {"nodes without any edge": n > 0})


def _case_hubs(R):
    n = 3000
    npc = R.pick_npc(n)
    fc, bc = R.fwd_cap, R.bwd_cap
    tile_first = 250 * npc
    in_fixed = {10: bc, 11: bc + 1, 1500: fc, 1501: fc + 1, tile_first: fc + 1, n - 1: fc + 1}
    out_fixed = {100: bc, 101: bc + 1, 8 * npc: 2 * bc, n - 1: bc + 1}
    dst, src = _from_degrees(n, 22, (1, 7), in_fixed, out_fixed)
    f = _route_facts(R, n, dst, src)
    fwd_hubs, dst_hubs, src_hubs = set(f["fwd"][1]), set(f["dst"][1]), set(f["src"][1])
    claims = {"not deep": not f["deep"], "not wide": not f["wide"],
              "forward hubs are the nodes above the forward cap": fwd_hubs == {1501, tile_first, n - 1},
              "forward hub at the first node of a tile": tile_first % npc == 0 and tile_first in fwd_hubs,
              "forward hub at the last node": n - 1 in fwd_hubs,
              "forward sub-tile of exactly the cap (in-degree = cap)": any(s == fc for _, _, s in f["fwd"][0]),
              "destination pass: in-degree = cap on the tile path, cap + 1 a hub": 10 not in dst_hubs and 11 in dst_hubs,
              "source pass: out-degree = cap on the tile path, cap + 1 a hub": 100 not in src_hubs and 101 in src_hubs,
              "max in-degree = forward cap + 1": int(f["in_deg"].max()) == fc + 1}
    return Case(n, dst, src, claims)


def _case_slot_totals(R):
    n = 800
    npc = R.pick_npc(n)
    fc, bc = R.fwd_cap, R.bwd_cap
    in_tiles = {10: fc, 20: fc + 1, 30: bc, 40: bc + 1}
    out_tiles = {50: bc, 60: bc + 1}
    in_fixed, out_fixed = {}, {}
    for fixed, tiles in ((in_fixed, in_tiles), (out_fixed, out_tiles)):
        for t, total in tiles.items():
            fixed.update({t * npc + i: d for i, d in enumerate(_spread(total, npc))})
    dst, src = _from_degrees(n, 23, (1, 5), in_fixed, out_fixed)
    f = _route_facts(R, n, dst, src)

    def tile_subs(kernel, t):
        return [s for s in f[kernel][0] if t * npc <= s[0] < (t + 1) * npc]
    claims = {"npc 8, not deep": npc == 8 and not f["deep"], "no hub": not (f["fwd"][1] or f["dst"][1] or f["src"][1]),
              "forward: a tile of exactly cap slots is one sub-tile": tile_subs("fwd", 10) == [(10 * npc, 11 * npc, fc)],
              "forward: cap + 1 slots split the tile": len(tile_subs("fwd", 20)) == 2,
              "destination pass: a tile of exactly cap slots is one sub-tile": tile_subs("dst", 30) == [(30 * npc, 31 * npc, bc)],
              "destination pass: cap + 1 slots split the tile": len(tile_subs("dst", 40)) == 2,
              "source pass: a tile of exactly cap slots is one sub-tile": tile_subs("src", 50) == [(50 * npc, 51 * npc, bc)],
              "source pass: cap + 1 slots split the tile": len(tile_subs("src", 60)) == 2}
    return Case(n, dst, src, claims)


def _case_deep_hubs(R):
    n = 600
    fc2, bc, sc = R.fwd_deep_factor * R.fwd_cap, R.bwd_cap, R.src_deep_cap
    mid = (R.fwd_cap + fc2) // 2
    in_fixed = {10: bc, 11: bc + 1, 100: fc2, 101: fc2 + 1, n - 1: mid}
    out_fixed = {200: sc, 201: sc + 1, 300: 0}
    dst, src = _from_degrees(n, 24, (20, 40), in_fixed, out_fixed)
    f = _route_facts(R, n, dst, src)
    fwd_hubs, dst_hubs, src_hubs = set(f["fwd"][1]), set(f["dst"][1]), set(f["src"][1])
    claims = {"deep": f["deep"], "forward hub only above the DEEP cap": fwd_hubs == {101},
              "DEEP forward tile path for in-degrees above FWD_CAP": R.fwd_cap < mid <= fc2 and n - 1 not in fwd_hubs,
              "DEEP forward sub-tile of exactly the cap": any(s == fc2 for _, _, s in f["fwd"][0]),
              "destination pass: in-degree = cap on the tile path, cap + 1 a hub": 10 not in dst_hubs and 11 in dst_hubs,
              "DEEP source pass: out-degree = cap on the tile path, cap + 1 a hub": 200 not in src_hubs and 201 in src_hubs}
    return Case(n, dst, src, claims)


def _case_deep_switch(R, below):
    n = 500
    hub = 250
    mid = R.fwd_cap + R.fwd_cap // 2      # a hub of the plain forward, on the tile path of the DEEP one
    dst, src = _from_degrees(n, 25, (16, 32), {hub: mid}, {}, total=R.deep_degree * n)
    if below:                             # drop one edge whose target keeps more than one
        keep = torch.ones(dst.numel(), dtype=torch.bool)
        keep[int(((dst != hub) & (torch.bincount(dst, minlength=n)[dst] > 1)).nonzero()[0])] = False
        dst, src = dst[keep].contiguous(), src[keep].contiguous()
    f = _route_facts(R, n, dst, src)
    claims = {"edges = DEEP degree x nodes" + (" - 1" if below else ""): dst.numel() == R.deep_degree * n - below,
              "deep" if not below else "not deep": f["deep"] != below,
              "the in-degree-%d node is a forward hub only without DEEP" % mid: (hub in f["fwd"][1]) == below}
    return Case(n, dst, src, claims)


def _case_npc(R, npc, below):
    t = R.npc_thresholds()[npc]
    n = t - 1 if below else t
    dst, src = _from_degrees(n, 26 + npc, (1, 5))
    want = npc // 2 if below else npc
    return Case(n, dst, src, {f"npc {want} at {n} nodes": R.pick_npc(n) == want, "not deep": not R.deep(n, dst.numel())})


def _case_loop_wide(R):
    n = R.wide_threshold() * 21 // 20           # ~5 % above the WIDE threshold
    fc, bc = R.fwd_cap, R.bwd_cap
    dst, src = _from_degrees(n, 27, (1, 5), {0: fc + 1, n // 2: 2 * fc, n - 1: bc + 1}, {7: bc + 1, n - 1: 2 * bc})
    f = _route_facts(R, n, dst, src)
    gf, gd, gs = f["grids"]
    groups = -(-gd // R.finish_group)
    claims = {"wide": f["wide"], "forward tiles > grid": f["tiles"] > gf,
              "destination pass tiles > grid": f["tiles"] > gd, "source pass tiles > grid": f["tiles"] > gs,
              "cta_finish over %d CTAs: %d groups, the last partial" % (gd, groups):
                  gd == R.n_sms * R.DST_PER_SM and gd % R.finish_group != 0,
              "hubs in every kernel": all(f[k][1] for k in ("fwd", "dst", "src"))}
    return Case(n, dst, src, claims)


def _case_loop_deep(R):
    n = R.deep_fwd_loop_threshold() * 41 // 40   # ~2.5 % above the DEEP forward looping threshold
    dst, src = _from_degrees(n, 28, (16, 32), {5: R.fwd_deep_factor * R.fwd_cap + 1}, {6: R.src_deep_cap + 1},
                             total=R.deep_degree * n)
    f = _route_facts(R, n, dst, src)
    gf, gd, gs = f["grids"]
    claims = {"deep": f["deep"], "DEEP forward tiles > grid": f["tiles"] > gf,
              "DEEP source pass tiles > grid": f["tiles"] > gs, "hubs in the forward and the source pass":
                  bool(f["fwd"][1]) and bool(f["src"][1])}
    return Case(n, dst, src, claims)


_BUILDERS = {
    "no_edges_nodes": _case_no_edges_nodes,
    "edgeless": _case_edgeless,
    "hubs": _case_hubs,
    "slot_totals": _case_slot_totals,
    "deep_hubs": _case_deep_hubs,
    "deep_switch_below": lambda R: _case_deep_switch(R, True),
    "deep_switch_at": lambda R: _case_deep_switch(R, False),
    **{f"npc{npc}_{side}": (lambda R, v=npc, b=(side == "below"): _case_npc(R, v, b))
       for npc in (16, 32, 64) for side in ("below", "at")},
    "loop_wide": _case_loop_wide,
    "loop_deep": _case_loop_deep,
}
LARGE = ("loop_wide", "loop_deep")
MODES = ("none", "affine1", "affine6", "table")


@functools.lru_cache(maxsize=None)
def case(name):
    c = _BUILDERS[name](Routes.parse())
    failed = [k for k, v in c.claims.items() if not v]
    assert not failed, f"{name}: the graph does not take the route it claims: {failed}"
    return c


# ------------------------------------------------------------------------------------------------
# the kernels, traced
def _traced(fn):
    """Run fn() under torch.profiler; returns (fn's result, [(kernel name, grid x)] in launch order)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    kernels = sorted((e for e in events if e.get("cat") == "kernel"), key=lambda e: e["ts"])
    return res, [(e["name"], int(e["args"]["grid"][0])) for e in kernels]


def _expect_launches(R, c, mode_id, launches, backward=True):
    """The instantiations and grids the route model predicts, checked against the trace."""
    from fragnet_b200 import ops
    deep, wide = R.deep(c.n, c.E), R.wide(c.n, c.E)
    b = lambda v: "true" if v else "false"
    gf, gd, gs = R.grids(c.n, c.E)
    dmode = mode_id if mode_id in (ops.EDGE_AFFINE1, ops.EDGE_AFFINE6) else ops.EDGE_NONE
    want = [(f"k_gat_fwd_tiled<{mode_id}, {b(deep)}, {b(wide)}>", gf)]
    if backward:
        want += [(f"k_gat_bwd_dst_tiled<{dmode}, false, {b(deep)}>", gd), (f"k_gat_bwd_src_tiled<{b(deep)}>", gs)]
    got = [(name, grid) for name, grid in launches if "k_gat_" in name]
    assert len(got) == len(want), (got, want)
    for (name, grid), (w, wg) in zip(got, want):
        assert w in name and grid == wg, (name, grid, w, wg)
    return [w for w, _ in want]


def _errors_ok(errs, name):
    tol = {"out": FP32_REL_TOL, "by_source": FP32_REL_TOL, "d_bias": BIAS_TOL}
    bad = {k: v for k, v in errs.items() if not v <= tol.get(k, GRAD_TOL)}
    print(f"{name}: " + ", ".join(f"{k} {v:.1e}" for k, v in errs.items()))
    assert not bad, f"{name}: {bad}"


def _scratch_clean():
    from fragnet_b200 import ops
    return int(ops.scratch(torch.device("cuda", torch.cuda.current_device()))[:256].view(torch.int32).abs().sum()) == 0


def _check_case(name, mode):
    from fragnet_b200 import ops
    R = Routes.parse()
    c = case(name)
    n, E = c.n, c.E
    dev = torch.device("cuda")
    gen = torch.Generator().manual_seed(1000 + n + E)
    rnd = lambda *shape: torch.randn(*shape, generator=gen)
    leaf = lambda t: t.to(dev, torch.float64).requires_grad_()
    dst, src = c.dst.to(dev), c.src.to(dev)
    h32, gout32 = rnd(n, 128).to(dev), rnd(n, 128).to(dev)
    stride, off_t, off_e, off_s = (96, 0, 32, 64) if mode != "table" else (192, 0, 32, 160)
    alpha32 = (rnd(4, stride) * 0.3).to(dev)
    h, alpha = leaf(h32), leaf(alpha32)
    graph = ops.csr_build(dst, src, n)
    mode_id = dict(none=ops.EDGE_NONE, affine1=ops.EDGE_AFFINE1, affine6=ops.EDGE_AFFINE6, table=ops.EDGE_TABLE)[mode]
    fwd_kw, bwd_kw, leaves = {}, {}, {}
    if mode == "none":
        a_used = torch.cat([alpha[:, 0:32], alpha[:, 64:96]], dim=1)
        edge_vec = torch.zeros(E, 0, dtype=torch.float64, device=dev)
    elif mode in ("affine1", "affine6"):
        k = 1 if mode == "affine1" else 6
        attr = rnd(E, k).to(dev)
        We32, be32 = (rnd(32, k) * 0.5).to(dev), rnd(32).to(dev)
        leaves = dict(We=leaf(We32), be=leaf(be32))
        edge_vec, a_used = F.linear(attr.double(), leaves["We"], leaves["be"]), alpha
        graph.attr = ops.gather_rows(attr, graph.eid, E)
        fwd_kw = dict(We=We32, be=be32, alpha_e=alpha32[:, off_e:], alpha_stride=stride)
        bwd_kw = dict(We=We32, be=be32)
    else:
        feat32 = rnd(E, 128).to(dev)
        leaves = dict(feat=leaf(feat32))
        edge_vec, a_used = leaves["feat"], alpha
        fwd_kw = dict(table=(feat32 @ alpha32[:, 32:160].t()).contiguous())
    gbase = rnd(E, 128).to(dev) if mode == "table" else None

    out_ref, w_ref, z = attention_ref(h.view(n, 4, 32), dst, src, edge_vec, a_used, n)
    (out_ref * gout32.double()).sum().backward()
    dz_ref = z.grad if z.grad is not None else torch.zeros_like(z)

    S = ops.node_scalars(h32, alpha32, stride, off_t, off_s)

    def run():
        out, _, p, _ = ops.gat_fwd_tiled(graph, h32, S, mode_id, **fwd_kw)
        w = ops.attn_by_source(graph, p)
        d_alpha = torch.full((4, stride), float("nan"), device=dev)
        dh, dz, db, dWe, dbe = ops.gat_bwd_tiled(graph, h32, gout32, p, mode_id, alpha32, stride, off_t, off_e, off_s,
                                                 d_alpha, want_bias_grad=True, **bwd_kw)
        r = dict(out=out, p=p, by_source=w, dh=dh, dz=dz, d_bias=db, dWe=dWe, dbe=dbe)
        if mode == "table":
            r["g_feat"] = ops.edge_table_bwd_fused(graph, dz, feat32, alpha32, stride, off_e, d_alpha, g_base=gbase)
        r["d_alpha"] = d_alpha
        return r

    r, launches = _traced(run)
    assert _scratch_clean()            # the arrival counters are back at zero for the next launch on the stream
    route = _expect_launches(R, c, mode_id, launches)
    r2 = run()
    for k, v in r.items():             # launch-to-launch bitwise reproducible (NaN: d_alpha slices left unwritten)
        assert (v is None) == (r2[k] is None) and (v is None or torch.equal(v.nan_to_num(), r2[k].nan_to_num())), k
    assert _scratch_clean()

    slot_of_eid = graph.slot_of_eid[:E].long()
    errs = dict(out=rel_err(r["out"], out_ref), by_source=rel_err(r["by_source"], w_ref),
                dz=rel_err(r["dz"].index_select(0, slot_of_eid), dz_ref), dh=rel_err(r["dh"], h.grad),
                d_bias=rel_err(r["d_bias"], h.grad.sum(0)))
    if mode == "none":      # the edge slice of d_alpha is not written without an edge term
        errs["d_alpha"] = max(rel_err(r["d_alpha"][:, 0:32], alpha.grad[:, 0:32]),
                              rel_err(r["d_alpha"][:, 64:96], alpha.grad[:, 64:96]))
    else:
        errs["d_alpha"] = rel_err(r["d_alpha"], alpha.grad)
    if mode.startswith("affine"):
        errs["dWe"], errs["dbe"] = rel_err(r["dWe"], leaves["We"].grad), rel_err(r["dbe"], leaves["be"].grad)
    if mode == "table":
        errs["g_feat"] = rel_err(r["g_feat"] - gbase, leaves["feat"].grad)
    f = _route_facts(R, n, c.dst, c.src)
    print(f"{name}/{mode}: n {n} E {E} npc {f['npc']} tiles {f['tiles']} grids {f['grids']} hubs "
          f"{tuple(len(f[k][1]) for k in ('fwd', 'dst', 'src'))} {route}")
    _errors_ok(errs, f"{name}/{mode}")


SMALL = [k for k in _BUILDERS if k not in LARGE]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", SMALL)
def test_attention_route(name, mode):
    _check_case(name, mode)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["none", "affine6"])     # affine6: coefficient gradients accumulated per CTA over tiles
@pytest.mark.parametrize("name", LARGE)
def test_attention_route_looping_ctas(name, mode):
    _check_case(name, mode)


# ------------------------------------------------------------------------------------------------
# large logits in exact arithmetic: the max subtraction of all three softmax codes, logits exactly 0, ties
def _exact_scalars(n, seed):
    """S [n,8] of multiples of 1/8, so that every logit St + Ss is exact in fp32: target terms mostly in +-300 (every
    segment shifted far beyond exp's range, both signs), source terms mostly in +-4 (so a segment's softmax is not one
    edge; 65 values, so segments have ties at their max), and a quarter of each on the other grid so that some
    logits are exactly 0."""
    g = torch.Generator().manual_seed(seed)
    big = lambda *s: torch.randint(-2400, 2401, s, generator=g).float() / 8
    small = lambda *s: torch.randint(-32, 33, s, generator=g).float() / 8
    pick = torch.rand(n, 1, generator=g) < 0.25
    st = torch.where(pick, small(n, 4), big(n, 4))
    ss = torch.where(pick, big(n, 4), small(n, 4))
    return torch.cat([st, ss], dim=1)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["hubs", "deep_hubs", "loop_wide"])
def test_attention_large_exact_logits(name):
    from fragnet_b200 import ops
    R = Routes.parse()
    c = case(name)
    n, E = c.n, c.E
    dev = torch.device("cuda")
    gen = torch.Generator().manual_seed(7 + n)
    h32, gout32 = torch.randn(n, 128, generator=gen).to(dev), torch.randn(n, 128, generator=gen).to(dev)
    alpha32 = (torch.randn(4, 96, generator=gen) * 0.3).to(dev)
    S32 = _exact_scalars(n, n).to(dev)
    dst, src = c.dst.to(dev), c.src.to(dev)
    z32 = S32[dst, :4] + S32[src, 4:]
    z64 = S32.double()[dst, :4] + S32.double()[src, 4:]
    assert torch.equal(z32.double(), z64)                                  # the logits are exact in fp32
    seg_max = torch.full((n, 4), float("-inf"), device=dev, dtype=torch.float64).scatter_reduce(
        0, dst[:, None].expand(-1, 4), z64, "amax")
    at_max = torch.zeros(n, 4, device=dev).index_add_(0, dst, (z64 == seg_max[dst]).float())
    assert bool((z64 == 0).any()) and bool((at_max > 1).any())          # zeros, and ties at a segment's max
    assert float(z64.abs().max()) > 200 and float(seg_max.min()) < -88 and float(seg_max.max()) > 88

    graph = ops.csr_build(dst, src, n)
    h, S = h32.double().requires_grad_(), S32.double().requires_grad_()
    out_ref, w_ref, z = attention_ref(h.view(n, 4, 32), dst, src, torch.zeros(E, 0, dtype=torch.float64, device=dev),
                                      torch.zeros(4, 0, dtype=torch.float64, device=dev), n, S=S)
    (out_ref * gout32.double()).sum().backward()
    # chain rule through the given S: the kernels take S = <h, alpha_t> | <h, alpha_s> as what it would have been
    a64 = alpha32.double()
    at, as_ = a64[:, 0:32], a64[:, 64:96]
    hv = h.detach().view(n, 4, 32)
    dh_ref = h.grad + (S.grad[:, :4, None] * at + S.grad[:, 4:, None] * as_).reshape(n, 128)
    dat_ref = (S.grad[:, :4, None] * hv).sum(0)
    das_ref = (S.grad[:, 4:, None] * hv).sum(0)

    def run():
        out, _, p, _ = ops.gat_fwd_tiled(graph, h32, S32, ops.EDGE_NONE)
        d_alpha = torch.full((4, 96), float("nan"), device=dev)
        dh, dz, db, _, _ = ops.gat_bwd_tiled(graph, h32, gout32, p, ops.EDGE_NONE, alpha32, 96, 0, 32, 64, d_alpha,
                                             want_bias_grad=True)
        return dict(out=out, p=p, by_source=ops.attn_by_source(graph, p), dh=dh, dz=dz, d_bias=db, d_alpha=d_alpha)

    r, launches = _traced(run)
    route = _expect_launches(R, c, ops.EDGE_NONE, launches)
    r2 = run()
    assert all(torch.equal(v.nan_to_num(), r2[k].nan_to_num()) for k, v in r.items())
    assert _scratch_clean()
    errs = dict(out=rel_err(r["out"], out_ref), by_source=rel_err(r["by_source"], w_ref),
                dz=rel_err(r["dz"].index_select(0, graph.slot_of_eid[:E].long()), z.grad),
                dh=rel_err(r["dh"], dh_ref), d_bias=rel_err(r["d_bias"], dh_ref.sum(0)),
                d_alpha=max(rel_err(r["d_alpha"][:, 0:32], dat_ref), rel_err(r["d_alpha"][:, 64:96], das_ref)))
    print(f"exact/{name}: {route}")
    _errors_ok(errs, f"exact logits/{name}")


# ------------------------------------------------------------------------------------------------
# the fused forward epilogue on hub rows and in the WIDE instantiation
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["hubs", "loop_wide"])
def test_fused_epilogue_on_hub_rows(name):
    from fragnet_b200 import ops
    R = Routes.parse()
    c = case(name)
    n = c.n
    hubs = _route_facts(R, n, c.dst, c.src)["fwd"][1]
    gen = torch.Generator().manual_seed(5 + n)
    h = torch.randn(n, 128, generator=gen).cuda()
    alpha = torch.randn(4, 96, generator=gen).cuda()
    nxt = torch.randn(4, 192, generator=gen).cuda()
    graph = ops.csr_build(c.dst.cuda(), c.src.cuda(), n)
    S = ops.node_scalars(h, alpha, 96, 0, 64)
    mask = (hubs[0], hubs[0] + 2)              # masks one hub row; the other hubs store through the epilogue
    assert any(v >= mask[1] for v in hubs)
    seed, offset, p = 987654, 31, 0.2
    (out, y, _, se), launches = _traced(lambda: ops.gat_fwd_tiled(
        graph, h, S, ops.EDGE_NONE, save_p=False, post=(p, 1, 1, seed, offset), mask=mask, next_alpha=nxt[:, 32:],
        next_alpha_stride=192))
    _expect_launches(R, c, ops.EDGE_NONE, launches, backward=False)
    out0, _, _, _ = ops.gat_fwd_tiled(graph, h, S, ops.EDGE_NONE, save_p=False)
    out0[mask[0]:mask[1]] = 0
    assert torch.equal(out, out0)
    assert torch.equal(y, ops.dropout_relu_fwd(out, p, True, True, seed, offset))
    assert rel_err(se, out.double() @ nxt[:, 32:160].double().t()) <= FP32_REL_TOL
    _, y2, _, _ = ops.gat_fwd_tiled(graph, h, S, ops.EDGE_NONE, save_p=False, want_out=False,
                                    post=(p, 1, 1, seed, offset), mask=mask)
    assert torch.equal(y, y2)
