"""Parity of the node-tiled attention kernels (gat_tiled.cu, through the C ABI) against the CPU oracle block, and
bit-level agreement of their fused epilogues with the standalone kernels they absorb."""
import pytest
import torch
import torch.nn.functional as F

from conftest import FP32_REL_TOL, rel_err

pytestmark = pytest.mark.gpu


def _graph(n_nodes, n_edges, seed, hub_edges=0, band=0):
    g = torch.Generator().manual_seed(seed)
    dst = torch.randint(0, n_nodes, (n_edges,), generator=g)
    if band:     # block-diagonal-like locality (sources within +-band of the destination), as in batched molecules
        src = (dst + torch.randint(-band, band + 1, (n_edges,), generator=g)).clamp_(0, n_nodes - 1)
    else:
        src = torch.randint(0, n_nodes, (n_edges,), generator=g)
    dst[:n_nodes] = torch.arange(n_nodes)           # every node is a target (reference requirement, App. B)
    if hub_edges:
        dst[n_nodes:n_nodes + hub_edges] = 1        # one destination segment far above the tile capacity
        src[n_nodes + hub_edges:n_nodes + 2 * hub_edges] = 2   # and one such source segment (reverse CSR)
    return dst, src


CASES = [
    (20000, 130000, -30),  # 64-node tiles with local sources (negative = band width)
    (20000, 130000, -100), # wider band: each tile's sources span a longer id range
    (40, 200, 0),          # one partial tile
    (64, 3000, 0),         # one tile, several sub-tiles (3000 slots > capacity)
    (50, 6000, 2500),      # hub paths: in-degree and out-degree above the capacity of a sub-tile
    (3000, 20000, 0),      # many tiles
    (1, 1, 0),
]


@pytest.mark.parametrize("mode", ["none", "affine1", "affine6", "table"])
@pytest.mark.parametrize("n_nodes,n_edges,hub", CASES)
def test_tiled_attention_forward_backward(mode, n_nodes, n_edges, hub):
    from fragnet_b200 import ops
    from oracle import gat2_oracle as O
    dst, src = _graph(n_nodes, n_edges, 11 + n_nodes, max(hub, 0), band=max(-hub, 0))
    # The reference side runs in float64 (the same reference algorithm, oracle/gat2_oracle.py): the check is "within
    # 1e-5 of the exact result", independent of the summation order / thread count of the host's fp32 kernels.
    gen = torch.Generator().manual_seed(n_edges)
    rnd = lambda *shape: torch.randn(*shape, generator=gen)
    leaf = lambda t: t.double().requires_grad_()
    h32 = rnd(n_nodes, 128)
    h = leaf(h32)
    gout = rnd(n_nodes, 128)
    graph = ops.csr_build(dst.cuda(), src.cuda(), n_nodes)
    assert torch.equal(graph.row.cpu().long(), dst[graph.eid.cpu().long()])     # row[slot] = destination of the slot
    stride, off_t, off_e, off_s = (96, 0, 32, 64) if mode != "table" else (192, 0, 32, 160)
    alpha32 = rnd(4, stride) * 0.3
    alpha = leaf(alpha32)
    We = be = feat = None
    fwd_kw, bwd_kw = {}, {}
    if mode == "none":
        a_used = torch.cat([alpha[:, 0:32], alpha[:, 64:96]], dim=1)
        edge_vec = torch.zeros(n_edges, 0, dtype=torch.float64)
    elif mode in ("affine1", "affine6"):
        k = 1 if mode == "affine1" else 6
        attr = rnd(n_edges, k)
        We32, be32 = rnd(32, k) * 0.5, rnd(32)
        We, be = leaf(We32), leaf(be32)
        edge_vec, a_used = F.linear(attr.double(), We, be), alpha
        graph.attr = ops.gather_rows(attr.cuda(), graph.eid, n_edges)
        ac_full = alpha32.cuda()
        fwd_kw = dict(We=We32.cuda(), be=be32.cuda(), alpha_e=ac_full[:, off_e:], alpha_stride=stride)
        bwd_kw = dict(We=fwd_kw["We"], be=fwd_kw["be"])
    else:
        feat32 = rnd(n_edges, 128)
        feat = leaf(feat32)
        edge_vec, a_used = feat, alpha
        fwd_kw = dict(table=(feat32 @ alpha32[:, 32:160].t()).contiguous().cuda())
    out_ref, w_ref = O.attention_block(h.view(n_nodes, 4, 32), dst, src, edge_vec, a_used)
    (out_ref * gout.double()).sum().backward()

    hc, ac = h32.cuda(), alpha32.cuda()
    S = ops.node_scalars(hc, ac, stride, off_t, off_s)
    mode_id = dict(none=ops.EDGE_NONE, affine1=ops.EDGE_AFFINE1, affine6=ops.EDGE_AFFINE6, table=ops.EDGE_TABLE)[mode]
    out, _, p, _ = ops.gat_fwd_tiled(graph, hc, S, mode_id, **fwd_kw)
    out2, _, p2, _ = ops.gat_fwd_tiled(graph, hc, S, mode_id, **fwd_kw)
    assert torch.equal(out, out2) and torch.equal(p, p2)          # launch-to-launch bitwise reproducible
    assert rel_err(out, out_ref) <= FP32_REL_TOL
    assert rel_err(ops.attn_by_source(graph, p), w_ref) <= FP32_REL_TOL
    d_alpha = torch.full((4, stride), float("nan"), device="cuda")
    dh, dz, dbias, dWe, dbe = ops.gat_bwd_tiled(graph, hc, gout.cuda(), p, mode_id, ac, stride, off_t, off_e, off_s,
                                                d_alpha, want_bias_grad=True, **bwd_kw)
    gtol = 2e-5      # gradients: sums of O(100..1000) fp32 products in a different (fixed) order
    assert rel_err(dh, h.grad) <= gtol
    assert rel_err(dbias, h.grad.sum(0)) <= 2e-4
    if mode.startswith("affine"):
        assert rel_err(dWe, We.grad) <= gtol and rel_err(dbe, be.grad) <= gtol
    if mode == "table":
        gbase = torch.randn(n_edges, 128, generator=gen).cuda()
        g_feat = ops.edge_table_bwd_fused(graph, dz, feat32.cuda(), ac, stride, off_e, d_alpha, g_base=gbase)
        assert rel_err(g_feat - gbase, feat.grad) <= gtol
    if mode == "none":
        want = alpha.grad
        assert rel_err(d_alpha[:, 0:32], want[:, 0:32]) <= gtol and rel_err(d_alpha[:, 64:96], want[:, 64:96]) <= gtol
    else:
        assert rel_err(d_alpha, alpha.grad) <= gtol
    # the arrival counters are back at zero, so the next launch on the stream starts clean
    assert int(ops.scratch(torch.device("cuda", 0))[:256].view(torch.int32).abs().sum()) == 0


def test_tiled_backward_is_deterministic():
    from fragnet_b200 import ops
    from oracle import gat2_oracle as O
    dst, src = _graph(5000, 40000, 5)
    gen = torch.Generator().manual_seed(9)
    h32 = torch.randn(5000, 128, generator=gen)
    go = torch.randn(5000, 128, generator=gen).cuda()
    alpha32 = torch.randn(4, 96, generator=gen) * 0.3
    h, alpha = h32.cuda(), alpha32.cuda()
    graph = ops.csr_build(dst.cuda(), src.cuda(), 5000)
    S = ops.node_scalars(h, alpha, 96, 0, 64)
    out, _, p, _ = ops.gat_fwd_tiled(graph, h, S, ops.EDGE_NONE)
    a64 = alpha32.double()
    out_ref, w_ref = O.attention_block(h32.double().view(5000, 4, 32), dst, src,
                                       torch.zeros(40000, 0, dtype=torch.float64),
                                       torch.cat([a64[:, 0:32], a64[:, 64:96]], dim=1))
    assert rel_err(out, out_ref) <= FP32_REL_TOL
    assert rel_err(ops.attn_by_source(graph, p), w_ref) <= FP32_REL_TOL
    runs = []
    for _ in range(3):
        d_alpha = torch.zeros(4, 96, device="cuda")
        dh, dz, db, _, _ = ops.gat_bwd_tiled(graph, h, go, p, ops.EDGE_NONE, alpha, 96, 0, 32, 64, d_alpha,
                                             want_bias_grad=True)
        runs.append((dh.clone(), dz.clone(), db.clone(), d_alpha.clone()))
    for r in runs[1:]:
        assert all(torch.equal(a, b) for a, b in zip(r, runs[0]))


def test_fused_post_activation_equals_standalone_dropout_relu():
    from fragnet_b200 import ops
    dst, src = _graph(777, 5000, 3)
    gen = torch.Generator().manual_seed(1)
    h = torch.randn(777, 128, generator=gen).cuda()
    alpha = torch.randn(4, 96, generator=gen).cuda()
    nxt = torch.randn(4, 192, generator=gen).cuda()
    graph = ops.csr_build(dst.cuda(), src.cuda(), 777)
    S = ops.node_scalars(h, alpha, 96, 0, 64)
    seed, offset, p = 1234567, 999, 0.2
    out, y, _, se = ops.gat_fwd_tiled(graph, h, S, ops.EDGE_NONE, save_p=False, post=(p, 1, 1, seed, offset),
                                      mask=(10, 12), next_alpha=nxt[:, 32:], next_alpha_stride=192)
    out0, _, _, _ = ops.gat_fwd_tiled(graph, h, S, ops.EDGE_NONE, save_p=False)
    out0[10:12] = 0
    assert torch.equal(out, out0)                   # masked rows are zero, every other row is unchanged
    assert torch.equal(y, ops.dropout_relu_fwd(out, p, True, True, seed, offset))
    assert rel_err(se, out @ nxt[:, 32:160].t()) <= FP32_REL_TOL
    # y only (inference / non-final layers): identical values without the pre-activation store
    _, y2, _, _ = ops.gat_fwd_tiled(graph, h, S, ops.EDGE_NONE, save_p=False, want_out=False,
                                    post=(p, 1, 1, seed, offset), mask=(10, 12))
    assert torch.equal(y, y2)
    _, y3, _, _ = ops.gat_fwd_tiled(graph, h, S, ops.EDGE_NONE, save_p=False, want_out=False, post=(0.0, 0, 1, 0, 0),
                                    mask=(10, 12))
    assert torch.equal(y3, torch.relu(out))


def test_fused_edge_table_backward_absorbs_dropout_relu_backward():
    from fragnet_b200 import ops
    dst, src = _graph(300, 2000, 8)
    gen = torch.Generator().manual_seed(2)
    graph = ops.csr_build(dst.cuda(), src.cuda(), 300)
    dz = torch.randn(2000, 4, generator=gen).cuda()
    feat = torch.randn(2000, 128, generator=gen).cuda()
    alpha = torch.randn(4, 192, generator=gen).cuda()
    dy = torch.randn(2000, 128, generator=gen).cuda()
    p = 0.25
    y = ops.dropout_relu_fwd(feat, p, True, True, 42, 7)
    d1, d2 = torch.zeros(4, 192, device="cuda"), torch.zeros(4, 192, device="cuda")
    base = ops.dropout_relu_bwd(dy, y, p, True)
    want = ops.edge_table_bwd_fused(graph, dz, feat, alpha, 192, 32, d1, g_base=base)
    got = ops.edge_table_bwd_fused(graph, dz, feat, alpha, 192, 32, d2, dy=dy, y=y, post_scale=1.0 / (1.0 - p))
    assert rel_err(got, want) <= 1e-6 and torch.equal(d1, d2)
    ref = base + dz[graph.slot_of_eid.long()] @ alpha[:, 32:160]
    assert rel_err(want, ref) <= FP32_REL_TOL
