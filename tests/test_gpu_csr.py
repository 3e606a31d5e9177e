"""Bit-exact index construction on the GPU (north-star kernel a) against a CPU stable sort."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _cpu_csr(dst, src, n_nodes, self_loops):
    dst, src = dst.clone(), src.clone()
    if self_loops:
        loops = torch.arange(n_nodes, dtype=torch.int64)
        dst, src = torch.cat([dst, loops]), torch.cat([src, loops])
    E = dst.numel()
    order = torch.sort(dst, stable=True).indices
    rowptr = torch.zeros(n_nodes + 1, dtype=torch.int64)
    rowptr[1:] = torch.cumsum(torch.bincount(dst, minlength=n_nodes), 0)
    slot_of_eid = torch.empty(E, dtype=torch.int64)
    slot_of_eid[order] = torch.arange(E)
    rorder = torch.sort(src, stable=True).indices
    rrowptr = torch.zeros(n_nodes + 1, dtype=torch.int64)
    rrowptr[1:] = torch.cumsum(torch.bincount(src, minlength=n_nodes), 0)
    return dict(rowptr=rowptr, col=src[order], eid=order, slot_of_eid=slot_of_eid, rrowptr=rrowptr,
                rslot=slot_of_eid[rorder], rdst=dst[rorder])


def _check(dst, src, n_nodes, self_loops):
    from fragnet_b200 import ops
    g = ops.csr_build(dst.cuda(), src.cuda(), n_nodes, self_loops=self_loops)
    want = _cpu_csr(dst, src, n_nodes, self_loops)
    assert int(g.status.item()) == 0
    for k, w in want.items():
        got = getattr(g, k).cpu().to(torch.int64)
        assert torch.equal(got, w), k


@pytest.mark.parametrize("n_nodes,n_edges,self_loops", [(0, 0, False), (1, 1, False), (7, 0, True), (50, 400, False),
                                                        (50, 400, True), (5000, 40000, True), (3, 5000, False),
                                                        (100000, 650000, False)])
def test_csr_equals_stable_sort(n_nodes, n_edges, self_loops):
    g = torch.Generator().manual_seed(n_nodes + n_edges)
    dst = torch.randint(0, max(n_nodes, 1), (n_edges,), generator=g)
    src = torch.randint(0, max(n_nodes, 1), (n_edges,), generator=g)
    _check(dst, src, n_nodes, self_loops)


def test_csr_on_batched_molecule_graphs():
    from fragnet_b200 import synth
    from fragnet_b200.dataset.data import collate_fn
    b = collate_fn(synth.make_dataset("stress", 3, seed=2) + synth.make_dataset("unimol", 20, seed=3)
                   + [synth.handmade(k) for k in ("two_atom", "ion_pair", "single_frag", "two_frag")])
    na, nb, nfb, nf = b["x_atoms"].shape[0], b["node_features_bonds"].shape[0], b["node_features_fbonds"].shape[0], \
        b["x_frags"].shape[0]
    _check(b["edge_index_bonds_graph"][0], b["edge_index_bonds_graph"][1], nb, False)
    _check(b["edge_index"][1], b["edge_index"][0], na, True)
    _check(b["edge_index_fbonds"][0], b["edge_index_fbonds"][1], nfb, False)
    _check(b["frag_index"][1], b["frag_index"][0], nf, False)


def test_membership_csr_offsets_and_narrowing():
    from fragnet_b200 import ops
    g = torch.Generator().manual_seed(0)
    a2f = torch.randint(0, 37, (900,), generator=g)
    a2f[:37] = torch.arange(37)
    pool = ops.csr_build(a2f.cuda(), None, 37, reverse=False)
    order = torch.sort(a2f, stable=True).indices
    assert torch.equal(pool.col.cpu().long(), order)
    assert torch.equal(pool.rowptr.cpu().long()[1:], torch.cumsum(torch.bincount(a2f, minlength=37), 0))
    batch = torch.sort(torch.randint(0, 64, (2000,), generator=g)).values
    batch[-1] = 63
    off = ops.segment_offsets(batch.cuda(), 64).cpu().long()
    want = torch.searchsorted(batch, torch.arange(65))
    assert torch.equal(off, want)
    assert torch.equal(ops.narrow_index(batch.cuda()).cpu().long(), batch)
    attr = torch.randn(900, 6)
    got = ops.gather_rows(attr.cuda(), pool.col, 900).cpu()
    assert torch.equal(got, attr[order])


def test_out_of_range_index_sets_status():
    from fragnet_b200 import ops
    dst = torch.tensor([0, 1, 9], dtype=torch.int64).cuda()
    src = torch.tensor([1, 0, 1], dtype=torch.int64).cuda()
    g = ops.csr_build(dst, src, 3)
    assert int(g.status.item()) == 1


@pytest.mark.parametrize("shape,n", [("unimol", 40), ("stress", 3), ("esol", 300)])
def test_batch_plan_one_call_equals_stable_sort(shape, n):
    """fnb_batch_plan_build (all five CSRs, attributes, offsets in one call) against the CPU stable sort, bit-exact."""
    from fragnet_b200 import ops, synth
    from fragnet_b200.dataset.data import collate_fn
    b = collate_fn(synth.make_dataset(shape, n, seed=4)
                   + [synth.handmade(k) for k in ("two_atom", "ion_pair", "single_frag", "two_frag")])
    na, nb, nfb, nf = b["x_atoms"].shape[0], b["node_features_bonds"].shape[0], b["node_features_fbonds"].shape[0], \
        b["x_frags"].shape[0]
    bc = {k: v.cuda() for k, v in b.items()}
    plan = ops.build_layer_plan(bc["edge_index"], bc["frag_index"], bc["atom_to_frag_ids"],
                                bc["edge_index_bonds_graph"], bc["edge_attr_bonds"], bc["edge_index_fbonds"],
                                bc["edge_attr_fbonds"], na, nf, nb, nfb, "cuda", bc["batch"], bc["frag_batch"])
    assert int(plan.status.item()) == 0
    specs = [("bond", b["edge_index_bonds_graph"][0], b["edge_index_bonds_graph"][1], nb, False),
             ("atom", b["edge_index"][1], b["edge_index"][0], na, True),
             ("fbond", b["edge_index_fbonds"][0], b["edge_index_fbonds"][1], nfb, False),
             ("frag", b["frag_index"][1], b["frag_index"][0], nf, False)]
    for name, dst, src, nn, loops in specs:
        g = getattr(plan, name)
        want = _cpu_csr(dst, src, nn, loops)
        for k, w in want.items():
            assert torch.equal(getattr(g, k).cpu().to(torch.int64), w), (name, k)
        dst_full = torch.cat([dst, torch.arange(nn)]) if loops else dst
        assert torch.equal(g.row.cpu().long(), dst_full[want["eid"]]), name
    # slot-ordered edge attributes
    assert torch.equal(plan.bond.attr.cpu().view(-1), b["edge_attr_bonds"].view(-1)[plan.bond.eid.cpu().long()])
    assert torch.equal(plan.fbond.attr.cpu(), b["edge_attr_fbonds"][plan.fbond.eid.cpu().long()])
    # membership CSR, narrowing, readout offsets
    a2f = b["atom_to_frag_ids"]
    order = torch.sort(a2f, stable=True).indices
    assert torch.equal(plan.pool.col.cpu().long(), order)
    assert torch.equal(plan.pool.rowptr.cpu().long()[1:], torch.cumsum(torch.bincount(a2f, minlength=nf), 0))
    assert torch.equal(plan.a2f32.cpu().long(), a2f)
    ro = plan.readout
    G = int(b["batch"][-1]) + 1
    assert ro.n_graphs == G
    # the offset arrays are sized by the upper bound n_frags; entries past the last molecule equal the totals
    assert torch.equal(ro.atom_ptr.cpu().long(), torch.searchsorted(b["batch"], torch.arange(nf + 1)))
    assert torch.equal(ro.frag_ptr.cpu().long(), torch.searchsorted(b["frag_batch"], torch.arange(nf + 1)))
    assert torch.equal(ro.batch32.cpu().long(), b["batch"]) and torch.equal(ro.frag_batch32.cpu().long(), b["frag_batch"])


def test_batch_plan_flags_out_of_range_indices():
    from fragnet_b200 import ops, synth
    from fragnet_b200.dataset.data import collate_fn
    b = collate_fn(synth.make_dataset("unimol", 4, seed=1))
    bc = {k: v.cuda() for k, v in b.items()}
    bad = bc["edge_index_bonds_graph"].clone()
    bad[0, 3] = 10 ** 6
    na, nb, nfb, nf = b["x_atoms"].shape[0], b["node_features_bonds"].shape[0], b["node_features_fbonds"].shape[0], \
        b["x_frags"].shape[0]
    plan = ops.build_layer_plan(bc["edge_index"], bc["frag_index"], bc["atom_to_frag_ids"], bad, bc["edge_attr_bonds"],
                                bc["edge_index_fbonds"], bc["edge_attr_fbonds"], na, nf, nb, nfb, "cuda")
    assert int(plan.status.item()) == 1
