"""Whole-path parity on the GPU: drop-in modules (CUDA kernels through the C ABI) against the CPU oracle on
identical seeded batches and weights, and against the committed golden vectors of the reference."""
import copy

import pytest
import torch

from conftest import FP32_REL_TOL, grad_errs, rel_err
from test_oracle import _rebuild

pytestmark = pytest.mark.gpu
GRAD_TOL = 5e-5      # parameter gradients: long fp32 reductions in two different orders (documented in DESIGN.md)


def _assert_grads(pairs):
    errs = grad_errs(pairs)
    bad = {k: v for k, v in errs.items() if v > GRAD_TOL}
    assert not bad, bad


def _batch(shape, n, seed, extra=True, pretrain=True):
    from fragnet_b200 import synth
    from fragnet_b200.dataset.data import collate_fn, collate_fn_pt
    mols = synth.make_dataset(shape, n, seed=seed)
    if extra:
        mols += [synth.handmade(k) for k in ("two_atom", "ion_pair", "single_frag", "two_frag")]
    return (collate_fn_pt if pretrain else collate_fn)(mols)


def _to(batch, dev):
    return {k: v.to(dev) for k, v in batch.items()}


def test_native_library_is_loaded():
    from fragnet_b200 import _abi
    lib = _abi.load()
    assert lib.fnb_version() == _abi.ABI_VERSION
    maps = open("/proc/self/maps").read()
    assert "libfragnet_b200.so" in maps


def test_layer_forward_backward_matches_oracle():
    """One FragNetLayerA call (layer >= 1 geometry, all-128 inputs) with gradients for inputs and parameters."""
    from fragnet.model.gat.gat2 import FragNetLayerA
    from oracle import gat2_oracle as O
    b = _batch("esol", 12, 5)
    torch.manual_seed(3)
    layer = FragNetLayerA(atom_in=128, atom_out=128, frag_in=128, frag_out=128, edge_in=128, edge_out=128,
                          fedge_in=128, num_heads=4, fbond_edge_in=6, return_attentions=True).cuda()
    gen = torch.Generator().manual_seed(9)
    na, ne, nfb, nf = b["x_atoms"].shape[0], b["edge_index"].shape[1], b["frag_index"].shape[1], b["x_frags"].shape[0]
    xa = torch.randn(na, 128, generator=gen)
    xb = torch.randn(ne, 128, generator=gen)
    xfb = torch.randn(nfb, 128, generator=gen)
    cu = lambda t: t.clone().cuda().requires_grad_()
    xa_c, xb_c, xfb_c = cu(xa), cu(xb), cu(xfb)
    bc = _to(b, "cuda")
    outs = layer(xa_c, bc["edge_index"], xb_c, bc["frag_index"], torch.zeros(nf, 128, device="cuda"),
                 bc["atom_to_frag_ids"], xb_c, bc["edge_index_bonds_graph"], bc["edge_attr_bonds"],
                 xfb_c, bc["edge_index_fbonds"], bc["edge_attr_fbonds"])
    P = O.params_from_module(layer)
    xa_o, xb_o, xfb_o = (t.clone().requires_grad_() for t in (xa, xb, xfb))
    ref = O.layer_forward(P, "", 4, xa_o, b["edge_index"], xb_o, b["frag_index"], torch.zeros(nf, 128),
                          b["atom_to_frag_ids"], xb_o, b["edge_index_bonds_graph"], b["edge_attr_bonds"],
                          xfb_o, b["edge_index_fbonds"], b["edge_attr_fbonds"])
    assert len(outs) == 8
    names = ("x_atoms", "x_frags", "bond", "fbond", "attn_atoms", "attn_frags", "attn_bonds", "attn_fbonds")
    # Unit-variance 128-d inputs drive the logits to |z| ~ 10, where the reference's OWN fp32 rounding (order of the
    # 96/192-term dot products) moves the softmax by ~1e-5; measure that noise against a float64 run of the same
    # oracle and allow for it (realistic activations, tested below on whole models, stay at ~1e-7).
    P64 = {k: v.detach().double() for k, v in P.items()}
    ref64 = O.layer_forward(P64, "", 4, xa.double(), b["edge_index"], xb.double(), b["frag_index"],
                            torch.zeros(nf, 128, dtype=torch.float64), b["atom_to_frag_ids"], xb.double(),
                            b["edge_index_bonds_graph"], b["edge_attr_bonds"].double(), xfb.double(),
                            b["edge_index_fbonds"], b["edge_attr_fbonds"].double())
    for n, a, r, r64 in zip(names, outs, ref, ref64):
        noise = rel_err(r, r64)
        assert rel_err(a, r64) <= max(FP32_REL_TOL, 3 * noise), (n, rel_err(a, r64), noise)
    ws = [torch.randn(t.shape, generator=gen) for t in ref[:4]]
    sum((o * w.cuda()).sum() for o, w in zip(outs[:4], ws)).backward()
    sum((o * w).sum() for o, w in zip(ref[:4], ws)).backward()
    for n, a, r in (("dx_atoms", xa_c, xa_o), ("dx_bond", xb_c, xb_o), ("dx_fbond", xfb_c, xfb_o)):
        assert rel_err(a.grad, r.grad) <= GRAD_TOL, n
    for k, p in layer.named_parameters():
        assert (p.grad is None) == (P[k].grad is None), k
    _assert_grads([(k, p.grad, P[k].grad) for k, p in layer.named_parameters() if p.grad is not None])


@pytest.mark.parametrize("shape,n", [("esol", 16), ("unimol", 64), ("stress", 3)])
def test_finetune_forward_backward_matches_oracle(shape, n):
    from fragnet.model.gat.gat2 import FragNetFineTune
    from oracle import gat2_oracle as O
    b = _batch(shape, n, 21, pretrain=False)
    torch.manual_seed(11)
    m = FragNetFineTune(n_classes=1, num_layer=4, drop_ratio=0.1, h1=128, h2=1024, h3=1024, h4=512, act="relu",
                        fthead="FTHead3").eval()
    P = O.params_from_module(m)
    m = m.cuda()
    pred = m(_to(b, "cuda"))
    ref = O.finetune_forward(P, b)
    assert pred.shape == ref.shape
    assert rel_err(pred, ref) <= FP32_REL_TOL
    pred.sum().backward()
    ref.sum().backward()
    for k, p in m.named_parameters():
        assert (p.grad is None) == (P[k].grad is None), k
    _assert_grads([(k, p.grad, P[k].grad) for k, p in m.named_parameters() if p.grad is not None])


def test_pretrain_step_matches_oracle_and_golden(golden, golden_batch):
    from fragnet_b200.train.pretrain_utils import pretrain_loss
    from oracle import gat2_oracle as O
    m = _rebuild(golden, "pt")
    P = O.params_from_module(m)
    m = m.cuda()
    bc = _to(golden_batch, "cuda")
    preds = m(bc)
    for a, r in zip(preds, golden["pt_preds"]):
        assert rel_err(a, r) <= FP32_REL_TOL
    loss = pretrain_loss(torch.nn.MSELoss(), preds, bc)
    assert rel_err(loss, golden["pt_loss"]) <= FP32_REL_TOL
    loss.backward()
    named = dict(m.named_parameters())
    _assert_grads([(k, named[k].grad, g) for k, g in golden["pt_grads"].items()])
    lo = O.pretrain_loss(O.pretrain_forward(P, golden_batch), golden_batch)
    lo.backward()
    _assert_grads([(k, p.grad, P[k].grad) for k, p in m.named_parameters() if P[k].grad is not None])


def test_finetune_against_golden_vectors(golden, golden_batch):
    m = _rebuild(golden, "ft").cuda()
    bc = _to(golden_batch, "cuda")
    pred = m(bc)
    assert rel_err(pred, golden["ft_pred"]) <= FP32_REL_TOL
    pred.sum().backward()
    named = dict(m.named_parameters())
    _assert_grads([(k, named[k].grad, g) for k, g in golden["ft_grads"].items()])
    for k in golden["ft_grad_none"]:
        assert named[k].grad is None, k
    with torch.no_grad():
        enc = m.pretrain.forward_with_attention(bc)
        for name, t in zip(golden["encoder"], enc):
            assert rel_err(t, golden["encoder"][name]) <= FP32_REL_TOL, name
        for attr, val in (("bond_mask", 2), ("atom_mask_individual", 3), ("frag_bond_mask", 0)):
            mm = copy.deepcopy(m)
            for layer in mm.pretrain.layers:
                setattr(layer, attr, val)
            assert rel_err(mm(bc), golden["ft_masked_pred"][attr]) <= FP32_REL_TOL, attr


def test_viz_arrangement_layer_calls_and_cpu_inputs(golden, golden_batch):
    """The reference's vizualize/model.py drives FragNetLayerA directly, on CPU tensors, with the last layer
    returning attentions; outputs must come back on the caller's device."""
    m = _rebuild(golden, "ft")           # parameters stay on the CPU, like the Streamlit app's model
    enc = m.pretrain
    b = golden_batch
    with torch.no_grad():
        x_atoms, x_frags = b["x_atoms"], b["x_frags"]
        bond_nodes, fbond_nodes, edge_attr = b["node_features_bonds"], b["node_features_fbonds"], b["edge_attr"]
        for li, layer in enumerate(enc.layers):
            layer.return_attentions = li == len(enc.layers) - 1
            out = layer(x_atoms, b["edge_index"], edge_attr, b["frag_index"], x_frags, b["atom_to_frag_ids"],
                        bond_nodes, b["edge_index_bonds_graph"], b["edge_attr_bonds"],
                        fbond_nodes, b["edge_index_fbonds"], b["edge_attr_fbonds"])
            assert len(out) == (8 if layer.return_attentions else 4)
            assert all(t.device.type == "cpu" for t in out)
            x_atoms, x_frags, bond_nodes, fbond_nodes = (torch.relu(t) for t in out[:4])
            edge_attr = bond_nodes
        got = (x_atoms, x_frags, bond_nodes, fbond_nodes) + tuple(out[4:])
    for name, t in zip(golden["encoder"], got):
        assert rel_err(t, golden["encoder"][name]) <= FP32_REL_TOL, name
    attn_atoms = got[4]
    assert abs(float(attn_atoms.sum()) - 4 * b["x_atoms"].shape[0]) < 1e-2
    pred = m(b)                           # whole model on CPU tensors -> CPU result
    assert pred.device.type == "cpu" and rel_err(pred, golden["ft_pred"]) <= FP32_REL_TOL


def test_training_mode_dropout_runs_and_is_seeded():
    from fragnet.model.gat.gat2_pretrain import FragNetPreTrain
    from fragnet_b200.train.pretrain_utils import pretrain_loss
    b = _to(_batch("unimol", 32, 2), "cuda")
    torch.manual_seed(0)
    m = FragNetPreTrain(num_layer=4, drop_ratio=0.2, edge_features=17).cuda().train()
    opt = torch.optim.Adam(m.parameters(), lr=1e-4)
    losses = []
    for _ in range(3):
        opt.zero_grad()
        loss = pretrain_loss(torch.nn.MSELoss(), m(b), b)
        loss.backward()
        opt.step()
        losses.append(loss.item())
    assert all(torch.isfinite(torch.tensor(losses)))
    live = [k for k, p in m.named_parameters() if p.grad is not None]
    assert "pretrain.layers.3.f" in live and "pretrain.layers.0.f" not in live


def test_gradients_are_run_to_run_deterministic():
    from fragnet.model.gat.gat2 import FragNetFineTune
    b = _to(_batch("esol", 24, 8, pretrain=False), "cuda")
    torch.manual_seed(2)
    m = FragNetFineTune(num_layer=2, drop_ratio=0.0, h1=32, h2=32, h3=32, h4=32, act="relu").cuda().eval()
    grads = []
    for _ in range(2):
        m.zero_grad()
        m(b).sum().backward()
        grads.append({k: p.grad.clone() for k, p in m.named_parameters() if p.grad is not None})
    for k in grads[0]:
        if "pretrain" in k:                # our kernels: bitwise; the torch head may use split-K atomics
            assert torch.equal(grads[0][k], grads[1][k]), k


def test_flat_adam_equals_torch_adam():
    """FlatAdam (one launch over a flat buffer) follows torch.optim.Adam step for step; state_dict keys survive."""
    from fragnet.model.gat.gat2 import FragNetFineTune
    from fragnet_b200.train.optim import FlatAdam
    b = _to(_batch("esol", 10, 3, pretrain=False), "cuda")
    torch.manual_seed(11)
    m1 = FragNetFineTune(num_layer=2, drop_ratio=0.0, h1=32, h2=32, h3=32, h4=32, act="relu").cuda()
    m2 = copy.deepcopy(m1)
    keys = list(m1.state_dict().keys())
    o1 = o2 = None
    for step in range(3):
        for m in (m1, m2):
            for p in m.parameters():
                p.grad = None
            m(b).pow(2).mean().backward()
        if o1 is None:
            o1 = torch.optim.Adam([p for p in m1.parameters() if p.grad is not None], lr=1e-3)
            o2 = FlatAdam([p for p in m2.parameters() if p.grad is not None], lr=1e-3)
        o1.step()
        o2.step()
    assert list(m2.state_dict().keys()) == keys
    for (k, a), (_, c) in zip(m1.state_dict().items(), m2.state_dict().items()):
        assert rel_err(c, a) <= 2e-5, k


def test_device_prefetcher_yields_identical_batches():
    from fragnet_b200.dataset.prefetch import DevicePrefetcher
    host = [_batch("esol", 6 + s, s) for s in range(7)]
    n = 0
    for h, d in zip(host, DevicePrefetcher(iter(host), "cuda", depth=2)):   # a batch is valid until 2 more are requested
        assert set(h) == set(d)
        for k in h:
            assert d[k].is_cuda and d[k].dtype == h[k].dtype and d[k].shape == h[k].shape
            assert torch.equal(d[k].cpu(), h[k]), k
        n += 1
    assert n == len(host)
    # hot_path_only: the tensors the GAT2 path never reads stay on the host; the model output is unchanged
    from fragnet.model.gat.gat2 import FragNetFineTune
    torch.manual_seed(0)
    m = FragNetFineTune(num_layer=2, drop_ratio=0.0, h1=32, h2=32, h3=32, h4=32).cuda().eval()
    lean = next(iter(DevicePrefetcher(iter(host[:1]), "cuda", hot_path_only=True)))
    assert "edge_attr" not in lean and "cnx_attr" not in lean and lean["x_frags"].device.type == "meta"
    assert lean["x_frags"].shape == host[0]["x_frags"].shape
    with torch.no_grad():
        assert torch.equal(m(lean), m({k: v.cuda() for k, v in host[0].items()}))


def test_unsorted_fragment_connections_match_oracle():
    """A batch whose fragment-connection list is not sorted by molecule (the nodes of the fragment-connection graph
    are then not grouped by molecule) gives the oracle's forward and gradients."""
    from fragnet.model.gat.gat2 import FragNetFineTune
    from oracle import gat2_oracle as O
    b = _batch("esol", 64, 4, pretrain=False)
    torch.manual_seed(6)
    m = FragNetFineTune(n_classes=1, num_layer=4, drop_ratio=0.0, h1=32, h2=32, h3=32, h4=32, act="relu").eval()
    P = O.params_from_module(m)
    # shuffle the fragment-connection list: nodes of the fragment-connection graph are no longer grouped by molecule
    # (everything that indexes them is permuted consistently, so the model output is unchanged)
    nfb = b["frag_index"].shape[1]
    assert nfb > 128
    perm = torch.randperm(nfb, generator=torch.Generator().manual_seed(0))
    inv = torch.empty_like(perm)
    inv[perm] = torch.arange(nfb)
    b2 = dict(b)
    b2["frag_index"] = b["frag_index"][:, perm]
    b2["cnx_attr"] = b["cnx_attr"][perm]
    b2["node_features_fbonds"] = b["node_features_fbonds"][perm]
    b2["edge_index_fbonds"] = inv[b["edge_index_fbonds"]]
    ref = O.finetune_forward(P, b2)
    ref.sum().backward()
    m = m.cuda()
    pred = m(_to(b2, "cuda"))
    assert rel_err(pred, ref) <= FP32_REL_TOL
    pred.sum().backward()
    _assert_grads([(k, p.grad, P[k].grad) for k, p in m.named_parameters() if p.grad is not None])


def test_input_dropout_fused_into_padding_draws_the_same_mask():
    """nn.Dropout on x_atoms (gat2.py:396) is applied by the layer-0 padding kernel unless d x_atoms is wanted, in which
    case the standalone kernel runs: same counters, same bits -- bitwise the same forward either way."""
    from fragnet.model.gat.gat2 import FragNetFineTune
    from fragnet_b200 import ops
    b = _to(_batch("esol", 20, 12, pretrain=False), "cuda")
    torch.manual_seed(3)
    m = FragNetFineTune(n_classes=1, num_layer=2, drop_ratio=0.3, h1=32, h2=32, h3=32, h4=32, act="relu").cuda().train()
    outs = []
    for want_dx in (False, True):
        torch.manual_seed(99)
        ops.clear_plan_cache()
        x = dict(b)
        x["x_atoms"] = b["x_atoms"].clone().requires_grad_(want_dx)
        outs.append(m.pretrain(x))
    for a, c in zip(outs[0], outs[1]):
        if isinstance(a, torch.Tensor):
            assert torch.equal(a, c)
