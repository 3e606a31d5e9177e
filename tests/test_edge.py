"""gat2_edge (bond graph + atom graph + pooling + fragment graph on connection attributes; reference
fragnet/model/gat/gat2_edge.py): the CPU restatement pinned against the unmodified reference module and the committed
golden vectors; the drop-in's surface; and -- on the GPU -- the CUDA path against both."""
import os
import sys

import pytest
import torch

from conftest import FP32_REL_TOL, ROOT, grad_errs, rel_err
from oracle import gat2_oracle as O, ref_import

sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
GOLDEN = os.path.join(ROOT, "tests", "golden", "gat2_edge_golden.pt")
needs_ref = pytest.mark.skipif(not ref_import.available(), reason="reference build not present")
GRAD_TOL = 5e-5


@pytest.fixture(scope="module")
def gold():
    return torch.load(GOLDEN)


@pytest.fixture(scope="module")
def batch():
    from make_golden_edge import edge_batch
    return edge_batch()


def _product(gold, train=False):
    from fragnet.model.gat.gat2_edge import FragNetFineTune
    torch.manual_seed(gold["weight_seed"])
    m = FragNetFineTune(**gold["kwargs"])
    return m.train() if train else m.eval()


def _product_layer(gold):
    from fragnet.model.gat.gat2_edge import FragNetLayerA
    torch.manual_seed(gold["weight_seed"] + 1)
    return FragNetLayerA(num_heads=4, return_attentions=True).eval()


def test_edge_surface_and_golden_inputs(gold, batch):
    m = _product(gold)
    sd = m.state_dict()
    assert list(sd) == gold["state_keys"]
    for k, v in gold["state_checksums"].items():
        assert abs(float(sd[k].double().abs().sum()) - v) <= 1e-9 * max(1.0, v), k
    for k, v in gold["batch_checksums"].items():
        assert abs(float(batch[k].double().abs().sum()) - v) <= 1e-9 * max(1.0, v), k
    assert list(_product_layer(gold).state_dict()) == gold["layer_state_keys"]
    assert batch["cnx_attr"].shape[1] == 8 and sd["pretrain.layers.0.cnx_attr_transform.weight"].shape == (128, 8)


def test_edge_oracle_against_golden_vectors(gold, batch):
    P = O.params_from_module(_product(gold))
    pred = O.edge_finetune_forward(P, batch, num_layer=gold["kwargs"]["num_layer"])
    assert rel_err(pred, gold["pred"]) <= 1e-6
    target = torch.linspace(-1.0, 1.0, pred.numel()).view_as(pred)
    torch.nn.functional.mse_loss(pred, target).backward()
    # grad_errs: the attention-vector and edge-embedding gradients of this model cancel to 1e-4..1e-6 of its largest
    # gradient, and their last bits follow the code path the host's BLAS picks for the fp32 products (which varies with
    # the CPU and, on some, with the process's allocation history); every other tensor gets the plain relative error
    errs = grad_errs([(k, P[k].grad, g) for k, g in gold["grads"].items()])
    assert max(errs.values()) <= 1e-6, {k: v for k, v in errs.items() if v > 1e-6}
    for k in gold["grad_none"]:
        assert P[k].grad is None, k
    with torch.no_grad():
        enc = O.edge_fragnet_forward(O.params_from_module(_product(gold), False), batch, gold["kwargs"]["num_layer"])
    for a, b in zip(enc, gold["encoder"]):
        assert rel_err(a, b) <= 1e-6
    from make_golden_edge import layer_inputs
    PL = O.params_from_module(_product_layer(gold), False)
    with torch.no_grad():
        out = O.edge_layer_forward(PL, "", 4, *layer_inputs(batch))
    for a, b in zip(out, gold["layer_out"]):
        assert rel_err(a, b) <= 1e-6


@needs_ref
def test_edge_oracle_equals_the_unmodified_reference(gold, batch):
    edge = ref_import.load_edge()
    torch.manual_seed(gold["weight_seed"])
    with ref_import.quiet():
        ref = edge.FragNetFineTune(**gold["kwargs"]).eval()
    ours = _product(gold)
    assert list(ref.state_dict()) == list(ours.state_dict())
    for (k, a), (_, b) in zip(ref.state_dict().items(), ours.state_dict().items()):
        assert a.shape == b.shape, k
        if not (k.endswith("bias") and k.split(".")[-2].isdigit()):      # the uninitialised `bias` (gat2_edge.py:35)
            assert torch.equal(a, b), k
    ours.load_state_dict(ref.state_dict(), strict=True)
    with ref_import.quiet(), torch.no_grad():
        want = ref(batch)
    got = O.edge_finetune_forward(O.params_from_module(ref, False), batch, num_layer=gold["kwargs"]["num_layer"])
    assert rel_err(got, want) == 0.0


@pytest.mark.gpu
def test_edge_model_matches_golden_on_gpu(gold, batch):
    m = _product(gold).cuda()
    bc = {k: v.cuda() for k, v in batch.items()}
    pred = m(bc)
    assert rel_err(pred, gold["pred"]) <= FP32_REL_TOL
    with torch.no_grad():
        enc = m.pretrain(bc)
    for a, b in zip(enc, gold["encoder"]):
        assert rel_err(a, b) <= FP32_REL_TOL
    target = torch.linspace(-1.0, 1.0, pred.numel()).view_as(pred).cuda()
    torch.nn.functional.mse_loss(pred, target).backward()
    named = dict(m.named_parameters())
    errs = grad_errs([(k, named[k].grad, g) for k, g in gold["grads"].items()])
    assert max(errs.values()) <= GRAD_TOL, {k: v for k, v in errs.items() if v > GRAD_TOL}
    for k in gold["grad_none"]:
        assert named[k].grad is None, k
    for k, v in gold["grad_checksums"].items():
        got = float(named[k].grad.double().abs().sum())
        assert abs(got - v) <= 2e-4 * max(v, 1e-6), k
    # CPU inputs: staged to the GPU, results back on the caller's device
    with torch.no_grad():
        cpu_enc = m.pretrain(batch)
    assert all(t.device.type == "cpu" for t in cpu_enc) and rel_err(cpu_enc[1], gold["encoder"][1]) <= FP32_REL_TOL


@pytest.mark.gpu
def test_edge_bare_layer_with_attention_on_gpu(gold, batch):
    from make_golden_edge import layer_inputs
    layer = _product_layer(gold).cuda()
    args = [t.cuda() for t in layer_inputs(batch)]
    with torch.no_grad():
        out = layer(*args)
    assert len(out) == 6
    for name, a, b in zip(("atoms", "frags", "bonds", "attn_atoms", "attn_frags", "attn_bonds"), out, gold["layer_out"]):
        assert a.shape == b.shape and rel_err(a, b) <= FP32_REL_TOL, name
    layer.return_attentions = False
    with torch.no_grad():
        assert len(layer(*args)) == 3
    # gradients flow to cnx_attr_transform and to the edge slice of f through the edge table
    xa = args[0].clone().requires_grad_()
    o = layer(xa, *args[1:])
    (o[0].sum() + o[1].square().sum()).backward()
    assert layer.cnx_attr_transform.weight.grad.abs().sum() > 0 and layer.f.grad[:, 32:160].abs().sum() > 0
    assert xa.grad is not None and torch.isfinite(xa.grad).all()


@pytest.mark.gpu
def test_edge_training_mode_is_seeded(gold, batch):
    mt = _product(gold, train=True).cuda()
    b = {k: v.cuda() for k, v in batch.items()}
    torch.manual_seed(5)
    y1 = mt(b)
    torch.manual_seed(5)
    y2 = mt(b)
    assert torch.isfinite(y1).all() and torch.equal(y1, y2) and not torch.equal(y1, mt(b))
    y1.sum().backward()
    assert all(torch.isfinite(p.grad).all() for p in mt.parameters() if p.grad is not None)
