"""The one-call finetuning step for the gat2_lite and gat2_edge model versions (``FusedLiteFineTuneStep`` /
``FusedEdgeFineTuneStep``, ``fnb_finetune_step`` with ``variant``) against the float64 oracle with the library's dropout
masks replayed on the host, and ``TrainerFineTune(fused=True)`` on both versions against the generic loop.

Counter layout of the step (``fnb_finetune_step_args`` in the header): the sites of one gat2 encoder call over
(Na, Nb, Nfb, Nf) rows -- Nfb = 0 for gat2_lite, whose last-layer fragment site covers ReLU(Dropout(pool(atoms))), and
the fragment-edge count for gat2_edge, whose fragment-connection sites stay reserved -- then the head's sites."""
import copy
import ctypes as C
import re

import pytest
import torch
import torch.nn.functional as F

from conftest import FP32_REL_TOL, rel_err
from test_gpu_dropout import (_check_grads, _f64, _gen, _last_only, _param_pairs, _params64, _sizes, _start_stream,
                              encoder_sites, keep_mask, replay, roundup4)
from test_gpu_finetune_step import W_ODD, _case_batch, _head_sites, _head_spec

pytestmark = pytest.mark.gpu


def _widen_cnx(hb, seed):
    """gat2_edge's connection attributes are 8 wide: two random columns the 6-wide featuriser lacks."""
    extra = torch.rand(hb["cnx_attr"].shape[0], 2, generator=torch.Generator().manual_seed(seed))
    hb["cnx_attr"] = torch.cat((hb["cnx_attr"], extra), dim=1)
    return hb


def _batch(variant, n_classes, loss_kind, seed):
    hb = _case_batch(n_classes, loss_kind, seed)
    return _widen_cnx(hb, seed) if variant == "edge" else hb


def _model(variant, fthead, act, n_classes, drop, widths, num_layer, seed):
    from fragnet_b200.model.gat import gat2_edge, gat2_lite
    mod = gat2_lite if variant == "lite" else gat2_edge
    torch.manual_seed(seed)
    h1, h2, h3, h4 = widths
    return mod.FragNetFineTune(n_classes=n_classes, num_layer=num_layer, drop_ratio=drop, h1=h1, h2=h2, h3=h3, h4=h4,
                               act=act, fthead=fthead, edge_features=17).cuda().train()


def _step(variant, m, **kw):
    from fragnet_b200.train.fused import FusedEdgeFineTuneStep, FusedLiteFineTuneStep
    return (FusedLiteFineTuneStep if variant == "lite" else FusedEdgeFineTuneStep)(m, **kw)


def _enc_sites(variant, hb, off0, num_layer):
    na, k_atom, nb, nfb, nf = _sizes(hb)
    return encoder_sites(off0, num_layer, na, k_atom, nb, 0 if variant == "lite" else nfb, nf)


def _oracle(variant, m, hb, fthead, act, n_classes, loss_kind, drop, training, seed_v, off0, num_layer):
    """float64 loss, predictions and parameter gradients with the masks of the step that started at ``off0``."""
    from oracle import gat2_oracle as O
    P = _params64(m)
    b = _f64(hb)
    g = b["y"].numel() // n_classes
    spec = _head_spec(m, fthead)
    fwd = O.lite_fragnet_forward if variant == "lite" else O.edge_fragnet_forward
    draws = training and (drop > 0 or any(pi > 0 or po > 0 for _, pi, po, _ in spec))
    sites = {}
    if draws:
        bases, enc_span = _enc_sites(variant, hb, off0, num_layer)
        widths = [tuple(P[name + ".weight"].shape[::-1]) for name, _, _, _ in spec]
        sites, _ = _head_sites(spec, widths, g, off0 + enc_span)
        x_atoms, x_frags = fwd(P, b, num_layer, drop_ratio=drop, training=True,
                               drop_fn=replay(_last_only(bases, num_layer), seed_v, drop))[:2]
    else:
        x_atoms, x_frags = fwd(P, b, num_layer, drop_ratio=0.0, training=False)[:2]
    x = O.readout(x_atoms, x_frags, b)
    fn = F.relu if fthead in ("FTHead1", "FTHead2") else O._ACTS[act]

    def mask(site, t, p):
        if site not in sites:
            return t
        keep = torch.from_numpy(keep_mask(seed_v, sites[site], t.numel(), p)).view(t.shape)
        return t * (keep.to(t.dtype) / (1.0 - p))
    for l, (name, p_in, p_out, hidden) in enumerate(spec):
        z = O._linear(P, name, mask((l, "in"), x, p_in))
        z = mask((l, "out"), z, p_out)
        x = fn(z) if hidden else z
    pred, y = x, b["y"]
    if loss_kind == "mse":
        loss = ((pred.reshape(-1) - y) ** 2).mean()
    else:
        lab = y.view(pred.shape)
        valid = lab > -0.5
        lm = F.binary_cross_entropy_with_logits(pred, lab.clamp_min(0), reduction="none")
        loss = torch.where(valid, lm, torch.zeros_like(lm)).sum() / valid.sum()
    loss.backward()
    return loss, pred.detach(), P


def _span(variant, m, hb, fthead, n_classes, num_layer):
    g = hb["y"].numel() // n_classes
    spec = _head_spec(m, fthead)
    widths = [tuple(dict(m.named_parameters())[n + ".weight"].shape[::-1]) for n, _, _, _ in spec]
    return _enc_sites(variant, hb, 0, num_layer)[1] + _head_sites(spec, widths, g, 0)[1]


def _lib_span(fused, b):
    from fragnet_b200 import ops
    a, _, _, _ = fused._args(b, True, False)
    return ops._lib().fnb_finetune_step_rng_span(C.byref(a))


CASES = [
    # fthead, act, n_classes, loss, drop, widths, num_layer
    ("FTHead3", "celu", 1, "mse", 0.2, W_ODD, 3),
    ("FTHead3", "celu", 3, "bce", 0.2, W_ODD, 1),
    ("FTHead4", "relu", 1, "mse", 0.2, W_ODD, 1),
    ("FTHead4", "relu", 3, "bce", 0.2, W_ODD, 3),
    ("FTHead1", "relu", 1, "mse", 0.2, W_ODD, 3),
    ("FTHead3", "celu", 1, "mse", 0.0, W_ODD, 3),        # training at p = 0: no site draws
]
IDS = ["-".join(map(str, c[:5])) + f"-L{c[6]}" for c in CASES]


@pytest.mark.parametrize("variant", ["lite", "edge"])
@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_fused_variant_step_matches_oracle_with_replayed_masks(variant, case):
    fthead, act, n_classes, loss_kind, drop, widths, num_layer = case
    seed = 500 + CASES.index(case) + (50 if variant == "edge" else 0)
    hb = _batch(variant, n_classes, loss_kind, seed)
    m = _model(variant, fthead, act, n_classes, drop, widths, num_layer, seed + 1)
    fused = _step(variant, m, lr=1e-3, loss=loss_kind)
    b = {k: v.cuda() for k, v in hb.items()}
    seed_v, off0 = _start_stream(seed + 2)
    loss = fused.forward_backward(b)
    off1 = _gen().get_offset()
    ref_loss, _, P = _oracle(variant, m, hb, fthead, act, n_classes, loss_kind, drop, True, seed_v, off0, num_layer)
    assert rel_err(loss, ref_loss) <= FP32_REL_TOL
    errs = _check_grads(_param_pairs(m.named_parameters(), P))
    top = f"pretrain.layers.{num_layer - 1}."
    if variant == "edge":        # the device-formed edge term reached cnx_attr_transform and both slices of f
        assert {top + "cnx_attr_transform.weight", top + "cnx_attr_transform.bias", top + "f"} <= set(errs)
        assert float(m.pretrain.layers[-1].f.grad[:, 32:160].abs().max()) > 0
    else:
        assert not any(k.endswith((".f", "projection_fb.weight", "f_a_b")) for k in errs)
    # counters: the documented layout, and the host reserved exactly that many
    span = _span(variant, m, hb, fthead, n_classes, num_layer)
    assert _lib_span(fused, b) == span
    draws = drop > 0
    assert off1 - off0 == (roundup4(span) if draws else 0)
    # evaluation: the oracle's eval forward, no counter drawn
    m.eval()
    loss_e, preds = fused.evaluate(b, return_predictions=True)
    torch.cuda.synchronize()
    assert _gen().get_offset() == off1
    ref_e, ref_pred, _ = _oracle(variant, m, hb, fthead, act, n_classes, loss_kind, drop, False, seed_v, off0, num_layer)
    assert preds.shape == (hb["y"].numel() // n_classes, n_classes)
    assert rel_err(preds, ref_pred) <= FP32_REL_TOL
    assert rel_err(loss_e, ref_e) <= FP32_REL_TOL


FREEZE = ["layer0", "encoder", "head0"]


@pytest.mark.parametrize("variant", ["lite", "edge"])
@pytest.mark.parametrize("how", FREEZE)
def test_frozen_parameters_of_the_variants(variant, how):
    fthead, act, num_layer, drop = "FTHead3", "celu", 2, 0.2
    seed = 600 + FREEZE.index(how) + (10 if variant == "edge" else 0)
    hb = _batch(variant, 1, "mse", seed)
    m = _model(variant, fthead, act, 1, drop, W_ODD, num_layer, seed + 1)
    if how == "layer0":
        frozen = list(m.pretrain.layers[0].parameters())
    elif how == "encoder":
        frozen = list(m.pretrain.parameters())
    else:
        frozen = list(m.fthead.predictor[0].parameters())
    for p in frozen:
        p.requires_grad_(False)
    before = {id(p): p.detach().clone() for p in frozen}
    fused = _step(variant, m, lr=1e-3)
    assert fused.first_trained_layer == {"layer0": 1, "encoder": num_layer, "head0": 0}[how]
    b = {k: v.cuda() for k, v in hb.items()}
    seed_v, off0 = _start_stream(seed + 2)
    fused.forward_backward(b)
    _, _, P = _oracle(variant, m, hb, fthead, act, 1, "mse", drop, True, seed_v, off0, num_layer)
    named = dict(m.named_parameters())
    pairs = [(k, p.grad, P[k].grad) for k, p in named.items() if p.requires_grad and p.grad is not None]
    assert pairs
    _check_grads(pairs)
    live = {id(p) for p in fused.live}
    for k, p in named.items():      # trained tensors are exactly the live ones that require a gradient
        if id(p) not in live:
            assert p.grad is None, k
    cnx = m.pretrain.layers[-1].cnx_attr_transform if variant == "edge" else None
    cnx_before = None if cnx is None else cnx.weight.detach().clone()
    fused.step(b)
    torch.cuda.synchronize()
    for p in frozen:
        assert torch.equal(p.detach(), before[id(p)]) and p.grad is None
    if cnx is not None:
        assert torch.equal(cnx.weight.detach(), cnx_before) == (how == "encoder")


@pytest.mark.parametrize("variant", ["lite", "edge"])
def test_two_identical_runs_and_single_stream_mode_give_the_same_bits(variant):
    import os
    import subprocess
    import sys
    code = (
        "import sys, torch\n"
        "sys.path.insert(0, 'tests')\n"
        "from test_gpu_finetune_variants import _model, _batch, _step, W_ODD\n"
        f"hb = _batch('{variant}', 1, 'mse', 70)\n"
        "b = {k: v.cuda() for k, v in hb.items()}\n"
        "out = []\n"
        "for _ in range(2):\n"
        f"    m = _model('{variant}', 'FTHead3', 'relu', 1, 0.2, W_ODD, 3, 71)\n"
        "    torch.manual_seed(3)\n"
        f"    f = _step('{variant}', m, lr=1e-3)\n"
        "    f.forward_backward(b)\n"
        "    out.append(f.flat_g.cpu().numpy().tobytes())\n"
        "assert out[0] == out[1]\n"
        "import hashlib\n"
        "print('RESULT', hashlib.sha256(out[0]).hexdigest())\n")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    digests = []
    for streams in (None, "1"):
        env = dict(os.environ, PYTHONPATH=root)
        env.pop("FNB_STREAMS", None)
        if streams:
            env["FNB_STREAMS"] = streams
        r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd=root, timeout=300)
        assert r.returncode == 0, r.stderr[-2000:]
        digests.append([l for l in r.stdout.splitlines() if l.startswith("RESULT")][0].split()[1])
    assert digests[0] == digests[1]


def _loader(variant, seed):
    from torch.utils.data import DataLoader
    from fragnet_b200 import synth
    from fragnet_b200.dataset.data import collate_fn_pt
    mols = synth.make_dataset("esol", 48, seed=seed)
    gen = torch.Generator().manual_seed(seed + 1)
    for mol in mols:
        mol.y = torch.randn(mol.y.shape, generator=gen)
        if variant == "edge":
            mol.cnx_attr = torch.cat((mol.cnx_attr, torch.rand(mol.cnx_attr.shape[0], 2, generator=gen)), dim=1)
    return DataLoader(mols, collate_fn=collate_fn_pt, batch_size=16, shuffle=False, drop_last=True)


@pytest.mark.parametrize("variant", ["lite", "edge"])
def test_trainer_fused_path_equals_generic_loop(variant):
    from fragnet_b200.train.utils import TrainerFineTune
    loader = _loader(variant, 12)
    m1 = _model(variant, "FTHead3", "celu", 1, 0.0, W_ODD, 2, 14)
    m2 = copy.deepcopy(m1)
    o1, o2 = torch.optim.Adam(m1.parameters(), lr=1e-3), torch.optim.Adam(m2.parameters(), lr=1e-3)
    t1, t2 = TrainerFineTune(fused=True), TrainerFineTune()
    l1 = t1.train(m1, loader, o1, None, "cuda", loader)
    l2 = t2.train(m2, loader, o2, None, "cuda", loader)       # the generic loop (gat2_edge: reads cnx_attr)
    assert abs(l1 - l2) <= 1e-5 * abs(l2)
    fs = t1._fused_for(m1, o1, "cuda", "mse")
    assert fs is not None and fs.plan_hits > 0 and not t2._fused_steps
    p2 = dict(m2.named_parameters())
    assert max(rel_err(p, p2[k]) for k, p in m1.named_parameters()) <= 5e-4
    for k, p in m1.named_parameters():      # dead tensors keep no gradient on either path
        assert (p.grad is None) == (p2[k].grad is None), k
    v1, v2 = t1.validate(m1, loader, "cuda"), t2.validate(m2, loader, "cuda")
    assert abs(v1 - v2) <= 1e-3 * abs(v2)


@pytest.mark.parametrize("variant", ["lite", "edge"])
def test_no_fragment_connection_attention_runs(variant):
    """The variants have no fragment-connection graph: no attention kernel for its edge mode (FNB_EDGE_AFFINE6 = 2)
    is launched by a fused training step."""
    from torch.profiler import ProfilerActivity, profile
    hb = _batch(variant, 1, "mse", 40)
    m = _model(variant, "FTHead3", "relu", 1, 0.2, W_ODD, 2, 41)
    fused = _step(variant, m, lr=1e-3)
    b = {k: v.cuda() for k, v in hb.items()}
    fused.step(b)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(2):      # (the kernels of the second step are in the trace whenever tracing starts)
            fused.step(b)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type.name == "CUDA"]
    assert any("k_gat_fwd_tiled" in n for n in names)
    assert not [n for n in names if re.search(r"k_gat_(fwd|bwd_dst)_tiled<2\b", n)]
    if variant == "edge":
        assert any("k_cnx_table<" in n or "k_cnx_table(" in n for n in names)
        assert any("k_cnx_table_bwd" in n for n in names)


def test_argument_errors_and_input_checks():
    from fragnet_b200 import _abi, ops
    hb = _batch("edge", 1, "mse", 20)
    m = _model("edge", "FTHead3", "relu", 1, 0.0, W_ODD, 2, 21)
    fused = _step("edge", m, lr=1e-3)
    b = {k: v.cuda() for k, v in hb.items()}
    lib = ops._lib()
    a, _, _, keep = fused._args(b, True, False)
    need = lib.fnb_finetune_step_workspace_bytes(C.byref(a))
    assert need > 0
    ws = torch.empty(need + 256, dtype=torch.uint8, device="cuda")
    scratch = ops._ptr(ops.scratch(ws.device))
    run = lambda args: lib.fnb_finetune_step(C.byref(args), ops._ptr(ws), need, scratch, ops._stream())
    bad = _abi.CFinetuneStepArgs.from_buffer_copy(a)
    bad.variant = 3
    assert run(bad) == -3
    assert lib.fnb_finetune_step_workspace_bytes(C.byref(bad)) == 0
    for field in ("cnx_attr", "W_cnx", "b_cnx"):
        bad = _abi.CFinetuneStepArgs.from_buffer_copy(a)
        setattr(bad, field, None)
        assert run(bad) == -1, field
    assert run(a) == 0
    torch.cuda.synchronize()
    # the 6-wide featuriser output cannot feed Linear(8, 128)
    b6 = dict(b, cnx_attr=b["cnx_attr"][:, :6].contiguous())
    with pytest.raises(ValueError):
        fused.forward_backward(b6)
    # the gat2 class stays gat2-only; each variant class takes its own model version only
    from fragnet_b200.train.fused import FusedFineTuneStep, finetune_step_class
    with pytest.raises(NotImplementedError):
        FusedFineTuneStep(m)
    with pytest.raises(NotImplementedError):
        _step("lite", m)
    assert finetune_step_class(m) is type(fused)
