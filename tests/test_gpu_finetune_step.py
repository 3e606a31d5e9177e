"""The one-call finetuning step (``fnb_finetune_step`` / ``FusedFineTuneStep``) against the float64 oracle, with the
library's dropout masks replayed on the host for every encoder and head dropout site, and ``TrainerFineTune(fused=True)``
against the generic loop.

Head dropout sites follow the encoder's counters: per head layer an input site (FTHead1 / FTHead4) and an output site
(FTHead2 / FTHead3) where the layer's p is non-zero, each ``ceil(G * width / 4)`` counters over the row-major
``[G, width]`` tensor.  The oracle's ``fthead_forward`` has no mask hook, so the head is restated here over the same
parameter mapping, site by site; at p = 0 the oracle's own ``finetune_forward`` is the reference."""
import copy
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from conftest import FP32_REL_TOL, rel_err
from test_gpu_dropout import (_check_grads, _f64, _gen, _host_batch, _last_only, _param_pairs, _params64, _seed,
                              _sizes, _start_stream, counters_of, encoder_sites, keep_mask, replay, roundup4)

pytestmark = pytest.mark.gpu

HEAD_NAMES = {"FTHead1": ("lin1", "out"), "FTHead4": ("dense", "out_proj")}


def _head_spec(m, fthead):
    """(parameter prefix, p_in, p_out, activation) per head layer, as gat2.py:569-751 arrange them."""
    head = m.fthead
    p = float(head.dropout.p)
    if fthead in HEAD_NAMES:
        a, b = HEAD_NAMES[fthead]
        return [(f"fthead.{a}", p, 0.0, True), (f"fthead.{b}", p, 0.0, False)]
    n = len(head.predictor)
    return [(f"fthead.predictor.{i}", 0.0, p if i + 1 < n else 0.0, i + 1 < n) for i in range(n)]


def _head_sites(spec, widths, g, start):
    """{(layer, "in" | "out"): counter base} of the head's dropout sites from counter ``start``; total counters."""
    c, sites = start, {}
    for l, (_, p_in, p_out, _) in enumerate(spec):
        if p_in > 0:
            sites[(l, "in")] = c
            c += counters_of(g * widths[l][0])
        if p_out > 0:
            sites[(l, "out")] = c
            c += counters_of(g * widths[l][1])
    return sites, c - start


def _oracle_step(m, hb, fthead, act, n_classes, loss_kind, drop, training, seed_v, off0, num_layer):
    """float64 loss, predictions and parameter gradients with the masks of the call that started at counter ``off0``."""
    from oracle import gat2_oracle as O
    P = _params64(m)
    b = _f64(hb)
    g = b["y"].numel() // n_classes
    spec = _head_spec(m, fthead)
    if not training or (drop == 0 and all(pi == 0 and po == 0 for _, pi, po, _ in spec)):
        pred = O.finetune_forward(P, b, num_layer, drop_ratio=0.0, training=False, fthead=fthead, act=act)
    else:
        bases, enc_span = encoder_sites(off0, num_layer, *_sizes(hb))
        widths = [tuple(P[name + ".weight"].shape[::-1]) for name, _, _, _ in spec]
        sites, _ = _head_sites(spec, widths, g, off0 + enc_span)
        x_atoms, x_frags, _, _ = O.fragnet_forward(P, b, num_layer, drop_ratio=drop, training=True,
                                                   drop_fn=replay(_last_only(bases, num_layer), seed_v, drop))
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
        pred = x
    y = b["y"]
    if loss_kind == "mse":
        loss = ((pred.reshape(-1) - y) ** 2).mean()
    else:
        lab = y.view(pred.shape)
        valid = lab > -0.5
        lm = F.binary_cross_entropy_with_logits(pred, lab.clamp_min(0), reduction="none")
        loss = torch.where(valid, lm, torch.zeros_like(lm)).sum() / valid.sum()
    loss.backward()
    return loss, pred.detach(), P


def _case_batch(n_classes, loss_kind, seed):
    hb = _host_batch(8, 10, seed)
    g = hb["y"].numel()
    gen = torch.Generator().manual_seed(seed + 5)
    if loss_kind == "mse":
        hb["y"] = torch.randn(g * n_classes, generator=gen)
    else:
        y = torch.randint(0, 2, (g * n_classes,), generator=gen).float()
        y[torch.rand(g * n_classes, generator=gen) < 0.25] = -1.0          # missing labels
        y[0] = 1.0
        hb["y"] = y
    return hb


def _model(fthead, act, n_classes, drop, widths, num_layer, seed):
    from fragnet.model.gat.gat2 import FragNetFineTune
    torch.manual_seed(seed)
    h1, h2, h3, h4 = widths
    return FragNetFineTune(n_classes=n_classes, num_layer=num_layer, drop_ratio=drop, h1=h1, h2=h2, h3=h3, h4=h4,
                           act=act, fthead=fthead).cuda().train()


def _lib_span(fused, b):
    from fragnet_b200 import ops
    a, _, _, _ = fused._args(b, True, False)
    return ops._lib().fnb_finetune_step_rng_span(C.byref(a))


W_ODD = (100, 64, 37, 48)          # widths that are not multiples of 32 (FTHead3 / FTHead4)
CASES = [
    # fthead, act, n_classes, loss, drop, widths, num_layer
    ("FTHead3", "relu", 1, "mse", 0.1, W_ODD, 4),
    ("FTHead3", "celu", 3, "bce", 0.5, W_ODD, 2),
    ("FTHead1", "relu", 1, "mse", 0.1, W_ODD, 2),
    ("FTHead1", "celu", 3, "bce", 0.5, W_ODD, 2),
    ("FTHead2", "relu", 1, "mse", 0.5, W_ODD, 2),
    ("FTHead2", "celu", 3, "bce", 0.1, W_ODD, 2),
    ("FTHead4", "relu", 1, "mse", 0.1, W_ODD, 2),
    ("FTHead4", "celu", 3, "bce", 0.5, W_ODD, 2),
    ("FTHead3", "gelu", 1, "mse", 0.1, W_ODD, 2),
    ("FTHead3", "silu", 3, "mse", 0.5, W_ODD, 2),
    ("FTHead4", "selu", 1, "bce", 0.1, W_ODD, 2),
    ("FTHead3", "celu", 1, "mse", 0.0, (256, 256, 256, 256), 2),     # p = 0 everywhere: no site draws
]


@pytest.mark.parametrize("case", CASES, ids=["-".join(map(str, c[:5])) for c in CASES])
def test_fused_finetune_step_matches_oracle_with_replayed_masks(case):
    from fragnet_b200.train.fused import FusedFineTuneStep
    fthead, act, n_classes, loss_kind, drop, widths, num_layer = case
    seed = 300 + CASES.index(case)
    hb = _case_batch(n_classes, loss_kind, seed)
    m = _model(fthead, act, n_classes, drop, widths, num_layer, seed + 1)
    fused = FusedFineTuneStep(m, lr=1e-3, loss=loss_kind)
    b = {k: v.cuda() for k, v in hb.items()}
    seed_v, off0 = _start_stream(seed + 2)
    loss = fused.forward_backward(b)
    off1 = _gen().get_offset()
    ref_loss, _, P = _oracle_step(m, hb, fthead, act, n_classes, loss_kind, drop, True, seed_v, off0, num_layer)
    assert rel_err(loss, ref_loss) <= FP32_REL_TOL
    _check_grads(_param_pairs(m.named_parameters(), P))
    # the call reserved exactly its counters: the encoder's, then the head's sites
    g = hb["y"].numel() // n_classes
    spec = _head_spec(m, fthead)
    widths_l = [tuple(dict(m.named_parameters())[n + ".weight"].shape[::-1]) for n, _, _, _ in spec]
    _, enc_span = encoder_sites(off0, num_layer, *_sizes(hb))
    span = enc_span + _head_sites(spec, widths_l, g, 0)[1]
    assert _lib_span(fused, b) == span
    draws = drop > 0 or any(pi > 0 or po > 0 for _, pi, po, _ in spec)
    assert off1 - off0 == (roundup4(span) if draws else 0)
    # evaluation in eval mode: the oracle's eval forward, predictions [G, n_classes], and no counter drawn
    m.eval()
    loss_e, preds = fused.evaluate(b, return_predictions=True)
    torch.cuda.synchronize()
    assert _gen().get_offset() == off1
    ref_e, ref_pred, _ = _oracle_step(m, hb, fthead, act, n_classes, loss_kind, drop, False, seed_v, off0, num_layer)
    assert preds.shape == (g, n_classes)
    assert rel_err(preds, ref_pred) <= FP32_REL_TOL
    assert rel_err(loss_e, ref_e) <= FP32_REL_TOL


def test_seed_and_counter_base_reach_the_head_sites():
    """The head's masks depend on the seed and on the counter base: a second step (the next counter block) and a
    re-seeded run give other gradients, and the second step matches the oracle with the masks of its own block."""
    from fragnet_b200.train.fused import FusedFineTuneStep
    hb = _case_batch(1, "mse", 90)
    m = _model("FTHead3", "relu", 1, 0.5, W_ODD, 2, 91)
    fused = FusedFineTuneStep(m, lr=1e-3)
    b = {k: v.cuda() for k, v in hb.items()}
    _start_stream(92)
    fused.forward_backward(b)
    g1 = fused.flat_g.clone()
    seed_v, mid = _seed(), _gen().get_offset()
    loss2 = fused.forward_backward(b)
    assert not torch.equal(g1, fused.flat_g)
    ref_loss, _, P = _oracle_step(m, hb, "FTHead3", "relu", 1, "mse", 0.5, True, seed_v, mid, 2)
    assert rel_err(loss2, ref_loss) <= FP32_REL_TOL
    _check_grads(_param_pairs(m.named_parameters(), P))


def test_masked_bce_without_valid_labels_is_nan_with_zero_gradients():
    from fragnet_b200.train.fused import FusedFineTuneStep
    hb = _case_batch(3, "bce", 40)
    hb["y"] = torch.full_like(hb["y"], -1.0)
    m = _model("FTHead4", "relu", 3, 0.0, W_ODD, 2, 41)
    fused = FusedFineTuneStep(m, lr=1e-3, loss="bce")
    loss = fused.forward_backward({k: v.cuda() for k, v in hb.items()})
    assert torch.isnan(loss).item()
    assert float(fused.flat_g.abs().max()) == 0.0


def _pair(fthead="FTHead3", act="celu", widths=W_ODD, seed=60):
    hb = _case_batch(1, "mse", seed)
    m1 = _model(fthead, act, 1, 0.0, widths, 2, seed + 1)
    return m1, copy.deepcopy(m1), {k: v.cuda() for k, v in hb.items()}


def test_fused_adam_equals_torch_adam_on_the_autograd_path():
    """After 1 and 5 steps at p = 0 the parameters are those of torch.optim.Adam driving model(batch) / backward."""
    from fragnet_b200.train.fused import FusedFineTuneStep
    m1, m2, b = _pair()
    fused = FusedFineTuneStep(m1, lr=1e-3)
    opt = torch.optim.Adam(m2.parameters(), lr=1e-3)
    for it in range(5):
        l1 = fused.step(b)
        opt.zero_grad()
        l2 = F.mse_loss(m2(b).view(-1), b["y"])
        l2.backward()
        opt.step()
        assert rel_err(l1, l2) <= FP32_REL_TOL, it
        if it in (0, 4):
            p2 = dict(m2.named_parameters())
            pairs = [(k, p.detach(), p2[k].detach()) for k, p in m1.named_parameters() if p2[k].grad is not None]
            _check_grads(pairs)


def test_two_identical_runs_and_single_stream_mode_give_the_same_bits():
    import os
    import subprocess
    import sys
    code = (
        "import sys, torch\n"
        "sys.path.insert(0, 'tests')\n"
        "from test_gpu_finetune_step import _model, _case_batch, W_ODD\n"
        "from fragnet_b200.train.fused import FusedFineTuneStep\n"
        "hb = _case_batch(1, 'mse', 70)\n"
        "b = {k: v.cuda() for k, v in hb.items()}\n"
        "out = []\n"
        "for _ in range(2):\n"
        "    m = _model('FTHead3', 'relu', 1, 0.2, W_ODD, 3, 71)\n"
        "    torch.manual_seed(3)\n"
        "    f = FusedFineTuneStep(m, lr=1e-3)\n"
        "    f.forward_backward(b)\n"
        "    out.append(f.flat_g.cpu().numpy().tobytes())\n"
        "assert out[0] == out[1]\n"
        "import hashlib\n"
        "print('RESULT', hashlib.sha256(out[0]).hexdigest())\n")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    digests = []
    for streams in ("0", "1"):
        env = dict(os.environ, FNB_STREAMS=streams, PYTHONPATH=root)
        r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd=root, timeout=300)
        assert r.returncode == 0, r.stderr[-2000:]
        digests.append([l for l in r.stdout.splitlines() if l.startswith("RESULT")][0].split()[1])
    assert digests[0] == digests[1]


def test_trainer_fused_path_equals_generic_loop():
    from torch.utils.data import DataLoader
    from fragnet_b200 import synth
    from fragnet_b200.dataset.data import collate_fn_pt
    from fragnet_b200.train.utils import TrainerFineTune
    mols = synth.make_dataset("esol", 48, seed=12)
    gen = torch.Generator().manual_seed(13)
    for mol in mols:
        mol.y = torch.randn(mol.y.shape, generator=gen)
    loader = DataLoader(mols, collate_fn=collate_fn_pt, batch_size=16, shuffle=False, drop_last=True)
    m1 = _model("FTHead3", "celu", 1, 0.0, W_ODD, 2, 14)
    m2 = copy.deepcopy(m1)
    o1, o2 = torch.optim.Adam(m1.parameters(), lr=1e-3), torch.optim.Adam(m2.parameters(), lr=1e-3)
    s1 = torch.optim.lr_scheduler.StepLR(o1, step_size=1, gamma=0.5)
    s2 = torch.optim.lr_scheduler.StepLR(o2, step_size=1, gamma=0.5)
    t1, t2 = TrainerFineTune(fused=True), TrainerFineTune()
    for _ in range(2):
        l1 = t1.train(m1, loader, o1, s1, "cuda", loader)
        l2 = t2.train(m2, loader, o2, s2, "cuda", loader)
        assert abs(l1 - l2) <= 1e-5 * abs(l2)
    assert t1._fused_for(m1, o1, "cuda", "mse") is not None and not t2._fused_steps
    # the optimizer's state is the fused step's (checkpointable), and the model round-trips its state_dict strictly
    st = o1.state_dict()["state"]
    assert len(st) == len(t1._fused_steps[0][2].live) and all(int(s["step"]) == 6 for s in st.values())
    p2 = dict(m2.named_parameters())
    assert max(rel_err(p, p2[k]) for k, p in m1.named_parameters()) <= 5e-4
    sd = {k: v.clone() for k, v in m1.state_dict().items()}
    m1.load_state_dict(sd, strict=True)
    v1, v2 = t1.validate(m1, loader, "cuda"), t2.validate(m2, loader, "cuda")
    assert abs(v1 - v2) <= 1e-3 * abs(v2)


def test_trainer_falls_back_silently():
    from torch.utils.data import DataLoader
    from fragnet_b200 import synth
    from fragnet_b200.dataset.data import collate_fn_pt
    from fragnet_b200.train.utils import TrainerFineTune
    loader = DataLoader(synth.make_dataset("esol", 16, seed=15), collate_fn=collate_fn_pt, batch_size=8)
    t = TrainerFineTune(fused=True)
    m = _model("FTHead3", "relu", 1, 0.0, W_ODD, 2, 16)
    sgd = torch.optim.SGD(m.parameters(), lr=1e-3)
    t.train(m, loader, sgd, None, "cuda", loader)
    assert t._fused_for(m, sgd, "cuda", "mse") is None
    prelu = _model("FTHead3", "prelu", 1, 0.0, W_ODD, 2, 17)
    adam = torch.optim.Adam(prelu.parameters(), lr=1e-3)
    t.train(prelu, loader, adam, None, "cuda", loader)
    assert t._fused_for(prelu, adam, "cuda", "mse") is None
    assert all(p.grad is not None for p in prelu.fthead.parameters())      # the generic loop trained it


def test_unsupported_models_raise():
    from fragnet_b200.model.gat import gat2_lite
    from fragnet_b200.train.fused import FusedFineTuneStep
    with pytest.raises(NotImplementedError):
        FusedFineTuneStep(_model("FTHead4", "rrelu", 1, 0.0, W_ODD, 2, 18))
    with pytest.raises(NotImplementedError):
        FusedFineTuneStep(gat2_lite.FragNetFineTune(num_layer=2).cuda())


def test_argument_errors():
    from fragnet_b200 import _abi, ops
    from fragnet_b200.train.fused import FusedFineTuneStep
    hb = _case_batch(1, "mse", 20)
    m = _model("FTHead3", "relu", 1, 0.0, W_ODD, 2, 21)
    fused = FusedFineTuneStep(m, lr=1e-3)
    b = {k: v.cuda() for k, v in hb.items()}
    lib = ops._lib()
    a, _, _, _ = fused._args(b, True, False)
    need = lib.fnb_finetune_step_workspace_bytes(C.byref(a))
    assert need > 0
    ws = torch.empty(need + 256, dtype=torch.uint8, device="cuda")
    scratch = ops._ptr(ops.scratch(ws.device))
    run = lambda args, w=ws, n=need: lib.fnb_finetune_step(C.byref(args), ops._ptr(w), n, scratch, ops._stream())
    assert lib.fnb_finetune_step(None, ops._ptr(ws), need, scratch, ops._stream()) == -1
    assert lib.fnb_finetune_step(C.byref(a), None, need, scratch, ops._stream()) == -1
    assert run(a, n=need - 256) == -4                                   # short workspace
    assert lib.fnb_finetune_step(C.byref(a), ops._ptr(ws) + 16, need, scratch, ops._stream()) == -5
    bad = _abi.CFinetuneStepArgs.from_buffer_copy(a)
    bad.target = None
    assert run(bad) == -1
    head = (_abi.CMlpLayer * 5)()
    C.memmove(head, fused._head, C.sizeof(fused._head))
    bad = _abi.CFinetuneStepArgs.from_buffer_copy(a)
    bad.head = C.cast(head, C.c_void_p)
    head[2].in_dim += 1                                                 # widths do not chain
    assert run(bad) == -2
    head[2].in_dim -= 1
    head[4].act = _abi.ACT_RELU                                         # the prediction must be a bare linear
    assert run(bad) == -3
    head[4].act = 99
    assert run(bad) == -3
    head[4].act = _abi.ACT_NONE
    head[1].p_out = 1.0
    assert run(bad) == -2
    head[1].p_out = 0.0
    bad.n_head_layers = 0
    assert run(bad) == -2
    bad = _abi.CFinetuneStepArgs.from_buffer_copy(a)
    bad.loss_kind = 7
    assert run(bad) == -3
    assert run(a) == 0
    torch.cuda.synchronize()
