"""Pretraining heads + loss programs (heads.cu) against the same heads written as separate ``nn.Linear`` calls
(the arrangement of the reference, fragnet/model/gat/pretrain_heads.py:64-102) and against the CPU oracle."""
import pytest
import torch

from conftest import FP32_REL_TOL, grad_errs, rel_err

pytestmark = pytest.mark.gpu
GRAD_TOL = 5e-5


def _batch(shape, n, seed):
    from fragnet_b200 import synth
    from fragnet_b200.dataset.data import collate_fn_pt
    mols = synth.make_dataset(shape, n, seed=seed) + [synth.handmade(k) for k in ("two_atom", "ion_pair", "two_frag")]
    return {k: v.cuda() for k, v in collate_fn_pt(mols).items()}


def _inputs(b, seed):
    gen = torch.Generator().manual_seed(seed)
    na, nf, ea = b["x_atoms"].shape[0], b["x_frags"].shape[0], b["edge_index"].shape[1]
    mk = lambda n: torch.randn(n, 128, generator=gen).cuda().requires_grad_()
    return mk(na), mk(nf), mk(ea)


def _away_from_relu_kinks(head, stack, x, margin=1e-4, seed=0):
    """Re-draws the rows of ``x`` for which some ReLU pre-activation of ``stack`` lies within ``margin`` of zero.

    The gradient of ReLU is discontinuous at 0: two correct fp32 evaluations whose pre-activations differ by 1e-7 can
    fall on different sides and then differ by a whole weight column in that row's input gradient (seen with the
    3xTF32 first layers: one row of 15 954, pre-activation 5.8e-8).  Parity of gradients is only defined away from
    the kink, so the max-norm gradient check runs on inputs conditioned to keep 100x the arithmetic error of distance
    from it; about 2 % of the rows get re-drawn."""
    gen = torch.Generator().manual_seed(1000 + seed)
    layers = [(l.weight.detach().double().cpu(), l.bias.detach().double().cpu()) for l in list(stack)[:-1]]
    x = x.detach().cpu().clone()
    for _ in range(20):
        h, close = x.double(), torch.zeros(x.shape[0], dtype=torch.bool)
        for W, b in layers:
            pre = h @ W.t() + b
            close |= pre.abs().amin(1) < margin
            h = pre.clamp_min(0)
        if not bool(close.any()):
            break
        x[close] = torch.randn(int(close.sum()), x.shape[1], generator=gen)
    assert not bool(close.any())
    return x.cuda().requires_grad_()


def _head(seed):
    from fragnet.model.gat.pretrain_heads import PretrainTask
    torch.manual_seed(seed)
    return PretrainTask(128, 1).cuda()


def _fro_errs(pairs):
    """TF32 first layers flip the ReLU mask of pre-activations within ~1e-3 of zero, which moves single gradient
    entries by whole weight columns: the TF32 gradient check is in the Frobenius norm, not the max norm."""
    out = {}
    for k, a, b in pairs:
        a, b = a.detach().double().cpu(), b.detach().double().cpu()
        out[k] = float((a - b).norm() / b.norm().clamp_min(1e-30))
    return out


@pytest.mark.parametrize("precision,tol,gtol", [("fp32", FP32_REL_TOL, GRAD_TOL), ("tf32", 2e-3, 6e-2)])
@pytest.mark.parametrize("shape,n", [("esol", 9), ("unimol", 300)])
def test_heads_forward_backward_match_separate_linears(precision, tol, gtol, shape, n):
    from fragnet_b200 import config
    old_tf32 = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    config.set_precision(precision)
    try:
        b = _batch(shape, n, 11)
        head = _head(5)
        xa, xf, xe = _inputs(b, 7)
        xa, xe = _away_from_relu_kinks(head, head.ba_layers, xa, seed=1), _away_from_relu_kinks(head, head.da_layers, xe, seed=2)
        outs = head(xa, xf, xe, b)
        gen = torch.Generator().manual_seed(3)
        ws = [torch.randn(o.shape, generator=gen).cuda() for o in outs]
        sum((o * w).sum() for o, w in zip(outs[1:], ws[1:])).backward()
        got_in = [t.grad.clone() for t in (xa, xf, xe)]
        got_p = {k: p.grad.clone() for k, p in head.named_parameters() if p.grad is not None}
        for t in (xa, xf, xe):
            t.grad = None
        head.zero_grad(set_to_none=True)
        ref = head._forward_linears(xa, xf, xe, b)
        sum((o * w).sum() for o, w in zip(ref[1:], ws[1:])).backward()
        for name, a, r in zip(("bond_length", "bond_angle", "dihedral", "energy"), outs, ref):
            assert a.shape == r.shape, name
            assert rel_err(a, r) <= tol, (name, rel_err(a, r))
        # the energy head is one exact-FP32 kernel in every precision mode
        assert rel_err(outs[3], ref[3]) <= FP32_REL_TOL, rel_err(outs[3], ref[3])
        pairs = [(nm, g, t.grad) for nm, g, t in zip(("x_atoms", "x_frags", "edge_feat"), got_in, (xa, xf, xe))]
        ref_p = {k: p.grad for k, p in head.named_parameters() if p.grad is not None}
        assert set(got_p) == set(ref_p) and not any(k.startswith("bl_") for k in got_p)
        pairs += [(k, got_p[k], ref_p[k]) for k in ref_p]
        errs = grad_errs(pairs) if precision == "fp32" else _fro_errs(pairs)
        bad = {k: v for k, v in errs.items() if v > gtol}
        assert not bad, bad
    finally:
        config.set_precision("fp32")
        torch.backends.cuda.matmul.allow_tf32 = old_tf32


def test_bond_length_gradient_path_and_cpu_inputs():
    """``bond_length_grad=True`` keeps the bond-length head differentiable; CPU inputs come back on the CPU."""
    b = _batch("esol", 5, 2)
    head = _head(1)
    xa, xf, xe = _inputs(b, 4)
    outs = head(xa, xf, xe, b, bond_length_grad=True)
    outs[0].sum().backward()
    assert head.bl_reduce_layer.weight.grad is not None and xa.grad is not None
    fused = head(xa, xf, xe, b)
    assert not fused[0].requires_grad and rel_err(fused[0], outs[0]) <= FP32_REL_TOL
    cpu = head(xa.detach().cpu(), xf.detach().cpu(), xe.detach().cpu(), {k: v.cpu() for k, v in b.items()})
    assert all(t.device.type == "cpu" for t in cpu) and rel_err(cpu[1], fused[1]) <= FP32_REL_TOL


def test_heads_tiny_batch():
    """Two three-atom ion pairs (2 directed bonds, 2 molecules): far fewer rows than one tile of any kernel."""
    from fragnet_b200 import synth
    from fragnet_b200.dataset.data import collate_fn_pt
    ion = synth.handmade("ion_pair")
    b = {k: v.cuda() for k, v in collate_fn_pt([ion, ion]).items()}
    head = _head(2)
    xa, xf, xe = _inputs(b, 1)
    outs = head(xa, xf, xe, b)
    ref = head._forward_linears(xa, xf, xe, b)
    for a, r in zip(outs, ref):
        assert a.shape == r.shape and rel_err(a, r) <= FP32_REL_TOL
    (outs[1].sum() + outs[3].sum() + outs[2].sum()).backward()
    assert torch.isfinite(xa.grad).all()


def test_fused_loss_matches_torch_and_is_deterministic():
    from fragnet_b200.train.pretrain_utils import pretrain_loss
    gen = torch.Generator().manual_seed(0)
    mk = lambda *s: torch.randn(*s, generator=gen).cuda()
    preds = [mk(700, 1), mk(333, 1).requires_grad_(), mk(700, 1).requires_grad_(), mk(40, 1).requires_grad_()]
    batch = {"dh_angl": mk(700, 1), "bnd_angl": mk(333, 1), "y": mk(40)}
    mse = torch.nn.MSELoss()
    loss = pretrain_loss(mse, preds, batch)
    (3.0 * loss).backward()
    got = [p.grad.clone() for p in preds[1:]]
    for p in preds[1:]:
        p.grad = None
    l_dh = mse(preds[2], batch["dh_angl"])
    ref = l_dh + mse(preds[1], batch["bnd_angl"]) + l_dh + mse(preds[3].view(-1), batch["y"])
    (3.0 * ref).backward()
    assert rel_err(loss, ref) <= 2e-6
    for g, p in zip(got, preds[1:]):
        assert rel_err(g, p.grad) <= 2e-6
    again = pretrain_loss(mse, preds, batch)
    assert torch.equal(again, loss)
    # any other criterion takes the generic path
    l1 = pretrain_loss(torch.nn.L1Loss(), preds, batch)
    assert l1.requires_grad and float(l1.detach()) > 0


def test_pretrain_model_training_step_matches_oracle():
    """Whole FragNetPreTrain step (encoder + fused heads + fused loss), drop_ratio 0, against the CPU oracle."""
    from fragnet.model.gat.gat2_pretrain import FragNetPreTrain
    from fragnet_b200 import synth
    from fragnet_b200.dataset.data import collate_fn_pt
    from fragnet_b200.train.pretrain_utils import pretrain_loss
    from oracle import gat2_oracle as O
    torch.manual_seed(8)
    hb = collate_fn_pt(synth.make_dataset("unimol", 20, seed=4) + [synth.handmade("ion_pair")])
    gen = torch.Generator().manual_seed(5)
    for k in ("bnd_lngth", "bnd_angl", "dh_angl"):
        hb[k] = torch.randn(hb[k].shape, generator=gen)
    hb["y"] = torch.randn(hb["y"].shape, generator=gen)
    m = FragNetPreTrain(num_layer=2, drop_ratio=0.0, edge_features=17)
    P = O.params_from_module(m)
    m = m.cuda().train()
    b = {k: v.cuda() for k, v in hb.items()}
    preds = m(b)
    loss = pretrain_loss(torch.nn.MSELoss(), preds, b)
    loss.backward()
    ref_preds = O.pretrain_forward(P, hb, num_layer=2)
    ref_loss = O.pretrain_loss(ref_preds, hb)
    ref_loss.backward()
    for a, r in zip(preds, ref_preds):
        assert rel_err(a, r) <= FP32_REL_TOL
    assert rel_err(loss, ref_loss) <= FP32_REL_TOL
    pairs = [(k, p.grad, P[k].grad) for k, p in m.named_parameters() if p.grad is not None]
    assert {k for k, _, _ in pairs} == {k for k, v in P.items() if v.grad is not None}
    bad = {k: v for k, v in grad_errs(pairs).items() if v > GRAD_TOL}
    assert not bad, bad


def _pretrain_pair(seed, num_layer=2, drop=0.0):
    """Two identically initialised FragNetPreTrain models and a batch with random targets."""
    import copy
    from fragnet.model.gat.gat2_pretrain import FragNetPreTrain
    from fragnet_b200 import synth
    from fragnet_b200.dataset.data import collate_fn_pt
    torch.manual_seed(seed)
    hb = collate_fn_pt(synth.make_dataset("unimol", 40, seed=seed) + [synth.handmade("ion_pair")])
    gen = torch.Generator().manual_seed(seed + 1)
    for k in ("bnd_lngth", "bnd_angl", "dh_angl"):
        hb[k] = torch.randn(hb[k].shape, generator=gen)
    hb["y"] = torch.randn(hb["y"].shape, generator=gen)
    m1 = FragNetPreTrain(num_layer=num_layer, drop_ratio=drop, edge_features=17).cuda().train()
    m2 = copy.deepcopy(m1)
    return m1, m2, {k: v.cuda() for k, v in hb.items()}


def test_fused_step_equals_autograd_path_and_torch_adam():
    """fnb_pretrain_step + fnb_adam_step against model(batch) / loss.backward() / torch.optim.Adam on a twin model."""
    from fragnet_b200.train.fused import FusedPretrainStep
    from fragnet_b200.train.pretrain_utils import pretrain_loss
    m1, m2, b = _pretrain_pair(3)
    fused = FusedPretrainStep(m1, lr=1e-3)
    opt = torch.optim.Adam(m2.parameters(), lr=1e-3)
    for it in range(3):
        loss1 = fused.step(b)
        opt.zero_grad()
        loss2 = pretrain_loss(torch.nn.MSELoss(), m2(b), b)
        loss2.backward()
        if it == 0:
            g1 = {k: p.grad.clone() for k, p in m1.named_parameters() if p.grad is not None}
            g2 = {k: p.grad for k, p in m2.named_parameters() if p.grad is not None}
            assert set(g1) == set(g2)
            # (the fused step forms the predictions inside the backward tails: same arithmetic, another summation order)
            bad = {k: v for k, v in grad_errs([(k, g1[k], g2[k]) for k in g2]).items() if v > 1e-5}
            assert not bad, bad
        opt.step()
        assert rel_err(loss1, loss2) <= 1e-6, it
    p1, p2 = dict(m1.named_parameters()), dict(m2.named_parameters())
    worst = max(rel_err(p1[k], p2[k]) for k in p2)
    assert worst <= 1e-4, worst
    # the model is still an ordinary nn.Module: state_dict round trip, eval-mode forward, evaluate() with predictions
    sd = {k: v.clone() for k, v in m1.state_dict().items()}
    m1.load_state_dict(sd, strict=True)
    m1.eval()
    loss_e, preds = fused.evaluate(b, return_predictions=True)
    with torch.no_grad():
        ref = m1(b)
    for a, r in zip(preds, ref):
        assert rel_err(a, r) <= 1e-6
    assert rel_err(loss_e, pretrain_loss(torch.nn.MSELoss(), ref, b)) <= 1e-6


@pytest.mark.parametrize("kinds", [("two_frag",), ("ion_pair", "two_atom", "single_frag"), None,
                                   ("two_atom", "ion_pair", "two_frag", "single_frag") * 500])
def test_fused_step_on_tiny_and_ragged_batches(kinds):
    """One molecule, three molecules, nine molecules (a partial 8-molecule tile of the fused energy-head kernel), 2 000
    molecules (250 tiles on 222 CTAs: more than one tile per CTA): loss and gradients of the one-call step against the
    autograd path."""
    import copy
    from fragnet.model.gat.gat2_pretrain import FragNetPreTrain
    from fragnet_b200 import synth
    from fragnet_b200.dataset.data import collate_fn_pt
    from fragnet_b200.train.fused import FusedPretrainStep
    from fragnet_b200.train.pretrain_utils import pretrain_loss
    mols = [synth.handmade(k) for k in kinds] if kinds else synth.make_dataset("esol", 9, seed=31)
    hb = collate_fn_pt(mols)
    gen = torch.Generator().manual_seed(3)
    for k in ("bnd_angl", "dh_angl"):
        hb[k] = torch.randn(hb[k].shape, generator=gen)
    hb["y"] = torch.randn(hb["y"].shape, generator=gen)
    b = {k: v.cuda() for k, v in hb.items()}
    torch.manual_seed(17)
    m1 = FragNetPreTrain(num_layer=2, drop_ratio=0.0, edge_features=17).cuda().train()
    m2 = copy.deepcopy(m1)
    loss1 = FusedPretrainStep(m1, lr=1e-3).forward_backward(b)
    loss2 = pretrain_loss(torch.nn.MSELoss(), m2(b), b)
    loss2.backward()
    assert rel_err(loss1, loss2) <= 1e-6
    g1 = {k: p.grad for k, p in m1.named_parameters() if p.grad is not None}
    g2 = {k: p.grad for k, p in m2.named_parameters() if p.grad is not None}
    assert set(g1) == set(g2)
    bad = {k: v for k, v in grad_errs([(k, g1[k], g2[k]) for k in g2]).items() if v > 1e-5}
    assert not bad, bad


def test_plan_prefetch_gives_bitwise_the_same_training_run():
    """The on-device collate of the next batch queued underneath the running step (FusedPretrainStep.prefetch_plan,
    fnb_pretrain_plan_prefetch) is the same plan as the one a step builds for itself: losses and parameters of a
    run over alternating batches are bitwise equal with and without it; a batch the prefetch was not made for (or one
    that needs a dtype conversion) falls back to the in-step collate."""
    import copy
    from fragnet_b200 import synth
    from fragnet_b200.dataset.data import collate_fn_pt
    from fragnet_b200.train.fused import FusedPretrainStep
    m1, m2, b0 = _pretrain_pair(9, num_layer=3, drop=0.1)
    hb = collate_fn_pt(synth.make_dataset("unimol", 23, seed=77) + [synth.handmade("two_frag")])
    b1 = {k: v.cuda() for k, v in hb.items()}
    batches = [b0, b1, b0, b1, b1, b0]
    runs = []
    for model, use in ((m1, True), (m2, False)):
        torch.manual_seed(5)
        fused = FusedPretrainStep(model, lr=1e-3)
        losses = []
        for i, b in enumerate(batches):
            nxt = batches[i + 1] if use and i + 1 < len(batches) else None
            if use and i == 3:
                nxt = b0                       # a wrong guess: the next step gets b1 and must collate by itself
            losses.append(fused.step(b, next_batch=nxt))
        runs.append(([float(x) for x in losses], {k: v.clone() for k, v in model.state_dict().items()}, fused.plan_hits))
    assert runs[0][2] == 4 and runs[1][2] == 0       # steps 1, 2, 3 and 5 found their plan; step 4 was guessed wrong
    assert runs[0][0] == runs[1][0]
    for k in runs[0][1]:
        assert torch.equal(runs[0][1][k], runs[1][1][k]), k
    # two prefetches in a row (the second replaces the first, never the arena of the step in flight), then the step
    fused = FusedPretrainStep(m1, lr=1e-3)
    fused.step(b0, next_batch=b1)
    fused.step(b1)                                  # reads the prefetched arena
    assert fused.prefetch_plan(b0) and fused.prefetch_plan(b1) and fused.prefetch_plan(b0)
    hits = fused.plan_hits
    m1.eval()
    l_pre = float(fused.evaluate(b0))
    assert fused.plan_hits == hits + 1
    assert l_pre == float(fused.evaluate(b0))       # the same loss from a plan built inside the call
    m1.train()
    # a batch with int32 indices would need a conversion: no prefetch, the step still works
    fused = FusedPretrainStep(m1, lr=1e-3)
    narrow = dict(b0)
    narrow["edge_index"] = b0["edge_index"].to(torch.int32)
    assert fused.prefetch_plan(narrow) is False
    m1.eval()
    assert float(fused.evaluate(narrow)) == float(fused.evaluate(b0))


def test_plan_prefetch_in_single_stream_mode_is_declined():
    """FNB_STREAMS=1 (everything on the caller's stream): fnb_pretrain_plan_prefetch queues nothing and says so, the
    step collates by itself and trains to the same losses (a fresh process: the stream mode is read once)."""
    import os
    import subprocess
    import sys
    code = (
        "import torch, sys\n"
        "sys.path.insert(0, 'tests')\n"
        "from test_gpu_heads import _pretrain_pair\n"
        "from fragnet_b200.train.fused import FusedPretrainStep\n"
        "m1, m2, b = _pretrain_pair(21, num_layer=2, drop=0.0)\n"
        "f = FusedPretrainStep(m1, lr=1e-3)\n"
        "ok = f.prefetch_plan(b)\n"
        "losses = [float(f.step(b, next_batch=b)) for _ in range(3)]\n"
        "print('RESULT', ok, f.plan_hits, ' '.join(repr(x) for x in losses))\n")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    outs = []
    for streams in ("1", "0"):
        env = dict(os.environ, FNB_STREAMS=streams, PYTHONPATH=root)
        r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd=root, timeout=300)
        assert r.returncode == 0, r.stderr[-2000:]
        outs.append([l for l in r.stdout.splitlines() if l.startswith("RESULT")][0].split())
    assert outs[0][1] == "False" and outs[0][2] == "0"          # single stream: declined, no hits
    assert outs[1][1] == "True" and outs[1][2] == "3"           # default: every step found its plan
    assert outs[0][3:] == outs[1][3:]                           # and the same training run either way


def test_fused_step_dropout_training_is_seeded_and_finite():
    from fragnet_b200 import ops
    from fragnet_b200.train.fused import FusedPretrainStep
    losses = []
    for _ in range(2):
        torch.manual_seed(11)          # re-seeding restarts the dropout counter as well (torch's CUDA generator offset)
        m1, _, b = _pretrain_pair(5, num_layer=4, drop=0.2)
        fused = FusedPretrainStep(m1, lr=1e-4)
        losses.append([float(fused.step(b)) for _ in range(3)])
    assert losses[0] == losses[1] and all(x == x and x < 1e6 for x in losses[0])


def test_trainer_fused_path_equals_generic_loop():
    """The reference's Trainer interface (pretrain_utils.py:4-57) through a DataLoader: the fused path (one library
    call per batch + prefetcher) and the generic nn.Module / autograd / torch.optim.Adam loop train twin models alike."""
    import copy
    from torch.utils.data import DataLoader
    from fragnet.model.gat.gat2_pretrain import FragNetPreTrain
    from fragnet.train.pretrain.pretrain_utils import Trainer
    from fragnet_b200 import synth
    from fragnet_b200.dataset.data import collate_fn_pt
    mols = synth.make_dataset("unimol", 48, seed=9)
    gen = torch.Generator().manual_seed(2)
    for m in mols:
        m.bnd_angl = torch.randn(m.bnd_angl.shape, generator=gen)
        m.dh_angl = torch.randn(m.dh_angl.shape, generator=gen)
        m.y = torch.randn(m.y.shape, generator=gen)
    loader = DataLoader(mols, collate_fn=collate_fn_pt, batch_size=16, shuffle=False, drop_last=True)
    torch.manual_seed(4)
    m1 = FragNetPreTrain(num_layer=2, drop_ratio=0.0, edge_features=17).cuda()
    m2 = copy.deepcopy(m1)
    o1 = torch.optim.Adam(m1.parameters(), lr=1e-3)
    o2 = torch.optim.Adam(m2.parameters(), lr=1e-3)
    t1, t2 = Trainer(torch.nn.MSELoss()), Trainer(torch.nn.MSELoss(), fused=False)
    for _ in range(2):
        l1 = t1.train(m1, loader, o1, "cuda")
        l2 = t2.train(m2, loader, o2, "cuda")
        assert abs(l1 - l2) <= 1e-5 * abs(l2)
    assert t1._fused_for(m1, o1, "cuda") is not None and not t2._fused_steps
    p2 = dict(m2.named_parameters())
    # six Adam steps: the update is ~lr * sign(g) for small g, so rounding-level gradient differences show up at 1e-5
    assert max(rel_err(p, p2[k]) for k, p in m1.named_parameters()) <= 5e-4
    v1, v2 = t1.validate(loader, m1, "cuda"), t2.validate(loader, m2, "cuda")
    assert abs(v1 - v2) <= 1e-5 * abs(v2)


def test_trainer_keeps_the_callers_optimizer_truthful_and_survives_moves():
    """The fused path must not hide the optimizer state (ADVICE r1): ``optimizer.state`` holds views of the fused moment
    buffers and the step count, a state dict saved from it resumes into a fresh trainer with identical results, an
    ArenaLoader can drive ``train`` (its ``dataset`` gives the divisor), and moving the model afterwards falls back to
    the generic loop instead of training an orphaned buffer."""
    import copy
    import warnings
    from fragnet.model.gat.gat2_pretrain import FragNetPreTrain
    from fragnet.train.pretrain.pretrain_utils import Trainer
    from fragnet_b200 import synth
    from fragnet_b200.dataset.arena import ArenaLoader, MoleculeArena
    mols = synth.make_dataset("unimol", 32, seed=19)
    arena = MoleculeArena(mols, "cuda")
    loader = ArenaLoader(arena, batch_size=16)
    assert len(loader.dataset) == 32
    torch.manual_seed(6)
    m1 = FragNetPreTrain(num_layer=2, drop_ratio=0.0, edge_features=17).cuda()
    o1 = torch.optim.Adam(m1.parameters(), lr=1e-3)
    t1 = Trainer(torch.nn.MSELoss())
    t1.train(m1, loader, o1, "cuda")
    fs = t1._fused_for(m1, o1, "cuda")
    assert fs is not None and fs.t == 2
    live = [p for p in m1.parameters() if p in o1.state]
    assert len(live) == len(fs.live) and all(int(o1.state[p]["step"]) == 2 for p in live)
    assert all(o1.state[p]["exp_avg"].data_ptr() >= fs.exp_avg.data_ptr() for p in live)
    assert float(sum(o1.state[p]["exp_avg_sq"].sum() for p in live)) > 0
    # checkpoint -> fresh model / optimizer / trainer -> one more epoch == continuing the original
    ck_m, ck_o = copy.deepcopy(m1.state_dict()), copy.deepcopy(o1.state_dict())
    m2 = FragNetPreTrain(num_layer=2, drop_ratio=0.0, edge_features=17).cuda()
    m2.load_state_dict(ck_m)
    o2 = torch.optim.Adam(m2.parameters(), lr=1e-3)
    o2.load_state_dict(ck_o)
    t2 = Trainer(torch.nn.MSELoss())
    l1 = t1.train(m1, loader, o1, "cuda")
    l2 = t2.train(m2, loader, o2, "cuda")
    assert t2._fused_for(m2, o2, "cuda").t == 4
    assert l1 == l2
    for (k, a), (_, b) in zip(m1.state_dict().items(), m2.state_dict().items()):
        assert torch.equal(a, b), k
    # a moved model: the binding check trips, the generic loop takes over (and still trains)
    m1.cpu()
    m1.cuda()
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        l3 = t1.train(m1, loader, o1, "cuda")
    assert any("falling back" in str(x.message) for x in w) and l3 == l3
    assert t1._fused_for(m1, o1, "cuda") is None
