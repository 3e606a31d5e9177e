"""Frozen parameters in the one-call finetuning step: ``FusedFineTuneStep`` trains only what requires a gradient, the
library stops the backward below the lowest trained layer, and ``TrainerFineTune(fused=True)`` takes the fused path
for the usual ``requires_grad = False`` finetuning set-ups.

Parity is against the float64 oracle with the library's dropout masks replayed (``_oracle_step`` of
``test_gpu_finetune_step.py``): the oracle differentiates every tensor, and the trained ones are compared."""
import copy
import ctypes as C

import pytest
import torch

from conftest import FP32_REL_TOL, rel_err
from test_gpu_dropout import _check_grads, _gen, _sizes, _start_stream, encoder_sites, roundup4
from test_gpu_finetune_step import W_ODD, _case_batch, _head_sites, _head_spec, _lib_span, _model, _oracle_step

pytestmark = pytest.mark.gpu


def _freeze(m, n_frozen_layers=0, frozen_head=()):
    """Freezes encoder layers ``0 .. n_frozen_layers - 1`` and the FTHead3 linears listed in ``frozen_head``."""
    for layer in m.pretrain.layers[:n_frozen_layers]:
        for p in layer.parameters():
            p.requires_grad_(False)
    for i in frozen_head:
        for p in m.fthead.predictor[i].parameters():
            p.requires_grad_(False)
    return m


# (encoder layers, frozen encoder layers, frozen head linears); FTHead3 with W_ODD has five linears
FREEZE_CASES = {
    "encoder": (2, 2, ()),
    "layer0_of_4": (4, 1, ()),
    "layers0to2_of_4": (4, 3, ()),
    "head0": (2, 0, (0,)),
    "encoder_and_head_but_last": (2, 2, (0, 1, 2, 3)),
}


@pytest.mark.parametrize("drop", [0.0, 0.2])
@pytest.mark.parametrize("case", list(FREEZE_CASES))
def test_frozen_step_matches_oracle_and_leaves_frozen_tensors_alone(case, drop):
    from fragnet_b200.train.fused import FusedFineTuneStep
    num_layer, k, frozen_head = FREEZE_CASES[case]
    seed = 500 + 10 * list(FREEZE_CASES).index(case) + int(drop * 10)
    hb = _case_batch(1, "mse", seed)
    m = _freeze(_model("FTHead3", "relu", 1, drop, W_ODD, num_layer, seed + 1), k, frozen_head)
    named = dict(m.named_parameters())
    frozen = {n for n, p in named.items() if not p.requires_grad}
    for n in sorted(frozen)[::3]:           # a .grad the step must leave alone
        named[n].grad = torch.randn_like(named[n])
    before = {n: (named[n].detach().clone(), None if named[n].grad is None else named[n].grad.clone()) for n in frozen}
    fused = FusedFineTuneStep(m, lr=1e-3)
    assert fused.first_trained_layer == k
    trained = {id(p) for p in fused.live}
    assert all(id(named[n]) not in trained for n in frozen)
    assert all(named[n].requires_grad for n in named if id(named[n]) in trained)
    b = {key: v.cuda() for key, v in hb.items()}
    seed_v, off0 = _start_stream(seed + 2)
    loss = fused.forward_backward(b)
    off1 = _gen().get_offset()
    ref_loss, _, P = _oracle_step(m, hb, "FTHead3", "relu", 1, "mse", drop, True, seed_v, off0, num_layer)
    assert rel_err(loss, ref_loss) <= FP32_REL_TOL
    _check_grads([(n, p.grad, P[n].grad) for n, p in named.items() if id(p) in trained])
    # the counters are those of the unfrozen step: freezing changes no mask
    spec = _head_spec(m, "FTHead3")
    widths = [tuple(named[n + ".weight"].shape[::-1]) for n, _, _, _ in spec]
    _, enc_span = encoder_sites(off0, num_layer, *_sizes(hb))
    span = enc_span + _head_sites(spec, widths, hb["y"].numel(), 0)[1]
    assert _lib_span(fused, b) == span
    assert off1 - off0 == (roundup4(span) if drop > 0 else 0)
    # predictions of the step's forward equal the oracle's eval forward in eval mode
    m.eval()
    _, preds = fused.evaluate(b, return_predictions=True)
    _, ref_pred, _ = _oracle_step(m, hb, "FTHead3", "relu", 1, "mse", drop, False, seed_v, off0, num_layer)
    assert rel_err(preds, ref_pred) <= FP32_REL_TOL
    m.train()
    fused.step(b)
    torch.cuda.synchronize()
    for n, (p0, g0) in before.items():
        assert torch.equal(named[n].detach(), p0), n
        assert (named[n].grad is None) == (g0 is None) and (g0 is None or torch.equal(named[n].grad, g0)), n


def test_freezing_shrinks_the_workspace_and_skips_the_encoder_backward():
    from torch.profiler import ProfilerActivity, profile

    from fragnet_b200 import ops
    from fragnet_b200.train.fused import FusedFineTuneStep
    hb = _case_batch(1, "mse", 80)
    b = {k: v.cuda() for k, v in hb.items()}
    lib = ops._lib()

    def workspace(k):
        m = _freeze(_model("FTHead3", "relu", 1, 0.1, W_ODD, 4, 81), k)
        a, _, _, _ = FusedFineTuneStep(m, lr=1e-3)._args(b, True, False)
        return lib.fnb_finetune_step_workspace_bytes(C.byref(a))
    full, lower, encoder = workspace(0), workspace(2), workspace(4)
    assert full > lower > encoder > 0

    def kernels(k):
        fused = FusedFineTuneStep(_freeze(_model("FTHead3", "relu", 1, 0.1, W_ODD, 4, 82), k), lr=1e-3)
        fused.step(b)                               # warm-up outside the trace
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fused.step(b)
            torch.cuda.synchronize()
        return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    encoder_bwd = ("k_gat_bwd_", "k_edge_table_bwd", "k_tc_dw")
    names = kernels(0)
    assert all(any(s in n for n in names) for s in encoder_bwd), sorted(set(names))     # the check can see them
    names = kernels(4)
    assert names and not [n for n in names if any(s in n for s in encoder_bwd)]


def _loader(seed=12):
    from torch.utils.data import DataLoader
    from fragnet_b200 import synth
    from fragnet_b200.dataset.data import collate_fn_pt
    mols = synth.make_dataset("esol", 48, seed=seed)
    gen = torch.Generator().manual_seed(seed + 1)
    for mol in mols:
        mol.y = torch.randn(mol.y.shape, generator=gen)
    return DataLoader(mols, collate_fn=collate_fn_pt, batch_size=16, shuffle=False, drop_last=True)


def _close(m1, m2):
    p2 = dict(m2.named_parameters())
    return max(rel_err(p, p2[k]) for k, p in m1.named_parameters())


def test_trainer_with_a_frozen_encoder_takes_the_fused_path():
    from fragnet_b200.train.utils import TrainerFineTune
    loader = _loader()
    m1 = _freeze(_model("FTHead3", "celu", 1, 0.0, W_ODD, 2, 14), 2)
    m2 = copy.deepcopy(m1)
    enc0 = {k: v.clone() for k, v in m1.pretrain.state_dict().items()}
    o1, o2 = torch.optim.Adam(m1.fthead.parameters(), lr=1e-3), torch.optim.Adam(m2.fthead.parameters(), lr=1e-3)
    t1, t2 = TrainerFineTune(fused=True), TrainerFineTune()
    for _ in range(2):
        l1 = t1.train(m1, loader, o1, None, "cuda", loader)
        l2 = t2.train(m2, loader, o2, None, "cuda", loader)
        assert abs(l1 - l2) <= 1e-5 * abs(l2)
    fs = t1._fused_for(m1, o1, "cuda", "mse")
    assert fs is not None and fs.first_trained_layer == 2
    assert _close(m1, m2) <= 5e-4
    assert all(torch.equal(v, enc0[k]) for k, v in m1.pretrain.state_dict().items())
    # a trainable encoder that the optimizer does not hold: the generic loop's semantics, so no fused step
    m3 = _model("FTHead3", "celu", 1, 0.0, W_ODD, 2, 15)
    o3 = torch.optim.Adam(m3.fthead.parameters(), lr=1e-3)
    t3 = TrainerFineTune(fused=True)
    assert t3._fused_for(m3, o3, "cuda", "mse") is None
    assert all(p.grad is None for p in m3.parameters())      # nothing was re-homed on the way


def test_unfreezing_between_epochs_rebuilds_the_step():
    """Encoder frozen for a warm-up epoch, then unfrozen: the fused step is rebuilt, trains the encoder from then on,
    and matches the generic loop, whose Adam starts the newly trained tensors at step 1."""
    from fragnet_b200.train.utils import TrainerFineTune
    loader = _loader(20)
    m1 = _freeze(_model("FTHead3", "relu", 1, 0.0, W_ODD, 2, 21), 2)
    m2 = copy.deepcopy(m1)
    o1, o2 = torch.optim.Adam(m1.parameters(), lr=1e-3), torch.optim.Adam(m2.parameters(), lr=1e-3)
    t1, t2 = TrainerFineTune(fused=True), TrainerFineTune()
    enc0 = {k: v.clone() for k, v in m1.pretrain.state_dict().items()}
    t1.train(m1, loader, o1, None, "cuda", loader)
    t2.train(m2, loader, o2, None, "cuda", loader)
    fs_warm = t1._fused_for(m1, o1, "cuda", "mse")
    assert fs_warm is not None and fs_warm.first_trained_layer == 2
    assert all(torch.equal(v, enc0[k]) for k, v in m1.pretrain.state_dict().items())
    for m in (m1, m2):
        for p in m.pretrain.parameters():
            p.requires_grad_(True)
    assert not fs_warm.bound_to_model()
    l1 = t1.train(m1, loader, o1, None, "cuda", loader)
    l2 = t2.train(m2, loader, o2, None, "cuda", loader)
    fs = t1._fused_for(m1, o1, "cuda", "mse")
    assert fs is not None and fs is not fs_warm and fs.first_trained_layer == 0
    assert abs(l1 - l2) <= 1e-5 * abs(l2)
    assert not torch.equal(m1.pretrain.layers[0].a.detach(), enc0["layers.0.a"])
    assert _close(m1, m2) <= 5e-4
    st = o1.state_dict()["state"]
    steps = {int(s["step"]) for s in st.values()}
    assert steps == {3, 6}, steps                           # 3 batches per epoch: encoder 3 steps, head 6


def test_unsupported_freezing_patterns_raise_and_the_trainer_falls_back():
    from fragnet_b200.train.fused import FusedFineTuneStep
    from fragnet_b200.train.utils import TrainerFineTune
    above = _model("FTHead3", "relu", 1, 0.0, W_ODD, 4, 30)
    for p in above.pretrain.layers[2].parameters():             # frozen layer above trained ones
        p.requires_grad_(False)
    mixed = _model("FTHead3", "relu", 1, 0.0, W_ODD, 2, 31)
    mixed.pretrain.layers[1].a.requires_grad_(False)            # one tensor of a trained layer
    half = _model("FTHead3", "relu", 1, 0.0, W_ODD, 2, 32)
    half.fthead.predictor[1].weight.requires_grad_(False)       # weight without its bias
    nothing = _freeze(_model("FTHead3", "relu", 1, 0.0, W_ODD, 2, 33), 2, range(5))
    loader = _loader(34)
    for m in (above, mixed, half, nothing):
        with pytest.raises(NotImplementedError):
            FusedFineTuneStep(m)
        if m is nothing:
            continue
        t = TrainerFineTune(fused=True)
        opt = torch.optim.Adam([p for p in m.parameters() if p.requires_grad], lr=1e-3)
        t.train(m, loader, opt, None, "cuda", loader)
        assert t._fused_for(m, opt, "cuda", "mse") is None
        assert all(p.grad is not None for p in m.fthead.parameters() if p.requires_grad)   # the generic loop trained


def test_argument_errors_of_frozen_steps():
    from fragnet_b200 import _abi, ops
    from fragnet_b200.train.fused import FusedFineTuneStep
    hb = _case_batch(1, "mse", 40)
    b = {k: v.cuda() for k, v in hb.items()}
    fused = FusedFineTuneStep(_model("FTHead3", "relu", 1, 0.0, W_ODD, 2, 41), lr=1e-3)
    lib = ops._lib()
    a, _, _, _ = fused._args(b, True, False)
    need = lib.fnb_finetune_step_workspace_bytes(C.byref(a))
    ws = torch.empty(need + 256, dtype=torch.uint8, device="cuda")
    scratch = ops._ptr(ops.scratch(ws.device))
    run = lambda args: lib.fnb_finetune_step(C.byref(args), ops._ptr(ws), need, scratch, ops._stream())
    for k in (-1, 3):                                            # outside 0 .. n_layers
        bad = _abi.CFinetuneStepArgs.from_buffer_copy(a)
        bad.first_trained_layer = k
        assert run(bad) == -2
        assert lib.fnb_finetune_step_workspace_bytes(C.byref(bad)) == 0
        assert lib.fnb_finetune_step_rng_span(C.byref(bad)) == 0
    head = (_abi.CMlpLayer * len(fused._head))()
    C.memmove(head, fused._head, C.sizeof(fused._head))
    bad = _abi.CFinetuneStepArgs.from_buffer_copy(a)
    bad.head, bad.first_trained_layer = C.cast(head, C.c_void_p), 2
    head[0].dW = None                                            # dW without db: neither trained nor frozen
    assert run(bad) == -1
    for h in head:
        h.dW = h.db = None
    assert run(bad) == -3                                        # a backward that trains nothing
    bad.backward = 0
    assert run(bad) == 0                                         # ... is a fine forward
    C.memmove(head, fused._head, C.sizeof(fused._head))
    bad.first_trained_layer, bad.backward, bad.layer_grads = 0, 1, None
    assert run(bad) == -1                                        # a trained encoder needs its gradient pointers
    bad.first_trained_layer = 2
    assert run(bad) == 0                                         # a frozen one does not; the head input gets none
    torch.cuda.synchronize()


def test_frozen_lower_layers_are_deterministic_in_both_stream_modes():
    import os
    import subprocess
    import sys
    code = (
        "import sys, torch, hashlib\n"
        "sys.path.insert(0, 'tests')\n"
        "from test_gpu_finetune_step import _model, _case_batch, W_ODD\n"
        "from test_gpu_finetune_freeze import _freeze\n"
        "from fragnet_b200.train.fused import FusedFineTuneStep\n"
        "b = {k: v.cuda() for k, v in _case_batch(1, 'mse', 70).items()}\n"
        "out = []\n"
        "for _ in range(2):\n"
        "    m = _freeze(_model('FTHead3', 'relu', 1, 0.2, W_ODD, 3, 71), 1, (0,))\n"
        "    torch.manual_seed(3)\n"
        "    f = FusedFineTuneStep(m, lr=1e-3)\n"
        "    f.forward_backward(b)\n"
        "    out.append(f.flat_g.cpu().numpy().tobytes())\n"
        "assert out[0] == out[1]\n"
        "print('RESULT', hashlib.sha256(out[0]).hexdigest())\n")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    digests = []
    for streams in ("0", "1"):
        env = dict(os.environ, FNB_STREAMS=streams, PYTHONPATH=root)
        r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd=root, timeout=300)
        assert r.returncode == 0, r.stderr[-2000:]
        digests.append([l for l in r.stdout.splitlines() if l.startswith("RESULT")][0].split()[1])
    assert digests[0] == digests[1]
