"""Tensor-core (tcgen05) projection path: TF32 mode within its stated tolerance against fp32 torch, and the 3xTF32
(error-compensated) mode -- the arithmetic of the default ``fp32`` parity mode -- against float64."""
import pytest
import torch
import torch.nn.functional as F

from conftest import rel_err

pytestmark = pytest.mark.gpu
TF32_TOL = 2e-3      # stated tolerance of the tensor-core mode: TF32 operands (10-bit mantissa), FP32 accumulate
X3_TOL = 4e-6        # 3xTF32: hi*hi + hi*lo + lo*hi, FP32 accumulate (measured 0.5e-6..2.2e-6, largest at K = 256)


@pytest.mark.parametrize("n,K", [(1, 128), (127, 128), (129, 128), (1000, 128), (54001, 128), (300, 32), (300, 64),
                                 (300, 256), (40000, 128), (9473, 128), (9473, 256)])
def test_x3_projection_forward_is_fp32_grade(n, K):
    from fragnet_b200 import ops
    g = torch.Generator().manual_seed(1000 + n + K)
    x = torch.randn(n, K, generator=g) * torch.exp(torch.randn(n, 1, generator=g))     # rows of mixed magnitude
    W = torch.randn(128, K, generator=g) * 0.2
    b = torch.randn(128, generator=g)
    alpha = torch.randn(4, 192, generator=g)
    h, S = ops.proj_fwd(x.cuda(), W.cuda(), b.cuda(), alpha.cuda(), 192, 0, 160, precision=ops.PRECISION_TF32X3)
    torch.cuda.synchronize()
    href = F.linear(x.double(), W.double(), b.double())
    assert rel_err(h, href) <= X3_TOL
    hv = href.view(n, 4, 32)
    ad = alpha.double()
    Sref = torch.cat([(hv * ad[:, 0:32]).sum(-1), (hv * ad[:, 160:192]).sum(-1)], dim=1)
    assert rel_err(S, Sref) <= X3_TOL
    # row-wise: every row within 1e-5 of its own scale (the per-tensor metric hides small rows behind large ones)
    row = (h.cpu().double() - href).abs().amax(1) / href.abs().amax(1).clamp_min(1e-30)
    assert float(row.max()) <= 1e-5
    # S without alpha, bias-free, integer operands: exact
    xi = torch.randint(-4, 5, (n, K), generator=g).float()
    Wi = torch.randint(-4, 5, (128, K), generator=g).float()
    hi, _ = ops.proj_fwd(xi.cuda(), Wi.cuda(), None, None, want_S=False, precision=ops.PRECISION_TF32X3)
    assert torch.equal(hi.cpu(), xi @ Wi.t())


def test_x3_projection_backward_is_fp32_grade():
    from fragnet_b200 import ops
    g = torch.Generator().manual_seed(33)
    n = 54001
    x = torch.randn(n, 128, generator=g)
    W = torch.randn(128, 128, generator=g) * 0.2
    dh = torch.randn(n, 128, generator=g) * torch.exp(torch.randn(n, 1, generator=g))
    for n2 in (1, 31, 33, 511, 513, 4800, 54001):
        xs, ds = x[:n2].contiguous(), dh[:n2].contiguous()
        dx, dW, _ = ops.proj_bwd(xs.cuda(), W.cuda(), ds.cuda(), True, ops.PRECISION_TF32X3, want_db=False)
        assert rel_err(dx, ds.double() @ W.double()) <= X3_TOL, n2
        assert rel_err(dW, ds.double().t() @ xs.double()) <= X3_TOL, n2
    x2 = torch.randn(3000, 256, generator=g)          # the energy head's 256-wide operand
    d2 = torch.randn(3000, 128, generator=g)
    W2 = torch.randn(128, 256, generator=g)
    _, dW2, _ = ops.proj_bwd(x2.cuda(), W2.cuda(), d2.cuda(), False, ops.PRECISION_TF32X3, want_db=False)
    assert rel_err(dW2, d2.double().t() @ x2.double()) <= X3_TOL


@pytest.mark.parametrize("n,K", [(1, 128), (127, 128), (128, 128), (129, 128), (1000, 128), (54001, 128),
                                 (300, 32), (300, 64), (300, 256), (40000, 128)])
def test_tc_projection_forward(n, K):
    from fragnet_b200 import ops
    g = torch.Generator().manual_seed(n + K)
    x = torch.randn(n, K, generator=g)
    W = torch.randn(128, K, generator=g) * 0.2
    b = torch.randn(128, generator=g)
    alpha = torch.randn(4, 192, generator=g)
    h, S = ops.proj_fwd(x.cuda(), W.cuda(), b.cuda(), alpha.cuda(), 192, 0, 160, precision=ops.PRECISION_TF32)
    torch.cuda.synchronize()
    href = F.linear(x, W, b)
    assert rel_err(h, href) <= TF32_TOL
    hv = href.view(n, 4, 32)
    Sref = torch.cat([(hv * alpha[:, 0:32]).sum(-1), (hv * alpha[:, 160:192]).sum(-1)], dim=1)
    assert rel_err(S, Sref) <= TF32_TOL
    # exactness of the data path: integer-valued operands are exact in TF32
    xi = torch.randint(-4, 5, (n, K), generator=g).float()
    Wi = torch.randint(-4, 5, (128, K), generator=g).float()
    hi, _ = ops.proj_fwd(xi.cuda(), Wi.cuda(), None, None, want_S=False, precision=ops.PRECISION_TF32)
    assert torch.equal(hi.cpu(), xi @ Wi.t())


def test_tc_projection_backward_dx():
    from fragnet_b200 import ops
    g = torch.Generator().manual_seed(3)
    n = 5000
    x = torch.randn(n, 128, generator=g)
    W = torch.randn(128, 128, generator=g) * 0.2
    dh = torch.randn(n, 128, generator=g)
    dx, dW, db = ops.proj_bwd(x.cuda(), W.cuda(), dh.cuda(), True, ops.PRECISION_TF32)
    assert rel_err(dx, dh @ W) <= TF32_TOL
    assert rel_err(dW, dh.t() @ x) <= TF32_TOL
    assert rel_err(db, dh.sum(0)) <= 1e-5
    for n2 in (1, 31, 32, 33, 4800, 54001):       # tensor-core weight gradient (no db): ragged row counts
        _, dW2, _ = ops.proj_bwd(x[:n2].cuda().contiguous(), W.cuda(), dh[:n2].cuda().contiguous(), False,
                                 ops.PRECISION_TF32, want_db=False) if n2 <= n else (None, None, None)
        if n2 <= n:
            assert rel_err(dW2, dh[:n2].t() @ x[:n2]) <= TF32_TOL, n2
    xi = torch.randint(-3, 4, (777, 128), generator=g).float()
    di = torch.randint(-3, 4, (777, 128), generator=g).float()
    _, dWi, _ = ops.proj_bwd(xi.cuda(), W.cuda(), di.cuda(), False, ops.PRECISION_TF32, want_db=False)
    assert torch.equal(dWi.cpu(), di.t() @ xi)


def test_unaligned_k_falls_back_to_fp32_kernel():
    from fragnet_b200 import ops
    g = torch.Generator().manual_seed(4)
    x = torch.randn(300, 167, generator=g)
    W = torch.randn(128, 167, generator=g) * 0.2
    h, _ = ops.proj_fwd(x.cuda(), W.cuda(), None, None, want_S=False, precision=ops.PRECISION_TF32)
    assert rel_err(h, x @ W.t()) <= 1e-5


def test_model_in_tf32_mode_within_stated_tolerance():
    from fragnet.model.gat.gat2 import FragNetFineTune
    from fragnet_b200 import config, synth
    from fragnet_b200.dataset.data import collate_fn
    from oracle import gat2_oracle as O
    b = collate_fn(synth.make_dataset("unimol", 48, seed=6))
    torch.manual_seed(5)
    m = FragNetFineTune(num_layer=4, drop_ratio=0.0, h1=128, h2=256, h3=256, h4=128, act="relu").eval()
    P = O.params_from_module(m)
    m = m.cuda()
    config.set_precision("tf32")
    try:
        pred = m({k: v.cuda() for k, v in b.items()})
        pred.sum().backward()
    finally:
        config.set_precision("fp32")
    ref = O.finetune_forward(P, b)
    ref.sum().backward()
    assert rel_err(pred, ref) <= 5e-3
    g = dict(m.named_parameters())["pretrain.layers.1.projection_b.weight"].grad
    assert rel_err(g, P["pretrain.layers.1.projection_b.weight"].grad) <= 2e-2
    # every gradient, including the layer-0 weight gradients that come from the zero-padded tensor-core path
    from conftest import grad_errs
    named = dict(m.named_parameters())
    errs = grad_errs([(k, named[k].grad, P[k].grad) for k in named if P[k].grad is not None])
    assert all(k in errs for k in ("pretrain.layers.0.projection_a.weight", "pretrain.layers.0.projection_b.weight",
                                   "pretrain.layers.0.projection_fb.weight"))
    bad = {k: v for k, v in errs.items() if v > 2e-2}
    assert not bad, bad
    for k in named:
        assert (named[k].grad is None) == (P[k].grad is None), k


def test_tc_projection_speed_report(capsys):
    from fragnet_b200 import ops
    n = 54000
    x = torch.randn(n, 128, device="cuda")
    W = torch.randn(128, 128, device="cuda")
    b = torch.randn(128, device="cuda")
    a = torch.randn(4, 96, device="cuda")
    out = {}
    for name, prec in (("fp32", 0), ("tf32", 1), ("x3", 2)):
        for _ in range(3):
            ops.proj_fwd(x, W, b, a, 96, 0, 64, precision=prec)
        e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
        e0.record()
        for _ in range(20):
            ops.proj_fwd(x, W, b, a, 96, 0, 64, precision=prec)
        e1.record()
        e1.synchronize()
        out[name] = e0.elapsed_time(e1) / 20 * 1e3
    with capsys.disabled():
        gb = n * 1024 / 1e9
        print(f"\n[proj_fwd 54000x128x128] fp32 FFMA {out['fp32']:.1f} us, tf32 {out['tf32']:.1f} us, 3xTF32 {out['x3']:.1f} us "
              f"({gb / (out['x3'] * 1e-6):.0f} GB/s algorithmic, L2-warm)")
