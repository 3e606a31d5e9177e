"""Dropout-mode training against the float64 oracle with the library's dropout masks replayed on the host.

The library never stores a dropout mask: every site regenerates its keep-bits from ``(seed, counter)`` with the integer
hash of csrc/common.cuh, and the counters of one call follow a fixed layout.  This file restates the hash, the threshold
and the layout independently in numpy, hands the resulting masks to the oracle through its ``drop_fn`` hook, and checks
the training-mode outputs and gradients of every dropout path (input dropout through the standalone kernel and through
the padding kernel, the fused post-activation epilogues, the backward folds of ``dy (y > 0) / (1 - p)``, the lite and
edge variants' standalone calls, the one-call pretraining step) against it, at the tolerances of record.  With
``p = 0`` every mask is all-ones and every scale 1, so the drop-free parity tests cannot see a wrong scale, a shifted
counter base or a mask indexed differently in two places; these can."""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import FP32_REL_TOL, grad_errs, rel_err

pytestmark = pytest.mark.gpu
GRAD_TOL = 5e-5
U32 = np.uint32
M64 = (1 << 64) - 1


# ---- host replica of the masks (common.cuh: mix32, dropout_bits, dropout_threshold) ---------------------------------
def _mix32(x):
    x = x ^ (x >> U32(17))
    x = x * U32(0xED5AD4BB)
    x = x ^ (x >> U32(11))
    x = x * U32(0xAC4C1B51)
    x = x ^ (x >> U32(15))
    x = x * U32(0x31848BAB)
    return x ^ (x >> U32(14))


def _bits(seed: int, counters: np.ndarray):
    """The two 32-bit words of every counter (``dropout_bits``): 64-bit seed and counter split into lo / hi words."""
    lo = (counters & np.uint64(0xFFFFFFFF)).astype(U32)
    hi = (counters >> np.uint64(32)).astype(U32)
    k0, k1 = U32(seed & 0xFFFFFFFF), U32((seed >> 32) & 0xFFFFFFFF)
    a = _mix32(lo ^ k0) ^ (hi * U32(0x9E3779B1))
    return _mix32(a + k1), _mix32(a ^ U32(0x85EBCA6B) ^ k1)


def threshold(p: float) -> int:
    """``(uint32)(p * 65536.0f + 0.5f)``, in float32 as on the device."""
    return int(np.float32(p) * np.float32(65536.0) + np.float32(0.5))


def scale32(p: float) -> np.float32:
    return np.float32(1.0) / (np.float32(1.0) - np.float32(p))


def keep_mask(seed: int, offset: int, n: int, p: float) -> np.ndarray:
    """bool[n]: element i draws from counter ``offset + i // 4``; positions 0 / 1 take the low / high half of the first
    word, positions 2 / 3 those of the second."""
    groups = (n + 3) // 4
    counters = np.uint64(offset) + np.arange(groups, dtype=np.uint64)
    x, y = _bits(seed, counters)
    r16 = np.stack((x & U32(0xFFFF), x >> U32(16), y & U32(0xFFFF), y >> U32(16)), axis=1).reshape(-1)[:n]
    return r16 >= U32(threshold(p))


def counters_of(n: int) -> int:
    return (n + 3) // 4


def roundup4(n: int) -> int:
    return (n + 3) // 4 * 4


def encoder_sites(offset, n_layers, na, k_atom, nb, nfb, nf):
    """Counter bases of one encoder call: the input site over ``na * k_atom`` elements, then per layer bond, atom,
    fragment-connection and fragment sites over 128-wide rows.  Returns ({site: base}, total counters)."""
    c = offset
    bases = {("input", "atoms"): c}
    c += counters_of(na * k_atom)
    for l in range(n_layers):
        for name, rows in (("bond", nb), ("atoms", na), ("fbond", nfb), ("frags", nf)):
            bases[(l, name)] = c
            c += counters_of(rows * 128)
    return bases, c - offset


def replay(bases, seed, p, shift=0, scale=None):
    """``drop_fn`` for the oracle: multiplies by ``keep * 1/(1-p)`` in the tensor's dtype.  Sites without a base
    (whose values nobody reads) keep everything.  ``shift`` / ``scale`` deliberately break the replay (self-check)."""
    s = 1.0 / (1.0 - p) if scale is None else scale

    def fn(site, t):
        if site not in bases:
            return t
        keep = torch.from_numpy(keep_mask(seed, bases[site] + shift, t.numel(), p)).view(t.shape)
        return t * (keep.to(t.dtype) * s)
    return fn


def _gen():
    return torch.cuda.default_generators[torch.cuda.current_device()]


def _seed():
    return torch.initial_seed() & M64


# Counter base of the calls under test.  torch.manual_seed resets the offset to 0; a base far from 0 (whose sites cross
# 2**32) and a seed with a non-zero high word make every comparison fail if the library drew from counter 0, dropped the
# high word of a counter or of the seed, or ignored the base the host reserved.
START = 2 ** 32 - 64


def _start_stream(k: int):
    """Seeds the dropout stream with a 64-bit seed and moves its counter to ``START``; returns (seed, first counter)."""
    torch.manual_seed(2 ** 40 + k)
    _gen().set_offset(START)
    return _seed(), _gen().get_offset()


# ---- shared fixtures ---------------------------------------------------------------------------------------------------
def _host_batch(n_esol, n_unimol, seed, handmade=("ion_pair", "two_atom", "two_frag", "single_frag")):
    from fragnet_b200 import synth
    from fragnet_b200.dataset.data import collate_fn_pt
    mols = synth.make_dataset("esol", n_esol, seed=seed) if n_esol else []
    mols += synth.make_dataset("unimol", n_unimol, seed=seed + 1) if n_unimol else []
    mols += [synth.handmade(k) for k in handmade]
    b = collate_fn_pt(mols)
    gen = torch.Generator().manual_seed(seed + 2)
    for k in ("bnd_angl", "dh_angl"):
        b[k] = torch.randn(b[k].shape, generator=gen)
    b["y"] = torch.randn(b["y"].shape, generator=gen)
    return b


def _f64(batch):
    return {k: v.double() if v.is_floating_point() else v for k, v in batch.items()}


def _cuda(batch):
    return {k: v.cuda() for k, v in batch.items()}


def _params64(module):
    """float64 leaf copies of a module's (or a state dict's) tensors."""
    out = {}
    for k, v in (module.state_dict() if hasattr(module, "state_dict") else module).items():
        t = v.detach().to("cpu", torch.float64).clone()
        out[k] = t.requires_grad_() if t.is_floating_point() else t
    return out


def _sizes(b):
    return (b["x_atoms"].shape[0], b["x_atoms"].shape[1], b["edge_index"].shape[1], b["frag_index"].shape[1],
            b["x_frags"].shape[0])


def _last_only(bases, n_layers, names=("frags",)):
    """The fragment output of a non-final layer is overwritten unread (gat2.py:234): no mask to replay."""
    return {s: v for s, v in bases.items() if not (s[0] != "input" and s[1] in names and s[0] != n_layers - 1)}


def _check_forward(got, want, names):
    errs = {n: rel_err(a, w) for n, a, w in zip(names, got, want)}
    bad = {n: e for n, e in errs.items() if e > FP32_REL_TOL}
    assert not bad, bad
    return errs


def _check_grads(pairs, tol=GRAD_TOL):
    errs = grad_errs(pairs)
    bad = {k: v for k, v in errs.items() if v > tol}
    assert not bad, bad
    return errs


def _param_pairs(named, P):
    named = dict(named)
    for k, p in named.items():
        assert (p.grad is None) == (P[k].grad is None), k
    return [(k, p.grad, P[k].grad) for k, p in named.items() if p.grad is not None]


# ---- 1. the replica is the kernel's mask, bit for bit --------------------------------------------------------------
@pytest.mark.parametrize("p", [0.1, 0.2, 0.5, 0.9])
def test_host_replica_equals_the_dropout_kernel_bitwise(p):
    from fragnet_b200 import ops
    s = scale32(p)
    crossed = False
    for n in (1, 3, 4, 5, 1001, 167 * 37, 128 * 4099):
        buf = torch.ones(n + 1, device="cuda")
        for view in (buf[:n], buf[1:]):           # buf[1:] is not 16-byte aligned: the scalar path of the kernel
            for seed in (0, 77, 2 ** 40 + 7, 2 ** 64 - 1):
                for offset in (0, 4, 2 ** 32 - 3, 2 ** 40):
                    y = ops.dropout_relu_fwd(view, p, True, False, seed, offset).cpu().numpy()
                    want = np.where(keep_mask(seed, offset, n, p), s, np.float32(0.0)).astype(np.float32)
                    assert np.array_equal(y, want), (n, view.data_ptr() % 16, seed, offset)
                    crossed |= offset < 2 ** 32 <= offset + (n - 1) // 4
    assert crossed          # some call's counters ran from below 2**32 to above it: the high counter word took part


@pytest.mark.parametrize("p", [0.2, 0.5])
def test_host_replica_equals_the_fused_attention_epilogue(p):
    """``y`` of the tiled attention forward with ``post`` = ReLU(Dropout) is relu(out * keep * scale), element
    (t, c) drawing from counter offset + (t * 128 + c) // 4."""
    from fragnet_b200 import ops
    n_nodes, n_edges = 777, 5000
    gen = torch.Generator().manual_seed(1)
    dst = torch.randint(0, n_nodes, (n_edges,), generator=gen)
    dst[:n_nodes] = torch.arange(n_nodes)
    src = torch.randint(0, n_nodes, (n_edges,), generator=gen)
    h = torch.randn(n_nodes, 128, generator=gen).cuda()
    alpha = torch.randn(4, 96, generator=gen).cuda()
    graph = ops.csr_build(dst.cuda(), src.cuda(), n_nodes)
    S = ops.node_scalars(h, alpha, 96, 0, 64)
    for seed, offset in ((1234567, 999), (2 ** 64 - 1, 2 ** 32 - 100)):
        out, y, _, _ = ops.gat_fwd_tiled(graph, h, S, ops.EDGE_NONE, save_p=False, post=(p, 1, 1, seed, offset))
        keep = torch.from_numpy(keep_mask(seed, offset, out.numel(), p)).view(out.shape)
        o = out.cpu()
        want = torch.where(keep, o * torch.tensor(float(scale32(p))), o * 0.0).clamp_min(0.0)
        assert torch.equal(y.cpu(), want), (seed, offset)


# ---- 2. the encoder in training mode --------------------------------------------------------------------------------
def _encoder_case(drop, num_layer, want_dx, seed=3):
    """FragNet (through FragNetPreTrain.pretrain) in training mode with random cotangents on its four outputs; with
    ``want_dx`` the three layer-0 inputs require grad.  Returns what the oracle needs to replay the call and the GPU
    results."""
    from fragnet.model.gat.gat2_pretrain import FragNetPreTrain
    hb = _host_batch(10, 14, 40 + seed)
    torch.manual_seed(100 + seed)
    m = FragNetPreTrain(num_layer=num_layer, drop_ratio=drop, edge_features=17).cuda().train()
    gen = torch.Generator().manual_seed(seed)
    b = _cuda(hb)
    ins = ("x_atoms", "node_features_bonds", "node_features_fbonds")
    if want_dx:
        for k in ins:
            b[k] = b[k].clone().requires_grad_()
    seed_v, off0 = _start_stream(7 + seed)         # the dropout stream: torch's seed, torch's CUDA generator offset
    outs = m.pretrain(b)
    off1 = _gen().get_offset()
    cots = [torch.randn(o.shape, generator=gen) for o in outs]
    sum((o * w.cuda()).sum() for o, w in zip(outs, cots)).backward()
    got = {"outs": [o.detach().cpu() for o in outs], "params": list(m.named_parameters()),
           "inputs": {k: b[k].grad.cpu() for k in ins} if want_dx else None}
    return m, hb, cots, seed_v, off0, off1, got


def _oracle_encoder(m, hb, cots, bases, seed_v, drop, num_layer, want_dx, **kw):
    from oracle import gat2_oracle as O
    P = _params64(m)
    b = _f64(hb)
    ins = ("x_atoms", "node_features_bonds", "node_features_fbonds")
    if want_dx:
        for k in ins:
            b[k] = b[k].clone().requires_grad_()
    outs = O.fragnet_forward(P, b, num_layer, drop_ratio=drop, training=True,
                             drop_fn=replay(bases, seed_v, drop, **kw))
    sum((o * w.double()).sum() for o, w in zip(outs, cots)).backward()
    return outs, P, ({k: b[k].grad for k in ins} if want_dx else None)


ENC_NAMES = ("x_atoms", "x_frags", "bond", "fbond")


ROUTES = {
    "pad_kernel_input_dropout": False,            # no input gradients: input dropout inside the layer-0 padding kernel
    "standalone_input_dropout": True,             # d x_atoms wanted: the standalone kernel, its mask re-applied to dx
    "pad_forward_dx_backward": True,              # a C caller that sets need_dx_* for the backward call only
}


@pytest.mark.parametrize("route", list(ROUTES))
@pytest.mark.parametrize("num_layer", [1, 4])
@pytest.mark.parametrize("drop", [0.2, 0.5])
def test_encoder_training_mode_matches_oracle_with_replayed_masks(drop, num_layer, route, monkeypatch):
    want_dx = ROUTES[route]
    if route == "pad_forward_dx_backward":
        # the forward call then takes the padding-kernel route and keeps no unpadded dropped copy of x_atoms; the
        # backward must still form the layer-0 weight gradient from what the forward multiplied
        from fragnet_b200 import _abi
        real = _abi.CEncoderOpts
        monkeypatch.setattr(_abi, "CEncoderOpts", lambda *a: real(*a[:8], 0, 0, 0))
    m, hb, cots, seed_v, off0, off1, got = _encoder_case(drop, num_layer, want_dx)
    bases, span = encoder_sites(off0, num_layer, *_sizes(hb))
    assert off1 - off0 == roundup4(span)
    outs, P, din = _oracle_encoder(m, hb, cots, _last_only(bases, num_layer), seed_v, drop, num_layer, want_dx)
    _check_forward(got["outs"], outs, ENC_NAMES)
    _check_grads(_param_pairs(got["params"], P))
    if want_dx:
        _check_grads([(k, got["inputs"][k], din[k]) for k in din])


# ---- 3. a pretraining step through autograd ---------------------------------------------------------------------------
def _pretrain_model(num_layer, drop, seed):
    from fragnet.model.gat.gat2_pretrain import FragNetPreTrain
    torch.manual_seed(seed)
    return FragNetPreTrain(num_layer=num_layer, drop_ratio=drop, edge_features=17).cuda().train()


def _oracle_pretrain(m, hb, bases, seed_v, drop, num_layer):
    from oracle import gat2_oracle as O
    P = _params64(m)
    b = _f64(hb)
    preds = O.pretrain_forward(P, b, num_layer, drop_ratio=drop, training=True,
                               drop_fn=replay(_last_only(bases, num_layer), seed_v, drop))
    loss = O.pretrain_loss(preds, b)
    loss.backward()
    return preds, loss, P


def test_pretrain_step_on_the_autograd_path_matches_oracle():
    from fragnet_b200.train.pretrain_utils import pretrain_loss
    hb = _host_batch(12, 20, 60)
    m = _pretrain_model(4, 0.2, 61)
    b = _cuda(hb)
    seed_v, off0 = _start_stream(62)
    preds = m(b)
    loss = pretrain_loss(torch.nn.MSELoss(), preds, b)
    loss.backward()
    bases, span = encoder_sites(off0, 4, *_sizes(hb))
    assert _gen().get_offset() - off0 == roundup4(span)
    ref_preds, ref_loss, P = _oracle_pretrain(m, hb, bases, seed_v, 0.2, 4)
    _check_forward(preds, ref_preds, ("bond_length", "bond_angle", "dihedral", "energy"))
    assert rel_err(loss, ref_loss) <= FP32_REL_TOL
    _check_grads(_param_pairs(m.named_parameters(), P))


# ---- 4. the one-call step -------------------------------------------------------------------------------------------
def _check_fused_against_oracle(m, hb, loss, seed_v, off0, num_layer, drop, state=None):
    """Loss and gradients (``p.grad`` of ``m``) of one step against the oracle at parameters ``state`` (default: the
    model's current ones) with the masks of the counter block starting at ``off0``."""
    bases, _ = encoder_sites(off0, num_layer, *_sizes(hb))
    _, ref_loss, P = _oracle_pretrain(m if state is None else state, hb, bases, seed_v, drop, num_layer)
    assert rel_err(loss, ref_loss) <= FP32_REL_TOL
    _check_grads(_param_pairs(m.named_parameters(), P))


def _step_rng_span(hb, num_layer, drop):
    """``fnb_pretrain_step_rng_span`` of a batch: the span depends on the batch sizes, the layer-0 atom width and the
    layer count only, so the arguments carry nothing else."""
    from fragnet_b200 import _abi, ops
    na, k_atom, nb, nfb, nf = _sizes(hb)
    a = _abi.CPretrainStepArgs()
    a.batch = _abi.CBatchInputs(*([None] * 9), na, nf, nb, hb["edge_index_bonds_graph"].shape[1], nfb,
                                hb["edge_index_fbonds"].shape[1], hb["y"].numel())
    layers = (_abi.CLayerParams * num_layer)()
    for l in range(num_layer):
        layers[l].K_atom, layers[l].K_bond, layers[l].K_fbond = (
            (k_atom, hb["node_features_bonds"].shape[1], hb["node_features_fbonds"].shape[1]) if l == 0 else (128,) * 3)
    heads = _abi.CPretrainHeadParams()
    a.n_layers, a.layers, a.heads = num_layer, C.cast(layers, C.c_void_p), C.cast(C.pointer(heads), C.c_void_p)
    a.drop_p, a.training = drop, 1
    return ops._lib().fnb_pretrain_step_rng_span(C.byref(a))


def test_fused_pretrain_step_matches_oracle_and_reserves_its_counters():
    from fragnet_b200.train.fused import FusedPretrainStep
    hb = _host_batch(12, 20, 70)
    m = _pretrain_model(4, 0.2, 71)
    fused = FusedPretrainStep(m, lr=1e-3)
    b = _cuda(hb)
    seed_v, off0 = _start_stream(72)
    loss = fused.forward_backward(b)
    off1 = _gen().get_offset()
    _check_fused_against_oracle(m, hb, loss, seed_v, off0, 4, 0.2)
    _, span = encoder_sites(off0, 4, *_sizes(hb))
    assert _step_rng_span(hb, 4, 0.2) == span
    assert off1 - off0 == roundup4(span)
    # consecutive training steps take consecutive, disjoint counter blocks, and the kernels draw from the block the
    # host reserved: the second step's loss and gradients (taken before its Adam update) are the oracle's at the
    # parameters the first step left, with the masks of the second block
    fused.step(b)
    mid = _gen().get_offset()
    assert mid - off1 == roundup4(span)
    state = {k: v.detach().clone() for k, v in m.state_dict().items()}
    loss2 = fused.step(b)
    after = _gen().get_offset()
    assert after - mid == roundup4(span)
    _check_fused_against_oracle(m, hb, loss2, seed_v, mid, 4, 0.2, state=state)
    # evaluation (eval mode: no dropout) draws no counters
    m.eval()
    fused.evaluate(b)
    torch.cuda.synchronize()
    assert _gen().get_offset() == after
    m.train()


# ---- 5. gat2_lite and gat2_edge ---------------------------------------------------------------------------------------
def _lite_edge_case(variant, num_layer, drop=0.2, seed=80):
    from fragnet_b200.model.gat import gat2_edge, gat2_lite
    from oracle import gat2_oracle as O
    hb = _host_batch(8, 10, seed)
    if variant == "edge":        # gat2_edge's connection attributes are 8 wide: two columns the 6-wide featuriser lacks
        extra = torch.rand(hb["cnx_attr"].shape[0], 2, generator=torch.Generator().manual_seed(seed))
        hb["cnx_attr"] = torch.cat((hb["cnx_attr"], extra), dim=1)
    mod = gat2_lite if variant == "lite" else gat2_edge
    torch.manual_seed(seed + 1)
    m = mod.FragNet(num_layer, drop_ratio=drop, edge_features=17).cuda().train()
    b = _cuda(hb)
    seed_v, off0 = _start_stream(seed + 2)
    outs = m(b)[:3]
    off1 = _gen().get_offset()
    gen = torch.Generator().manual_seed(seed + 3)
    cots = [torch.randn(o.shape, generator=gen) for o in outs]
    sum((o * w.cuda()).sum() for o, w in zip(outs, cots)).backward()
    na, k_atom, nb, nfb, nf = _sizes(hb)
    if variant == "edge":
        # one encoder call; the fragment-connection graph keeps its nodes (zero features), so its sites are reserved
        bases, span = encoder_sites(off0, num_layer, na, k_atom, nb, nfb, nf)
        assert off1 - off0 == roundup4(span)
        bases = _last_only(bases, num_layer)
        fwd = O.edge_fragnet_forward
    else:
        # every layer but the last in one encoder call (no fragment-connection graph); then ReLU(Dropout) of the last
        # layer's atoms, pooled fragments and bonds, each a call of its own that takes the next counters
        c = off0
        if num_layer > 1:
            bases, span = encoder_sites(c, num_layer - 1, na, k_atom, nb, 0, nf)
            c += roundup4(span)
        else:
            bases = {("input", "atoms"): c}
            c += roundup4(counters_of(na * k_atom))
        last = num_layer - 1
        for name, rows in (("atoms", na), ("frags", nf), ("bond", nb)):
            bases[(last, name)] = c
            c += roundup4(counters_of(rows * 128))
        assert off1 == c
        bases = _last_only(bases, num_layer)
        fwd = O.lite_fragnet_forward
    P = _params64(m)
    ref = fwd(P, _f64(hb), num_layer, drop_ratio=drop, training=True, prefix="",
              drop_fn=replay(bases, seed_v, drop))[:3]
    sum((o * w.double()).sum() for o, w in zip(ref, cots)).backward()
    _check_forward(outs, ref, ENC_NAMES[:3])
    _check_grads(_param_pairs(m.named_parameters(), P))


@pytest.mark.parametrize("variant,num_layer", [("lite", 1), ("lite", 3), ("edge", 3)])
def test_lite_and_edge_encoders_match_oracle_with_replayed_masks(variant, num_layer):
    _lite_edge_case(variant, num_layer)


# ---- 6. the benchmark's headline step -----------------------------------------------------------------------------------
def _away_from_relu_kinks(m, hb, bases, seed_v, drop, num_layer, margin=2e-6, rounds=30):
    """Perturbs the input features of every molecule that has a kept ReLU pre-activation (encoder sites and the
    heads' hidden layers) within ``margin`` x the site's largest magnitude of zero, until none has.

    ReLU's derivative is discontinuous at 0 (see ``test_gpu_heads._away_from_relu_kinks``): at the bench batch the
    encoder has ~2.5e7 ReLU inputs, a few dozen of them within 1e-6 relative of zero, and two correct fp32 evaluations
    flip one of those (even the fp32 oracle against the float64 one: a rank-one gap of 9e-5 in one layer's
    projection_b gradient).  Only feature values change -- rows keep their positions -- so the dropout masks stay
    those of the counters the step will draw."""
    from oracle import gat2_oracle as O
    P = {k: v.detach().to("cpu", torch.float64) for k, v in m.state_dict().items()}
    hb = dict(hb)
    owners = {"atoms": hb["batch"], "frags": hb["frag_batch"], "bond": hb["batch"][hb["edge_index"][0]],
              "fbond": hb["frag_batch"][hb["frag_index"][0]]}
    rep = replay(_last_only(bases, num_layer), seed_v, drop)
    gen = torch.Generator().manual_seed(0)
    for _ in range(rounds):
        close = torch.zeros(hb["y"].numel(), dtype=torch.bool)

        def mark(owner, pre):
            a = pre.abs()
            near = ((a < margin * a.max()) & (a != 0)).any(1)
            close[owner[near]] = True

        def fn(site, t):
            y = rep(site, t)
            if site[0] != "input" and (site[1] != "frags" or site[0] == num_layer - 1):
                mark(owners[site[1]], y)
            return y
        with torch.no_grad():
            x_atoms, x_frags, edge, _ = O.fragnet_forward(P, _f64(hb), num_layer, drop_ratio=drop, training=True,
                                                          drop_fn=fn)
            for stack, x, owner in (("ba_layers", x_atoms, owners["atoms"]), ("da_layers", edge, owners["bond"]),
                                    ("FC_layers", O.readout(x_atoms, x_frags, hb), torch.arange(close.numel()))):
                for l in range(2):
                    x = O._linear(P, f"head.{stack}.{l}", x)
                    mark(owner, x)
                    x = x.clamp_min(0)
        if not bool(close.any()):
            return hb
        for key, owner in (("x_atoms", owners["atoms"]), ("node_features_bonds", owners["bond"]),
                           ("node_features_fbonds", owners["fbond"])):
            rows = close[owner]
            x = hb[key].clone()
            x[rows] *= 1 + 0.1 * (torch.rand(x[rows].shape, generator=gen) - 0.5)
            hb[key] = x
    raise AssertionError("could not condition the batch away from the ReLU kinks")


def test_bench_configuration_fused_step_matches_oracle():
    """One FusedPretrainStep.forward_backward at bench.py's headline configuration: 1 024 unimol molecules, four
    layers, drop 0.2, against the float64 oracle."""
    from fragnet_b200.train.fused import FusedPretrainStep
    hb = _host_batch(0, 1024, 90, handmade=())
    m = _pretrain_model(4, 0.2, 91)
    fused = FusedPretrainStep(m, lr=1e-3)
    seed_v, off0 = _start_stream(92)
    bases, span = encoder_sites(off0, 4, *_sizes(hb))
    hb = _away_from_relu_kinks(m, hb, bases, seed_v, 0.2, 4)       # host-side only: the generator does not move
    loss = fused.forward_backward(_cuda(hb))
    assert _gen().get_offset() - off0 == roundup4(span)
    _check_fused_against_oracle(m, hb, loss, seed_v, off0, 4, 0.2)


# ---- 7. the harness rejects a wrong counter base and a wrong scale -------------------------------------------------------
def test_replay_with_shifted_counters_or_missing_scale_fails_by_far():
    """The comparison above would catch an off-by-one counter base or a scale applied zero times: the same GPU run
    against an oracle with every base moved by one counter, or with the right masks but scale 1, misses the
    tolerances by at least 100x."""
    drop, num_layer = 0.2, 4
    m, hb, cots, seed_v, off0, _, got = _encoder_case(drop, num_layer, True)
    bases = _last_only(encoder_sites(off0, num_layer, *_sizes(hb))[0], num_layer)
    params = list(got["params"])
    for kw in ({"shift": 1}, {"scale": 1.0}):
        outs, P, din = _oracle_encoder(m, hb, cots, bases, seed_v, drop, num_layer, True, **kw)
        fwd = max(rel_err(a, w) for a, w in zip(got["outs"], outs))
        grads = max(grad_errs(_param_pairs(params, P)).values())
        dx = max(grad_errs([(k, got["inputs"][k], din[k]) for k in din]).values())
        assert fwd >= 100 * FP32_REL_TOL and grads >= 100 * GRAD_TOL and dx >= 100 * GRAD_TOL, (kw, fwd, grads, dx)
