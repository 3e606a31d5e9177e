"""``torch.autograd.Function`` wrappers over the library's encoder programs.

One Function for the WHOLE encoder (all layers of ``FragNet.forward``, reference fragnet/model/gat/gat2.py:381-442,
or one bare ``FragNetLayerA.forward``, gat2.py:121-330) rather than one per op or per layer: the forward is a single
``fnb_encoder_forward`` call and the backward a single ``fnb_encoder_backward`` call (encoder.cu sequences every
launch in C++), so a training step crosses the Python boundary twice for the message passing instead of ~190 times,
and autograd keeps exactly one workspace tensor alive for the backward.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import List, Optional

import torch

from . import _abi, ops
from .ops import LayerPlan

N_PARAMS = len(_abi.PARAM_FIELDS)     # live tensors per layer, in ``FragNetLayerA._live_parameters`` order
_F_INDEX = _abi.PARAM_FIELDS.index("f")


@dataclass
class LayerSwitches:
    """Per-layer switches that are not tensors (mirrors the non-pointer tail of ``fnb_layer_params``)."""
    run_frag_block: bool = True
    want_attention: bool = False
    bond_mask: object = None            # int m (rows m, m+1: gat2.py:173-176), or a sequence / tensor of such m
    frag_bond_mask: object = None       # int k (rows 2k, 2k+1: gat2.py:275-278), or a sequence / tensor of such k
    atom_mask: object = None            # int, or a sequence / tensor of atom rows (gat2.py:227-231)


@dataclass
class EncoderConfig:
    layers: List[LayerSwitches]
    post_act: bool                      # True: FragNet.forward (ReLU(Dropout) everywhere); False: one bare layer
    drop_p: float = 0.0
    training: bool = False
    precision: int = 0
    grad_enabled: bool = True           # torch.is_grad_enabled() at the call site (it is always off inside forward)
    frag_table: bool = False            # gat2_edge: the LAST tensor passed to EncoderFn is the fragment graph's edge
                                        # term [Ef,4] (edge-id order), used instead of the fragment-connection block's
    _keep: list = field(default_factory=list, repr=False)   # tensors the C structs point into


def _has_mask(cfg: EncoderConfig) -> bool:
    return any(s.bond_mask is not None or s.frag_bond_mask is not None or s.atom_mask is not None for s in cfg.layers)


def _layer_structs(cfg: EncoderConfig, params, dev):
    n = len(cfg.layers)
    arr = (_abi.CLayerParams * n)()
    for l, sw in enumerate(cfg.layers):
        ps = params[l * N_PARAMS:(l + 1) * N_PARAMS]
        for name, t in zip(_abi.PARAM_FIELDS, ps):
            setattr(arr[l], name, t.data_ptr())
        arr[l].K_bond, arr[l].K_fbond, arr[l].K_atom = ps[0].shape[1], ps[2].shape[1], ps[8].shape[1]
        arr[l].run_frag_block, arr[l].want_attention = int(sw.run_frag_block), int(sw.want_attention)
        arr[l].bond_mask, arr[l].frag_bond_mask = -1, -1
        arr[l].bond_mask_rows, arr[l].n_bond_mask_rows, arr[l].fbond_mask_rows, arr[l].n_fbond_mask_rows = None, 0, None, 0
        for value, scale, single, rows_f, n_f in ((sw.bond_mask, 1, "bond_mask", "bond_mask_rows", "n_bond_mask_rows"),
                                                  (sw.frag_bond_mask, 2, "frag_bond_mask", "fbond_mask_rows",
                                                   "n_fbond_mask_rows")):
            if value is None:
                continue
            if isinstance(value, int):
                setattr(arr[l], single, value)
                continue
            first = torch.as_tensor(value, device=dev).reshape(-1).to(torch.int64) * scale     # first row of each pair
            rows = torch.stack((first, first + 1), dim=1).reshape(-1).to(torch.int32).contiguous()
            cfg._keep.append(rows)
            setattr(arr[l], rows_f, rows.data_ptr())
            setattr(arr[l], n_f, rows.numel())
        arr[l].atom_mask, arr[l].atom_mask_list, arr[l].n_atom_mask = -1, None, 0
        am = sw.atom_mask
        if am is not None:
            if isinstance(am, int):
                arr[l].atom_mask = am
            else:
                idx = torch.as_tensor(am, device=dev).reshape(-1).to(torch.int32).contiguous()
                cfg._keep.append(idx)
                arr[l].atom_mask_list, arr[l].n_atom_mask = idx.data_ptr(), idx.numel()
    return arr


class EncoderFn(torch.autograd.Function):
    """inputs: plan, cfg, x_atoms, x_bond, x_fbond, then 14 live parameter tensors per layer.
    outputs: atoms, frags, bond, fbond [, attn_atoms, attn_frags, attn_bonds, attn_fbonds of the attention layer]."""

    @staticmethod
    def forward(ctx, plan: LayerPlan, cfg: EncoderConfig, x_atoms, x_bond, x_fbond, *params):
        f32 = ops._f32c
        x_atoms, x_bond, x_fbond = f32(x_atoms), f32(x_bond), f32(x_fbond)
        params = [f32(t) for t in params]
        frag_table = params.pop() if cfg.frag_table else None
        dev = x_atoms.device
        n_layers = len(cfg.layers)
        assert len(params) == n_layers * N_PARAMS
        if frag_table is not None and tuple(frag_table.shape) != (plan.frag.n_real, ops.H):
            raise ValueError(f"EncoderFn: frag_table must be [{plan.frag.n_real}, {ops.H}], got {tuple(frag_table.shape)}")
        need_grad = cfg.grad_enabled and any(ctx.needs_input_grad)
        if need_grad and _has_mask(cfg):
            raise NotImplementedError(
                "fragnet_b200: bond/atom/fragment-bond masks are inference-only (the reference applies them "
                "in-place under no_grad, gat2.py:173-176,227-231,275-278); run under torch.no_grad()")
        lib = ops._lib()
        layers = _layer_structs(cfg, params, dev)
        dropping = cfg.post_act and cfg.training and cfg.drop_p > 0
        # the forward gets the backward's need_dx_* as well: with a wanted d x_atoms, input dropout then runs as its own
        # kernel instead of inside the padding kernel (the backward's results do not depend on which one ran)
        need_dx = [int(need_grad and n) for n in ctx.needs_input_grad[2:5]]
        opts = _abi.CEncoderOpts(n_layers, int(cfg.post_act), float(cfg.drop_p), int(cfg.training),
                                 torch.initial_seed() & 0xFFFFFFFFFFFFFFFF, 0, cfg.precision, int(need_grad),
                                 *need_dx)
        cplan = plan.cstruct()
        if dropping:
            opts.offset = ops.reserve_rng(lib.fnb_encoder_rng_span(C.byref(cplan), C.byref(opts), layers))
        new = lambda rows, cols=ops.D: torch.empty((rows, cols), dtype=torch.float32, device=dev)
        run_frag_last = cfg.layers[-1].run_frag_block
        out_atoms, out_bond, out_fbond = new(plan.n_atoms), new(plan.bond.n_nodes), new(plan.fbond.n_nodes)
        out_frags = new(plan.n_frags) if run_frag_last else None
        attn_layer = next((l for l, s in enumerate(cfg.layers) if s.want_attention), None)
        attn = [None] * 4
        if attn_layer is not None:
            attn = [new(plan.n_atoms, ops.H), new(plan.n_frags, ops.H) if cfg.layers[attn_layer].run_frag_block else None,
                    new(plan.bond.n_nodes, ops.H), new(plan.fbond.n_nodes, ops.H)]
        ws_bytes = lib.fnb_encoder_workspace_bytes(C.byref(cplan), C.byref(opts), layers)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        pt = ops._ptr
        io = _abi.CEncoderIO(pt(x_atoms), pt(x_bond), pt(x_fbond), pt(out_atoms), pt(out_frags), pt(out_bond),
                             pt(out_fbond), pt(attn[0]), pt(attn[1]), pt(attn[2]), pt(attn[3]))
        io.frag_table = pt(frag_table)
        _abi.check(lib.fnb_encoder_forward(C.byref(cplan), C.byref(opts), layers, C.byref(io), pt(ws), ws_bytes,
                                           pt(ops.scratch(dev)), ops._stream()), "encoder_forward")
        if out_frags is None:
            out_frags = out_atoms.new_zeros((plan.n_frags, ops.D))     # placeholder nobody reads
        outs = [out_atoms, out_frags, out_bond, out_fbond]
        if attn_layer is not None:
            if attn[1] is None:
                attn[1] = out_atoms.new_zeros((plan.n_frags, ops.H))
            outs += attn
            ctx.mark_non_differentiable(*attn)
        if need_grad:
            ctx.set_materialize_grads(False)
            ctx.plan, ctx.cfg, ctx.opts, ctx.ws = plan, cfg, opts, ws
            ctx.has_table = frag_table is not None
            ctx.save_for_backward(x_atoms, x_bond, x_fbond, *params, out_atoms, out_frags, out_bond, out_fbond,
                                  *([frag_table] if frag_table is not None else []))
        return tuple(outs)

    @staticmethod
    def backward(ctx, g_atoms, g_frags, g_bond, g_fbond, *_attn_grads):
        plan, cfg, opts, ws = ctx.plan, ctx.cfg, ctx.opts, ctx.ws
        saved = list(ctx.saved_tensors)
        frag_table = saved.pop() if ctx.has_table else None
        x_atoms, x_bond, x_fbond = saved[:3]
        params = list(saved[3:-4])
        out_atoms, out_frags, out_bond, out_fbond = saved[-4:]
        dev = x_atoms.device
        needs = ctx.needs_input_grad          # 2 x_atoms, 3 x_bond, 4 x_fbond, 5.. parameters
        lib = ops._lib()
        c = lambda t: None if t is None else ops._f32c(t)
        g_atoms, g_frags, g_bond, g_fbond = c(g_atoms), c(g_frags), c(g_bond), c(g_fbond)
        layers = _layer_structs(cfg, params, dev)
        # every parameter gradient of the pass lives in ONE flat buffer (views are handed to autograd)
        sizes = [p.numel() for p in params]
        flat = torch.empty(sum(sizes), dtype=torch.float32, device=dev)
        views = [v.view_as(p) for v, p in zip(flat.split(sizes), params)]
        grads = (_abi.CLayerGrads * len(cfg.layers))()
        for l in range(len(cfg.layers)):
            for name, v in zip(_abi.PARAM_FIELDS, views[l * N_PARAMS:(l + 1) * N_PARAMS]):
                setattr(grads[l], name, v.data_ptr())
        opts.need_dx_atoms, opts.need_dx_bond, opts.need_dx_fbond = int(needs[2]), int(needs[3]), int(needs[4])
        dx = [torch.empty_like(x) if n else None for x, n in zip((x_atoms, x_bond, x_fbond), needs[2:5])]
        cplan = plan.cstruct()
        bws_bytes = lib.fnb_encoder_bwd_workspace_bytes(C.byref(cplan), C.byref(opts), layers)
        bws = torch.empty(bws_bytes, dtype=torch.uint8, device=dev)
        pt = ops._ptr
        run_frag_last = cfg.layers[-1].run_frag_block
        io = _abi.CEncoderIO(pt(x_atoms), pt(x_bond), pt(x_fbond), pt(out_atoms), pt(out_frags) if run_frag_last else None,
                             pt(out_bond), pt(out_fbond), None, None, None, None, pt(g_atoms),
                             pt(g_frags) if run_frag_last else None, pt(g_bond), pt(g_fbond), pt(dx[0]), pt(dx[1]), pt(dx[2]))
        d_table = None
        if frag_table is not None:
            io.frag_table = pt(frag_table)
            # zero where no gradient reaches the fragment block (its backward does not run then)
            d_table = torch.zeros_like(frag_table)
            io.d_frag_table = pt(d_table)
        _abi.check(lib.fnb_encoder_backward(C.byref(cplan), C.byref(opts), layers, grads, C.byref(io), pt(ws), ws.numel(),
                                            pt(bws), bws_bytes, pt(ops.scratch(dev)), ops._stream()), "encoder_backward")
        out = []
        for l, sw in enumerate(cfg.layers):
            for j in range(N_PARAMS):
                k = l * N_PARAMS + j
                dead = j == _F_INDEX and not (sw.run_frag_block and g_frags is not None and l == len(cfg.layers) - 1)
                out.append(views[k] if needs[5 + k] and not dead else None)
        if frag_table is not None:
            out.append(d_table if needs[5 + len(params)] else None)
        return (None, None, dx[0], dx[1], dx[2], *out)


class DropoutReluFn(torch.autograd.Function):
    """y = ReLU(Dropout_p(x)) (reference gat2.py:414-418) or plain Dropout_p(x) with ``relu=False``
    (gat2.py:396) as a standalone op.  Nothing but y is kept for backward."""

    @staticmethod
    def forward(ctx, x, p: float, training: bool, relu: bool):
        x = ops._f32c(x)
        seed, offset = ops.next_rng(x.numel()) if (training and p > 0) else (0, 0)
        y = ops.dropout_relu_fwd(x, p, training, relu, seed, offset)
        ctx.cfg = (p, training, relu, seed, offset)
        if relu:
            ctx.save_for_backward(y)
        return y

    @staticmethod
    def backward(ctx, dy):
        p, training, relu, seed, offset = ctx.cfg
        dy = ops._f32c(dy)
        if relu:
            (y,) = ctx.saved_tensors
            return ops.dropout_relu_bwd(dy, y, p, training), None, None, None
        # plain dropout: the same keep-mask applied to dy (regenerated from the RNG counters)
        return ops.dropout_relu_fwd(dy, p, training, False, seed, offset), None, None, None


class PoolFn(torch.autograd.Function):
    """x_frags = scatter_add(x_atoms, atom_to_frag_ids) (reference gat2.py:234, gat2_lite.py:140) as a standalone op
    over the membership CSR of the batch plan; backward gathers the fragment gradient back to the member atoms."""

    @staticmethod
    def forward(ctx, plan: LayerPlan, x_atoms):
        x_atoms = ops._f32c(x_atoms)
        ctx.plan, ctx.n = plan, x_atoms.shape[0]
        pool = plan.pool
        return ops.segment_sum(pool.rowptr, pool.col, plan.n_frags, x_atoms)[0]

    @staticmethod
    def backward(ctx, g):
        return None, ops.segment_gather(ops._f32c(g), ops.D, ctx.plan.a2f32, ctx.n)


class ReadoutFn(torch.autograd.Function):
    """cat(scatter_add(x_atoms, batch), scatter_add(x_frags, frag_batch)) written in place into one
    [G,256] tensor (reference gat2.py:820-823, pretrain_heads.py:93-96)."""

    @staticmethod
    def forward(ctx, rp: ops.ReadoutPlan, x_atoms, x_frags):
        x_atoms, x_frags = ops._f32c(x_atoms), ops._f32c(x_frags)
        out = torch.empty((rp.n_graphs, 2 * ops.D), dtype=torch.float32, device=x_atoms.device)
        ops.segment_sum(rp.atom_ptr, None, rp.n_graphs, x_atoms, out=out, out_stride=2 * ops.D)
        ops.segment_sum(rp.frag_ptr, None, rp.n_graphs, x_frags, out=out[:, ops.D:], out_stride=2 * ops.D)
        ctx.rp, ctx.sizes = rp, (x_atoms.shape[0], x_frags.shape[0])
        return out

    @staticmethod
    def backward(ctx, g):
        rp, (na, nf) = ctx.rp, ctx.sizes
        g = ops._f32c(g)
        ga = ops.segment_gather(g, 2 * ops.D, rp.batch32, na)
        gf = ops.segment_gather(g[:, ops.D:], 2 * ops.D, rp.frag_batch32, nf)
        return None, ga, gf


# ------------------------------------------------------------------------------------------------
# Pretraining heads + loss (heads.cu)
HEAD_PARAM_COUNT = 26     # Wr, br, then (W0, b0, W1, b1, W2, b2) of bl, ba, da, fc


def _head_struct(tensors):
    s = _abi.CPretrainHeadParams()
    s.Wr, s.br = tensors[0].data_ptr(), tensors[1].data_ptr()
    for gi, group in enumerate(("bl", "ba", "da", "fc")):
        g = getattr(s, group)
        for fi, name in enumerate(_abi.MLP3_FIELDS):
            setattr(g, name, tensors[2 + gi * 6 + fi].data_ptr())
    return s


class PretrainHeadsFn(torch.autograd.Function):
    """``PretrainTask.forward`` (reference fragnet/model/gat/pretrain_heads.py:64-102) as one library call per
    direction.  inputs: readout plan, edge_index [2,Ea] int64, precision id, grad_enabled, x_atoms, x_frags,
    edge_feat, then the 26 head parameters (``HEAD_PARAM_COUNT``).  outputs: bond_length [Ea,1], bond_angle [Na,1],
    dihedral [Ea,1], energy [G,1].  The bond-length output has no library backward (the reference's loss never uses
    it); a gradient arriving there is handled by ``PretrainTask`` with library GEMMs instead."""

    @staticmethod
    def forward(ctx, rp, edge_index, precision: int, grad_enabled: bool, x_atoms, x_frags, edge_feat, *params):
        f32 = ops._f32c
        x_atoms, x_frags, edge_feat = f32(x_atoms), f32(x_frags), f32(edge_feat)
        params = [f32(t) for t in params]
        assert len(params) == HEAD_PARAM_COUNT
        dev = x_atoms.device
        lib = ops._lib()
        na, nf, ea, g = x_atoms.shape[0], x_frags.shape[0], edge_feat.shape[0], rp.n_graphs
        ei = edge_index if edge_index.is_contiguous() else edge_index.contiguous()
        assert ei.dtype == torch.int64 and ei.shape == (2, ea) and ei.device == dev
        new = lambda n: torch.empty((n, 1), dtype=torch.float32, device=dev)
        bl, ba, da, en = new(ea), new(na), new(ea), new(g)
        ws_bytes = lib.fnb_pretrain_heads_workspace_bytes(na, ea, g)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        pt = ops._ptr
        P = _head_struct(params)
        io = _abi.CPretrainHeadIO(pt(x_atoms), pt(x_frags), pt(edge_feat), pt(ei), pt(rp.atom_ptr), pt(rp.frag_ptr),
                                  pt(rp.batch32), pt(rp.frag_batch32), na, nf, ea, g, pt(bl), pt(ba), pt(da), pt(en))
        _abi.check(lib.fnb_pretrain_heads_forward(C.byref(P), C.byref(io), precision, pt(ws), ws_bytes,
                                                  pt(ops.scratch(dev)), ops._stream()), "pretrain_heads_forward")
        if grad_enabled and any(ctx.needs_input_grad):
            ctx.set_materialize_grads(False)
            ctx.rp, ctx.ei, ctx.precision, ctx.ws, ctx.sizes = rp, ei, precision, ws, (na, nf, ea, g)
            ctx.save_for_backward(x_atoms, x_frags, edge_feat, *params)
        return bl, ba, da, en

    @staticmethod
    def backward(ctx, g_bl, g_ba, g_da, g_en):
        if g_bl is not None:
            raise NotImplementedError("PretrainHeadsFn: the bond-length output has no library backward")
        rp, ei, ws = ctx.rp, ctx.ei, ctx.ws
        na, nf, ea, g = ctx.sizes
        saved = ctx.saved_tensors
        x_atoms, x_frags, edge_feat = saved[:3]
        params = list(saved[3:])
        dev = x_atoms.device
        lib = ops._lib()
        zeros = lambda n: torch.zeros((n, 1), dtype=torch.float32, device=dev)
        c = lambda t, n: zeros(n) if t is None else ops._f32c(t)
        g_ba, g_da, g_en = c(g_ba, na), c(g_da, ea), c(g_en, g)
        sizes = [p.numel() for p in params[8:]]          # ba, da, fc (the bond-length group gets no gradient)
        flat = torch.empty(sum(sizes), dtype=torch.float32, device=dev)
        views = [v.view_as(p) for v, p in zip(flat.split(sizes), params[8:])]
        D = _head_struct(params[:8] + views)              # Wr / br / bl slots are ignored by the library
        new = lambda n: torch.empty((n, ops.D), dtype=torch.float32, device=dev)
        d_atoms, d_frags, d_edge = new(na), new(nf), new(ea)
        bws_bytes = lib.fnb_pretrain_heads_bwd_workspace_bytes(na, ea, g)
        bws = torch.empty(bws_bytes, dtype=torch.uint8, device=dev)
        pt = ops._ptr
        P = _head_struct(params)
        io = _abi.CPretrainHeadIO(pt(x_atoms), pt(x_frags), pt(edge_feat), pt(ei), pt(rp.atom_ptr), pt(rp.frag_ptr),
                                  pt(rp.batch32), pt(rp.frag_batch32), na, nf, ea, g, None, None, None, None,
                                  pt(g_ba), pt(g_da), pt(g_en), pt(d_atoms), pt(d_frags), pt(d_edge))
        _abi.check(lib.fnb_pretrain_heads_backward(C.byref(P), C.byref(D), C.byref(io), ctx.precision, pt(ws), ws.numel(),
                                                   pt(bws), bws_bytes, pt(ops.scratch(dev)), ops._stream()),
                   "pretrain_heads_backward")
        needs = ctx.needs_input_grad
        pg = [None] * 8 + [v if needs[7 + 8 + i] else None for i, v in enumerate(views)]
        return (None, None, None, None, d_atoms if needs[4] else None, d_frags if needs[5] else None,
                d_edge if needs[6] else None, *pg)


class MseSumLossFn(torch.autograd.Function):
    """``sum_t w_t * MSELoss()(pred_t, target_t)`` in one launch; the gradients of the predictions are produced by
    the same launch and only scaled in backward.  inputs: weights tuple, then pred_0, target_0, pred_1, ..."""

    @staticmethod
    def forward(ctx, weights, *tensors):
        preds = [ops._f32c(t) for t in tensors[0::2]]
        targets = [ops._f32c(t) for t in tensors[1::2]]
        n = len(preds)
        assert n == len(weights) == len(targets) and 1 <= n <= 4
        dev = preds[0].device
        need = [ctx.needs_input_grad[1 + 2 * i] for i in range(n)]
        grads = [torch.empty_like(p) if nd else None for p, nd in zip(preds, need)]
        terms = (_abi.CMseTerm * n)()
        for i in range(n):
            assert preds[i].numel() == targets[i].numel() and preds[i].numel() > 0
            terms[i] = _abi.CMseTerm(ops._ptr(preds[i]), ops._ptr(targets[i]), preds[i].numel(), float(weights[i]),
                                     ops._ptr(grads[i]))
        loss = torch.empty((), dtype=torch.float32, device=dev)
        _abi.check(ops._lib().fnb_mse_sum_loss(terms, n, ops._ptr(loss), ops._ptr(ops.scratch(dev)), ops._stream()),
                   "mse_sum_loss")
        ctx.grads = grads
        return loss

    @staticmethod
    def backward(ctx, g):
        live = [x for x in ctx.grads if x is not None]
        if live:
            torch._foreach_mul_(live, g)
        out = [None]
        for x in ctx.grads:
            out += [x, None]
        return tuple(out)
