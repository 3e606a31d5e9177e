"""One training step per library call: ``FusedPretrainStep`` (pretraining) and ``FusedFineTuneStep`` (finetuning).

The reference's loop body (fragnet/train/pretrain/pretrain_utils.py:12-30) is::

    optimizer.zero_grad(); preds = model(batch); loss = 2*MSE(dihedral)+MSE(angle)+MSE(energy)
    loss.backward(); optimizer.step()            # torch.optim.Adam(model.parameters(), lr)  (pretrain_gat2.py:165)

Through ``nn.Module`` / autograd this works unchanged on the drop-in modules; it costs ~2.4 ms of host time per step
at batch 1024, more than the device needs.  ``FusedPretrainStep`` runs the same arithmetic for a ``FragNetPreTrain``
model as ``fnb_pretrain_step`` (collate, forward, loss, backward: one call) + optional gradient all-reduce +
``fnb_adam_step`` (one launch over a flat parameter buffer).  The model's parameters stay ordinary ``nn.Parameter``
objects with their names and shapes (``state_dict`` round-trips); those that receive gradients are re-homed as views
into one flat buffer and their ``.grad`` are views into a second one.

``FusedFineTuneStep`` does the same for a ``FragNetFineTune`` model and the finetuning loop's body
(fragnet/train/utils.py:330-470: ``model(batch)`` -> MSE or masked BCE -> backward -> Adam) with ``fnb_finetune_step``.
It honours frozen parameters (``requires_grad = False``) in the layout the library supports -- the lower encoder layers
or the whole encoder, and any of the head's linears: only the trained tensors are re-homed and updated, and the
backward stops below the lowest trained layer.  Both steps train data-parallel over a process group: the mean of the
ranks' gradients and Adam in one kernel over NVLink peer memory (``fnb_allreduce_adam_runs``), or NCCL.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional

import torch
import torch.distributed as dist

from .. import _abi, config, ops
from ..autograd import N_PARAMS, _F_INDEX

from .optim import flat_views as _flat_views


def _on(batch, k, dev, dtype):
    t = batch[k]
    if t.device != dev or t.dtype != dtype or not t.is_contiguous():
        t = t.to(device=dev, dtype=dtype).contiguous()
    return t


def _encoder_structs(layer_params, grad_of, frag_block=True):
    """``fnb_layer_params`` / ``fnb_layer_grads`` arrays of an encoder's layers (fragment block in the last one only,
    or with ``frag_block=False`` in none).  A ``None`` tensor is one the program does not read (a fragment-connection
    tensor of gat2_lite / gat2_edge)."""
    n_layers = len(layer_params)
    layers, grads = (_abi.CLayerParams * n_layers)(), (_abi.CLayerGrads * n_layers)()
    for li, ps in enumerate(layer_params):
        L, G = layers[li], grads[li]
        for name, p in zip(_abi.PARAM_FIELDS, ps):
            setattr(L, name, None if p is None else p.data_ptr())
            g = None if p is None else grad_of.get(id(p))
            setattr(G, name, None if g is None else g.data_ptr())
        L.K_bond, L.K_atom = ps[0].shape[1], ps[8].shape[1]
        L.K_fbond = ops.D if ps[2] is None else ps[2].shape[1]
        L.run_frag_block, L.want_attention = int(frag_block and li == n_layers - 1), 0
        L.bond_mask = L.frag_bond_mask = L.atom_mask = -1
        L.atom_mask_list, L.n_atom_mask = None, 0
    assert len(layer_params[0]) == N_PARAMS
    return layers, grads


def _same_on_every_rank(value, group, what: str) -> None:
    """Collective: ``ValueError`` on every rank of ``group`` unless ``value`` (picklable) is equal on all of them.  A
    step whose ranks disagree on its layout would otherwise wait forever in the first exchange, or read past a buffer."""
    got = [None] * dist.get_world_size(group)
    dist.all_gather_object(got, value, group=group)
    if any(v != got[0] for v in got):
        raise ValueError(f"fragnet_b200: {what} differ between the ranks of the process group")


class _FlatStep:
    """What the one-call steps share: the live parameters re-homed as views of one flat buffer (their ``.grad`` views
    of a second one), the flat Adam update, a caller's ``torch.optim.Adam`` kept truthful, the gradient exchange of
    data-parallel training, and the collate of the next batch underneath the running step."""

    def _bind_flat(self, live, dev, group=None, also=()):
        """Re-homes ``live`` into the flat buffers; returns the gradient views.  ``group``: the ``torch.distributed``
        process group of data-parallel training (``None``: the default group if one is initialised); with more than one
        rank the gradient buffer is set up for the exchange, and the flat parameters and the tensors ``also`` are
        broadcast from the group's rank 0.  Collective in that case: every rank of the group has to call it."""
        self.group, self._peers = group, None
        g_store = self._symmetric_gradient_buffer(live, dev, group)
        self.live = live
        self.flat_p, p_views = _flat_views(live, dev)
        self.flat_g, g_views = _flat_views(live, dev, storage=g_store)
        with torch.no_grad():
            torch._foreach_copy_(p_views, [p.data for p in live])
            for p, v, g in zip(live, p_views, g_views):
                p.data = v
                p.grad = g
            if self.world_size > 1:
                # DDP / Fabric broadcast rank 0's parameters at wrap time (finetune_gat2_pl.py:230): differently seeded
                # ranks, or a checkpoint loaded on one rank only, must not diverge silently
                src = dist.get_global_rank(group, 0) if group is not None else 0
                for t in (self.flat_p, *(p.data for p in also)):
                    dist.broadcast(t, src=src, group=group)
        self.exp_avg = torch.zeros_like(self.flat_p)
        self.exp_avg_sq = torch.zeros_like(self.flat_p)
        self.t = 0
        self._adam_runs = [(0, self.flat_p.numel(), 0)]    # (first, end, steps behind self.t) of the flat buffer
        self._p_views = p_views
        self._ws: Optional[torch.Tensor] = None
        self._loss = torch.zeros(8, dtype=torch.float32, device=dev)      # ring of loss scalars
        self._loss_i = 0
        # collate of the next batch underneath the running step (prefetch_plan): two alternating plan arenas
        self._plan_arenas: List[Optional[torch.Tensor]] = [None, None]
        self._step_parity: Optional[int] = None     # arena the step launched last reads, if it found its plan prefetched
        self._prefetched = None          # (key of the batch inputs, arena, tensors kept alive)
        self.plan_hits = 0               # steps that found their plan prefetched
        return g_views

    def bound_to_model(self) -> bool:
        """True while every live parameter still is its view of the flat buffer (``model.to()``, ``.cpu()`` or a
        re-assigned ``p.data`` break the binding; the caller then has to fall back to the generic loop)."""
        return all(p.data_ptr() == v.data_ptr() and p.device == v.device for p, v in zip(self.live, self._p_views))

    def attach_optimizer(self, optimizer) -> None:
        """Keep a caller-owned ``torch.optim.Adam`` truthful: its ``state`` entries of the live parameters become VIEWS
        of this object's moment buffers plus step counters, so ``optimizer.state_dict()`` checkpoints the real state;
        moments already present in ``optimizer.state`` (a resumed run) are adopted first.  Step counts stay per
        parameter, as in ``torch.optim.Adam``: when some parameters have state and others not (a layer unfrozen
        after the others trained for a while), the new ones start from step 1.  With several ranks this is collective,
        and the ranks' step counts must agree (``ValueError`` on every rank otherwise): each rank updates its own
        moments, as DDP's optimizers do, so a rank resumed from another checkpoint would diverge."""
        from .optim import flat_views
        _, m_views = flat_views(self.live, self.dev, storage=self.exp_avg)
        _, v_views = flat_views(self.live, self.dev, storage=self.exp_avg_sq)
        steps = [int(optimizer.state[p]["step"]) if "step" in optimizer.state.get(p, {}) else None for p in self.live]
        with torch.no_grad():
            for p, m, v in zip(self.live, m_views, v_views):
                st = optimizer.state.get(p)
                if st and "exp_avg" in st:
                    m.copy_(st["exp_avg"])
                    v.copy_(st["exp_avg_sq"])
        known = [s for s in steps if s is not None]
        if known:
            self.t = max(known)
        lags = [self.t - s if s is not None else (self.t if known else 0) for s in steps]
        # contiguous runs of the flat buffer whose parameters are equally many steps behind (one run in a plain run)
        base = self.flat_p.data_ptr()
        starts = [(v.data_ptr() - base) // self.flat_p.element_size() for v in self._p_views] + [self.flat_p.numel()]
        self._adam_runs = []
        for i, lag in enumerate(lags):
            if self._adam_runs and self._adam_runs[-1][2] == lag:
                self._adam_runs[-1] = (self._adam_runs[-1][0], starts[i + 1], lag)
            else:
                self._adam_runs.append((starts[i], starts[i + 1], lag))
        if self.world_size > 1:
            _same_on_every_rank((self.t, self._adam_runs), self.group, "the optimizer's step counts")
        self._opt_steps = {lag: torch.tensor(float(self.t - lag)) for lag in set(lags)}
        for p, m, v, lag in zip(self.live, m_views, v_views, lags):
            optimizer.state[p] = {"step": self._opt_steps[lag], "exp_avg": m, "exp_avg_sq": v}

    def _sync_opt_steps(self) -> None:
        for lag, t in getattr(self, "_opt_steps", {}).items():
            t.fill_(float(self.t - lag))

    def _adam(self) -> None:
        """``fnb_adam_step`` over the flat buffers at step ``self.t`` (one launch per run of equal step counts)."""
        for lo, hi, lag in self._adam_runs:
            _abi.check(ops._lib().fnb_adam_step(
                ops._p(self.flat_p[lo:]), ops._p(self.flat_g[lo:]), ops._p(self.exp_avg[lo:]),
                ops._p(self.exp_avg_sq[lo:]), hi - lo, self.lr, self.betas[0], self.betas[1], self.eps,
                self.weight_decay, self.t - lag, ops._stream()), "adam_step")
        self._sync_opt_steps()

    def _exchange_adam(self) -> None:
        """Mean of the ranks' gradients + Adam at step ``self.t``, per run of equal step counts: one
        ``fnb_allreduce_adam_runs`` kernel over NVLink peer memory (csrc/dist.cu) when the exchange buffer is set up,
        else ``dist.all_reduce`` + scale + ``_adam()`` (a single rank: ``_adam()`` alone)."""
        if self._peers is not None and len(self._adam_runs) <= _abi.MAX_ADAM_RUNS:
            self._epoch += 1
            runs = (_abi.CAdamRun * len(self._adam_runs))(*((lo, hi, self.t - lag) for lo, hi, lag in self._adam_runs))
            _abi.check(ops._lib().fnb_allreduce_adam_runs(
                C.byref(self._peers), ops._p(self.flat_p), ops._p(self.exp_avg), ops._p(self.exp_avg_sq),
                self.flat_p.numel(), runs, len(runs), self.lr, self.betas[0], self.betas[1], self.eps,
                self.weight_decay, self._epoch & 0xFFFFFFFF, ops._p(self._done), ops._stream()), "allreduce_adam_runs")
            self._sync_opt_steps()
            return
        w = self.world_size
        if w > 1:
            dist.all_reduce(self.flat_g, op=dist.ReduceOp.SUM, group=self.group)
            self.flat_g.mul_(1.0 / w)
        self._adam()

    def _symmetric_gradient_buffer(self, live, dev, group):
        """World > 1: the flat gradient buffer is allocated in symmetric memory (peer-mapped over NVLink at rendezvous)
        so that ``fnb_allreduce_adam_runs`` can read every rank's gradients directly -- exchange, mean and Adam are then
        one kernel instead of ncclAllReduce + scale + Adam.  Returns the storage tensor, or None (single rank, no NVLink
        peer access, a backend other than NCCL, ``FNB_FUSED_ALLREDUCE=0``): ``step`` then uses ``dist.all_reduce`` +
        ``fnb_adam_step``."""
        import os
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) < 2:
            return None
        w = dist.get_world_size(group)
        if os.environ.get("FNB_FUSED_ALLREDUCE", "1") == "0" or w > 8 or dist.get_backend(group) != "nccl":
            return None
        from .optim import ALIGN
        total = sum((p.numel() + ALIGN - 1) // ALIGN * ALIGN for p in live)
        try:
            import torch.distributed._symmetric_memory as symm
            pg = group if group is not None else dist.group.WORLD
            g = symm.empty(total, dtype=torch.float32, device=dev)
            flags = symm.empty(2 * w, dtype=torch.int32, device=dev)
            g.zero_()
            flags.zero_()
            hg, hf = symm.rendezvous(g, pg), symm.rendezvous(flags, pg)
            ps = _abi.CPeerSet()
            for r in range(w):
                ps.grads[r], ps.flags[r] = hg.buffer_ptrs[r], hf.buffer_ptrs[r]
            ps.world, ps.rank = w, hg.rank
            ok = torch.ones(1, device=dev)
        except Exception as ex:          # no P2P between these devices, or an older torch: NCCL path
            import warnings
            warnings.warn(f"fragnet_b200: symmetric-memory gradient exchange unavailable ({type(ex).__name__}: {ex}); "
                          "using ncclAllReduce", RuntimeWarning)
            g, ok = None, torch.zeros(1, device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)       # all ranks take the same path (zeroed flags visible)
        if float(ok) < 1.0 or g is None:
            return None
        self._peers, self._flags, self._epoch = ps, flags, 0
        self._done = torch.zeros(1, dtype=torch.int32, device=dev)
        self._symm_keep = (hg, hf)
        return g

    @property
    def world_size(self) -> int:
        return dist.get_world_size(self.group) if dist.is_available() and dist.is_initialized() else 1

    def _next_loss(self) -> torch.Tensor:
        self._loss_i = (self._loss_i + 1) % self._loss.numel()
        return self._loss[self._loss_i]

    def _plan_inputs(self, b, g: int, convert: bool = True):
        """``ops.batch_inputs`` of a batch dict with ``g`` molecules (``prefetch_plan`` and the step build the same)."""
        return ops.batch_inputs(b["edge_index"], b["frag_index"], b["atom_to_frag_ids"], b["edge_index_bonds_graph"],
                                b["edge_attr_bonds"], b["edge_index_fbonds"], b["edge_attr_fbonds"], b["batch"],
                                b["frag_batch"], b["x_atoms"].shape[0], b["x_frags"].shape[0],
                                b["node_features_bonds"].shape[0], b["node_features_fbonds"].shape[0], g, self.dev,
                                convert)

    def _batch_inputs(self, batch, g: int):
        """``fnb_batch_inputs`` of a batch dict with ``g`` molecules, the tensors it points into, and the raw features."""
        inp, keep = self._plan_inputs(batch, g)
        feats = tuple(_on(batch, k, self.dev, torch.float32) for k in ("x_atoms", "node_features_bonds",
                                                                        "node_features_fbonds"))
        return inp, keep + feats, feats

    def _take_prefetched(self, inp) -> Optional[int]:
        """Arena address of the plan ``prefetch_plan`` built for exactly these batch inputs, or None."""
        pre, self._prefetched = self._prefetched, None       # one prefetch serves one step
        self._step_parity = None
        if pre is not None and pre[0] == self._plan_key(inp):
            self._step_parity = pre[3]             # this arena is now in use until the step has run
            self.plan_hits += 1
            return pre[1].data_ptr()
        return None

    # ---- collate of the next batch underneath the running step -------------------------------------------------------
    @staticmethod
    def _plan_key(inp: "_abi.CBatchInputs"):
        return tuple(getattr(inp, n) for n, _ in _abi.CBatchInputs._fields_)

    def prefetch_plan(self, next_batch, ready_event: Optional["torch.cuda.Event"] = None) -> bool:
        """Queue the on-device collate (``fnb_batch_plan_build``) of the batch the NEXT ``step`` call will get, on a
        library stream underneath the step that is running -- the plan depends on nothing but the batch's index tensors,
        and without it the first attention kernel of a step waits ~50 us for nine small launches that compete with the
        layer-0 GEMMs for SMs.  ``ready_event``: recorded once the tensors of ``next_batch`` are complete (a
        ``DevicePrefetcher`` slot still being copied); None if they already are.  Only batches that need no dtype /
        device conversion qualify (returns False otherwise: the step then collates by itself, as always).  The tensors
        must not be modified until that step has been launched."""
        self._prefetched = None
        dev = self.dev
        got = self._plan_inputs(next_batch, next_batch["y"].numel() // self._y_width, convert=False)
        if got is None:
            return False
        inp, keep = got
        lib = ops._lib()
        need = lib.fnb_batch_plan_bytes(C.byref(inp))
        if need == 0:
            return False
        # never the arena the step launched last reads (its backward still needs the plan); a second prefetch before the
        # next step simply replaces the first
        parity = 0 if self._step_parity is None else 1 - self._step_parity
        arena = self._plan_arenas[parity]
        if arena is None or arena.numel() < need:
            # (re)allocation: the block may have been freed by work still running on the compute stream, and the collate
            # writes it from another stream -- rare (first steps, a larger batch), so simply wait
            torch.cuda.current_stream(dev).synchronize()
            arena = torch.empty(int(need * 1.25) + 256, dtype=torch.uint8, device=dev)
            self._plan_arenas[parity] = arena
        ev = C.c_void_p(ready_event.cuda_event) if ready_event is not None else None
        rc = lib.fnb_pretrain_plan_prefetch(C.byref(inp), ops._ptr(arena), arena.numel(), ev)
        if rc != 0:
            return False                 # single-stream mode: the step collates by itself
        self._prefetched = (self._plan_key(inp), arena, keep, parity)
        return True

    # ---- the step: what the subclass's _args / _NATIVE describe --------------------------------------------------------
    _y_width = 1          # entries of batch["y"] per molecule

    def _run(self, batch, backward: bool, want_preds: bool = False):
        lib = ops._lib()
        a, loss, preds, keep = self._args(batch, backward, want_preds)
        if self._draws(a):
            a.offset = ops.reserve_rng(getattr(lib, f"fnb_{self._NATIVE}_rng_span")(C.byref(a)))
        need = getattr(lib, f"fnb_{self._NATIVE}_workspace_bytes")(C.byref(a))
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(int(need * 1.25) + 256, dtype=torch.uint8, device=self.dev)
        _abi.check(getattr(lib, f"fnb_{self._NATIVE}")(C.byref(a), ops._ptr(self._ws), self._ws.numel(),
                                                       ops._ptr(ops.scratch(self.dev)), ops._stream()), self._NATIVE)
        del keep        # stream-ordered allocator: safe to release once the launches are queued on this stream
        return loss, preds

    def step(self, batch, next_batch=None, next_ready=None) -> torch.Tensor:
        """collate + forward + loss + backward (+ all-reduce) + Adam on one batch dict; returns the loss.
        ``next_batch`` (optional): the batch of the following call, whose collate is then queued underneath this step
        (``prefetch_plan``); ``next_ready``: the CUDA event after which its tensors are complete, if they are not yet."""
        loss = self._step(batch)
        if next_batch is not None:
            self.prefetch_plan(next_batch, next_ready)
        return loss

    def _step(self, batch) -> torch.Tensor:
        loss, _ = self._run(batch, backward=True)
        self.t += 1
        self._exchange_adam()
        return loss

    def forward_backward(self, batch) -> torch.Tensor:
        """Gradients only (``p.grad`` of the live parameters are views of ``flat_g``), no parameter update."""
        return self._run(batch, backward=True)[0]

    @torch.no_grad()
    def evaluate(self, batch, return_predictions: bool = False):
        """Forward + loss without gradients (validation)."""
        loss, preds = self._run(batch, backward=False, want_preds=return_predictions)
        return (loss, preds) if return_predictions else loss


class FusedPretrainStep(_FlatStep):
    """``step(batch) -> loss`` (0-dim CUDA tensor) for a ``FragNetPreTrain`` model; Adam hyper-parameters as
    ``torch.optim.Adam``.  ``group``: a ``torch.distributed`` process group for data-parallel training (mean of the
    per-rank gradients, the DDP semantics of finetune_gat2_pl.py:230); ``None`` uses the default group if one is
    initialised."""

    def __init__(self, model, lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 0.0,
                 group=None):
        enc, head = model.pretrain, model.head
        if not head._library_shapes():
            raise NotImplementedError("FusedPretrainStep needs PretrainTask(128, 1, L=2)")
        self.model = model
        self.lr, self.betas, self.eps, self.weight_decay = float(lr), betas, float(eps), float(weight_decay)
        self.dev = dev = ops.require_cuda(enc.layers[0].a.device)
        for layer in enc.layers:
            layer._check_geometry()
        n_layers = len(enc.layers)
        layer_params = [list(layer._live_parameters()) for layer in enc.layers]
        head_params = head._parameters_in_library_order()
        # parameters that receive a gradient, in flat-buffer order
        live: List[torch.nn.Parameter] = []
        for li, ps in enumerate(layer_params):
            live += [p for j, p in enumerate(ps) if j != _F_INDEX or li == n_layers - 1]
        live += head_params[8:]                       # ba, da, FC stacks (the bond-length head is never trained)
        if any(p.dtype != torch.float32 or p.device != dev for p in live):
            raise ValueError("FusedPretrainStep needs fp32 parameters on one CUDA device")
        g_views = self._bind_flat(live, dev, group)
        p_views = self._p_views
        grad_of: Dict[int, torch.Tensor] = {id(p): g for p, g in zip(live, g_views)}
        # ---- C structs (built once: parameter storage never moves afterwards)
        self._layers, self._layer_grads = _encoder_structs(layer_params, grad_of)
        self._heads, self._head_grads = _abi.CPretrainHeadParams(), _abi.CPretrainHeadParams()
        self._heads.Wr, self._heads.br = head_params[0].data_ptr(), head_params[1].data_ptr()
        for gi, group_name in enumerate(("bl", "ba", "da", "fc")):
            for fi, fname in enumerate(_abi.MLP3_FIELDS):
                p = head_params[2 + gi * 6 + fi]
                setattr(getattr(self._heads, group_name), fname, p.data_ptr())
                g = grad_of.get(id(p))
                setattr(getattr(self._head_grads, group_name), fname, None if g is None else g.data_ptr())
        self._keep = (layer_params, head_params, p_views, g_views)
        self.n_layers = n_layers

    def _args(self, batch, backward: bool, want_preds: bool):
        dev = self.dev
        f32 = lambda k: _on(batch, k, dev, torch.float32)
        t_ba, t_dh, y = f32("bnd_angl"), f32("dh_angl"), f32("y")
        g = y.numel()
        inp, tensors, (xa, xb, xfb) = self._batch_inputs(batch, g)
        na, nb = inp.n_atoms, inp.n_bonds
        if t_ba.numel() != na or t_dh.numel() != nb:
            raise ValueError("fragnet_b200: bnd_angl / dh_angl must have one entry per atom / directed bond")
        pt = ops._ptr
        a = _abi.CPretrainStepArgs()
        a.batch = inp
        a.x_atoms, a.x_bond, a.x_fbond = pt(xa), pt(xb), pt(xfb)
        a.t_bond_angle, a.t_dihedral, a.t_energy = pt(t_ba), pt(t_dh), pt(y)
        a.n_layers = self.n_layers
        a.layers = C.cast(self._layers, C.c_void_p)
        a.layer_grads = C.cast(self._layer_grads, C.c_void_p)
        a.heads = C.cast(C.pointer(self._heads), C.c_void_p)
        a.head_grads = C.cast(C.pointer(self._head_grads), C.c_void_p)
        enc = self.model.pretrain
        training = bool(self.model.training)
        a.drop_p, a.training = float(enc.dropout.p), int(training)
        a.seed, a.offset = torch.initial_seed() & 0xFFFFFFFFFFFFFFFF, 0
        a.precision, a.backward = config.precision_id(), int(backward)
        loss = self._next_loss()
        a.loss = loss.data_ptr()
        preds = None
        if want_preds:
            new = lambda n: torch.empty((n, 1), dtype=torch.float32, device=dev)
            preds = (new(nb), new(na), new(nb), new(g))
            a.bond_length, a.bond_angle, a.dihedral, a.energy = (pt(t) for t in preds)
        keep = tensors + (t_ba, t_dh, y)
        a.plan_arena = self._take_prefetched(a.batch)       # collated ahead of this step (see prefetch_plan)
        return a, loss, preds, keep

    _NATIVE = "pretrain_step"

    @staticmethod
    def _draws(a) -> bool:
        return bool(a.training and a.drop_p > 0)


def _act_id(module) -> Optional[int]:
    """The library's activation code of an FTHead activation module, or None if it has none."""
    import torch.nn as nn
    exact = {nn.ReLU: _abi.ACT_RELU, nn.SiLU: _abi.ACT_SILU, nn.SELU: _abi.ACT_SELU, nn.ReLU6: _abi.ACT_RELU6}
    if type(module) in exact:
        return exact[type(module)]
    if type(module) is nn.CELU and module.alpha == 1.0:
        return _abi.ACT_CELU
    if type(module) is nn.GELU and module.approximate == "none":
        return _abi.ACT_GELU
    if type(module) is nn.LeakyReLU and module.negative_slope == 0.01:
        return _abi.ACT_LEAKYRELU
    return None


def _head_layers(head):
    """(linears, p_in, p_out, act) per layer of an FTHead1-4, the arrangement of gat2.py:569-751."""
    from ..model.gat import gat2
    kind = type(head)
    if kind in (gat2.FTHead3, gat2.FTHead2):
        # act(dropout(linear(x))) per hidden layer, bare last linear; FTHead2: ReLU, its own p = 0.1 (gat2.py:745-751)
        act = _abi.ACT_RELU if kind is gat2.FTHead2 else _act_id(getattr(head, "activation", None))
        lins = list(head.predictor)
        p = float(head.dropout.p)
        return [(lin, 0.0, p if i + 1 < len(lins) else 0.0, act if i + 1 < len(lins) else _abi.ACT_NONE)
                for i, lin in enumerate(lins)]
    if kind in (gat2.FTHead1, gat2.FTHead4):
        # out(dropout(act(linear(dropout(x))))) (gat2.py:580-588, :669-675)
        first, last = (head.lin1, head.out) if kind is gat2.FTHead1 else (head.dense, head.out_proj)
        act = _abi.ACT_RELU if kind is gat2.FTHead1 else _act_id(getattr(head, "activation", None))
        p = float(head.dropout.p)
        return [(first, p, 0.0, act), (last, p, 0.0, _abi.ACT_NONE)]
    return None


def _check_model(model, module, who: str):
    """The head spec of a ``module.FragNetFineTune`` the one-call step covers, or ``NotImplementedError``."""
    if type(model) is not module.FragNetFineTune:
        raise NotImplementedError(f"{who} needs {module.__name__}.FragNetFineTune "
                                  f"(got {type(model).__module__}.{type(model).__name__})")
    spec = _head_layers(getattr(model, "fthead", None))
    if spec is None or any(act is None for _, _, _, act in spec):
        raise NotImplementedError(f"{who} needs an FTHead1-4 head with a relu, celu, silu, gelu, selu, relu6 or "
                                  "leakyrelu activation")
    if len(spec) > _abi.MLP_MAX_LAYERS or spec[0][0].in_features != 2 * ops.D:
        raise NotImplementedError(f"{who}: unsupported head shape")
    for layer in model.pretrain.layers:
        layer._check_geometry()
    return spec


def _trained_set(spec, layer_params, units):
    """``_analyse``'s result from the encoder's freezable units (one per layer); the head's linears are appended."""
    n_layers = len(layer_params)
    units = units + [[lin.weight, lin.bias] for lin, _, _, _ in spec]
    trained = []
    for u in units:
        if len({p.requires_grad for p in u}) > 1:
            raise NotImplementedError("FusedFineTuneStep: every live tensor of an encoder layer, and weight and bias "
                                      "of a head linear, must be frozen or trained together")
        trained.append(u[0].requires_grad)
    enc_trained = trained[:n_layers]
    first = enc_trained.index(True) if any(enc_trained) else n_layers
    if not all(enc_trained[first:]):
        raise NotImplementedError("FusedFineTuneStep: frozen encoder layers must be the lowest ones (0 .. k-1)")
    live = [p for u, t in zip(units, trained) if t for p in u]
    if not live:
        raise NotImplementedError("FusedFineTuneStep: the model has no parameter to train")
    return spec, layer_params, units, live, first


class FusedFineTuneStep(_FlatStep):
    """``step(batch) -> loss`` (0-dim CUDA tensor) for this package's gat2 ``FragNetFineTune`` with an FTHead1-4 head:
    collate, encoder, readout, head, loss and every gradient in one ``fnb_finetune_step`` call, then Adam over the flat
    buffers (hyper-parameters as ``torch.optim.Adam``).  ``loss``: ``"mse"`` (``nn.MSELoss`` over the flattened
    predictions, ``TrainerFineTune.train_regr``) or ``"bce"`` (BCE-with-logits over the labels > -0.5,
    ``TrainerFineTune.train_clsf_bce``).

    Frozen parameters (``requires_grad = False``, read at construction) are honoured: the trained set is the library's
    live tensors that require a gradient, and only those go into the flat buffers and get Adam state; frozen tensors
    keep their storage and their ``.grad``.  The library freezes whole units: all live tensors of one encoder layer (the
    last layer's ``f`` included), ``weight`` and ``bias`` of one head linear, and frozen encoder layers must be the
    lowest ones (``0 .. k-1``, or all of them).  The backward then stops at the lowest trained layer.

    ``FusedLiteFineTuneStep`` and ``FusedEdgeFineTuneStep`` do the same for the ``gat2_lite`` and ``gat2_edge``
    versions of ``FragNetFineTune``; ``finetune_step_class(model)`` picks the class of a model.

    Data-parallel training (``group``: a ``torch.distributed`` process group, ``dist.group.WORLD`` included) follows
    DDP: every rank computes the gradient of its own batch's loss (MSE or masked BCE divided by its own count, as Fabric
    DDP does), and Adam applies the mean of the ranks' gradients; the parameters stay bitwise identical on every rank.
    The construction is collective: it checks that every rank built the same layout (the same trained set, shapes and
    lowest trained layer; ``ValueError`` on every rank otherwise) and broadcasts the model's parameters, trained and
    frozen, and buffers from the group's rank 0, as DDP does at wrap time.  The exchange is ``fnb_allreduce_adam_runs`` over NVLink peer memory on NCCL
    groups of up to 8 ranks with peer access, else ``dist.all_reduce`` + ``fnb_adam_step``.  Dropout counters stay per
    rank.  A ``requires_grad`` change needs a new step, built by every rank in the same step.  Without ``group``, an
    initialised default group of more than one rank is refused (``NotImplementedError``): one model per rank is then
    trained on its own by the generic loop, e.g. one hyper-parameter trial per rank.

    Models the library does not cover raise ``NotImplementedError``: other heads or activations (PReLU and RReLU among
    them), another model version than the class's, other encoder geometries, other freezing patterns (a frozen layer
    above a trained one, a frozen tensor inside a trained layer or linear) and a model with nothing to train."""

    _NATIVE = "finetune_step"
    _VARIANT = _abi.VARIANT_GAT2
    _EXTRA_KEYS = ()          # batch entries the step reads beyond the gat2 hot path (DevicePrefetcher's ``keep``)

    def __init__(self, model, lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 0.0,
                 loss: str = "mse", group=None):
        if loss not in ("mse", "bce"):
            raise ValueError(f"FusedFineTuneStep: loss must be 'mse' or 'bce', got {loss!r}")
        spec, layer_params, units, live, self.first_trained_layer = self._analyse(model)
        if group is None and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            raise NotImplementedError(f"{type(self).__name__} runs on one GPU unless a process group is passed (group=)")
        self.model, self.loss_kind = model, loss
        self.lr, self.betas, self.eps, self.weight_decay = float(lr), betas, float(eps), float(weight_decay)
        self.dev = dev = ops.require_cuda(model.pretrain.layers[0].a.device)
        if any(p.dtype != torch.float32 or p.device != dev for u in units for p in u):
            raise ValueError("FusedFineTuneStep needs fp32 parameters on one CUDA device")
        self._requires = [p.requires_grad for u in units for p in u]
        n_layers = len(layer_params)
        if group is not None and dist.get_world_size(group) > 1:
            _same_on_every_rank((type(self).__name__, [tuple(p.shape) for u in units for p in u], self._requires,
                                 self.first_trained_layer), group, "the models' trained sets, shapes or frozen layers")
        trained = {id(p) for p in live}
        g_views = self._bind_flat(live, dev, group, also=[t for t in (*model.parameters(), *model.buffers())
                                                          if id(t) not in trained])
        grad_of: Dict[int, torch.Tensor] = {id(p): g for p, g in zip(live, g_views)}
        self._grad_of = grad_of
        self._layers, self._layer_grads = _encoder_structs(layer_params, grad_of, self._VARIANT != _abi.VARIANT_LITE)
        self._head = (_abi.CMlpLayer * len(spec))()
        for h, (lin, p_in, p_out, act) in zip(self._head, spec):
            h.W, h.b = lin.weight.data_ptr(), lin.bias.data_ptr()
            if id(lin.weight) in grad_of:                   # frozen linear: dW = db = NULL
                h.dW, h.db = grad_of[id(lin.weight)].data_ptr(), grad_of[id(lin.bias)].data_ptr()
            h.in_dim, h.out_dim, h.p_in, h.p_out, h.act = lin.in_features, lin.out_features, p_in, p_out, act
        self.n_classes = self._y_width = spec[-1][0].out_features
        self._head_drops = any(p_in > 0 or p_out > 0 for _, p_in, p_out, _ in spec)
        self._keep = (layer_params, self._p_views, g_views)
        self._units = units
        self.n_layers = n_layers

    @staticmethod
    def _analyse(model):
        """(head spec, encoder live tensors per layer, freezable units, trained tensors in flat-buffer order, first
        trained encoder layer) of a model, or ``NotImplementedError`` for one the library does not cover."""
        from ..model.gat import gat2
        spec = _check_model(model, gat2, "FusedFineTuneStep")
        enc = model.pretrain
        n_layers = len(enc.layers)
        layer_params = [list(layer._live_parameters()) for layer in enc.layers]
        # the library's live tensors per unit it can freeze: encoder layers (the dead f of lower layers left out), then
        # the head's linears
        units = [[p for j, p in enumerate(ps) if j != _F_INDEX or li == n_layers - 1] for li, ps in enumerate(layer_params)]
        return _trained_set(spec, layer_params, units)

    @classmethod
    def trained_parameters(cls, model) -> List[torch.nn.Parameter]:
        """The tensors a step built for ``model`` now would train (``NotImplementedError`` as the constructor)."""
        return cls._analyse(model)[3]

    def bound_to_model(self) -> bool:
        """As ``_FlatStep.bound_to_model, and False as well once a parameter's ``requires_grad`` has changed since
        construction (the trained set is fixed here)."""
        return super().bound_to_model() and [p.requires_grad for u in self._units for p in u] == self._requires

    def _draws(self, a) -> bool:
        return bool(a.training and (a.drop_p > 0 or self._head_drops))

    def _args(self, batch, backward: bool, want_preds: bool):
        dev = self.dev
        y = _on(batch, "y", dev, torch.float32)
        if y.numel() % self.n_classes:
            raise ValueError(f"fragnet_b200: batch['y'] has {y.numel()} entries, not a multiple of the head's "
                             f"{self.n_classes} outputs")
        g = y.numel() // self.n_classes
        inp, tensors, (xa, xb, xfb) = self._batch_inputs(batch, g)
        pt = ops._ptr
        a = _abi.CFinetuneStepArgs()
        a.batch = inp
        a.x_atoms, a.x_bond, a.x_fbond, a.target = pt(xa), pt(xb), pt(xfb), pt(y)
        a.n_layers = self.n_layers
        a.layers = C.cast(self._layers, C.c_void_p)
        a.layer_grads = C.cast(self._layer_grads, C.c_void_p)
        a.n_head_layers, a.head = len(self._head), C.cast(self._head, C.c_void_p)
        a.loss_kind = _abi.LOSS_MSE if self.loss_kind == "mse" else _abi.LOSS_BCE_MASKED
        a.drop_p, a.training = float(self.model.pretrain.dropout.p), int(bool(self.model.training))
        a.seed, a.offset = torch.initial_seed() & 0xFFFFFFFFFFFFFFFF, 0
        a.precision, a.backward = config.precision_id(), int(backward)
        a.first_trained_layer = self.first_trained_layer
        a.variant = self._VARIANT
        loss = self._next_loss()
        a.loss = loss.data_ptr()
        preds = None
        if want_preds:
            preds = torch.empty((g, self.n_classes), dtype=torch.float32, device=dev)
            a.predictions = pt(preds)
        a.plan_arena = self._take_prefetched(a.batch)
        return a, loss, preds, tensors + (y,)


_EMPTY_GRAPH = {}


def _empty_graph(dev):
    """An empty edge list and its empty 6-wide attributes; persistent, so that the plan key of a batch is stable."""
    key = str(dev)
    if key not in _EMPTY_GRAPH:
        _EMPTY_GRAPH[key] = (torch.zeros((2, 0), dtype=torch.int64, device=dev),
                             torch.zeros((0, 6), dtype=torch.float32, device=dev))
    return _EMPTY_GRAPH[key]


class _VariantStep(FusedFineTuneStep):
    """What the gat2_lite and gat2_edge steps share: a batch without the fragment-connection graph (its features are
    never read) and, for gat2_lite, without fragment edges."""

    def _plan_inputs(self, b, g: int, convert: bool = True):
        e_idx, e_attr = _empty_graph(self.dev)
        frag_index = e_idx if self._VARIANT == _abi.VARIANT_LITE else b["frag_index"]
        return ops.batch_inputs(b["edge_index"], frag_index, b["atom_to_frag_ids"], b["edge_index_bonds_graph"],
                                b["edge_attr_bonds"], e_idx, e_attr, b["batch"], b["frag_batch"], b["x_atoms"].shape[0],
                                b["x_frags"].shape[0], b["node_features_bonds"].shape[0], frag_index.shape[1], g,
                                self.dev, convert)

    def _batch_inputs(self, batch, g: int):
        inp, keep = self._plan_inputs(batch, g)
        feats = tuple(_on(batch, k, self.dev, torch.float32) for k in ("x_atoms", "node_features_bonds"))
        return inp, keep + feats, feats + (None,)

    @staticmethod
    def _layer_units(model, extra_last=()):
        """Per encoder layer: the 14 program tensors (None where the variant has none or never reads them) and the
        freezable unit of live tensors; ``extra_last``: live tensors of the last layer that the program does not take."""
        layer_params, units = [], []
        n_layers = len(model.pretrain.layers)
        for li, layer in enumerate(model.pretrain.layers):
            top = li == n_layers - 1
            t = dict(Wb=layer.projection_b.weight, bb=layer.projection_b.bias, We_b=layer.edge_attr_bond_embed.weight,
                     be_b=layer.edge_attr_bond_embed.bias, Wa=layer.projection_a.weight, ba=layer.projection_a.bias,
                     a_b=layer.a_b, a=layer.a)
            unit = list(t.values())
            if extra_last and top:
                t["f"] = layer.f
                unit += [layer.f, *extra_last]
            layer_params.append([t.get(n) for n in _abi.PARAM_FIELDS])
            units.append(unit)
        return layer_params, units


class FusedLiteFineTuneStep(_VariantStep):
    """``FusedFineTuneStep`` for this package's ``gat2_lite.FragNetFineTune``: bond graph, atom graph and the pooled
    fragments ``ReLU(Dropout(pool(atoms)))`` of the last layer.  A layer's live tensors are ``projection_b``,
    ``edge_attr_bond_embed``, ``projection_a``, ``a_b`` and ``a``; the fragment-side tensors never get a gradient.
    Dropout counters: those of a gat2 encoder without fragment-connection nodes (``fnb_finetune_step_args``), which
    is not the layout of the autograd ``gat2_lite`` path."""

    _VARIANT = _abi.VARIANT_LITE

    @staticmethod
    def _analyse(model):
        from ..model.gat import gat2_lite
        spec = _check_model(model, gat2_lite, "FusedLiteFineTuneStep")
        return _trained_set(spec, *_VariantStep._layer_units(model))


class FusedEdgeFineTuneStep(_VariantStep):
    """``FusedFineTuneStep`` for this package's ``gat2_edge.FragNetFineTune``.  The fragment graph's edge term
    ``<cnx_attr_transform(cnx_attr[e]), f_e[h]>`` of the last layer is formed and differentiated on the device; the
    batch needs 8-wide ``cnx_attr`` (``ValueError`` otherwise, as ``Linear(8, 128)`` upstream).  Live tensors: those of
    ``FusedLiteFineTuneStep`` per layer, plus ``f`` and ``cnx_attr_transform`` in the last layer (frozen with it)."""

    _VARIANT = _abi.VARIANT_EDGE
    _EXTRA_KEYS = ("cnx_attr",)

    def __init__(self, model, *args, **kw):
        super().__init__(model, *args, **kw)
        self._cnx = model.pretrain.layers[-1].cnx_attr_transform

    @staticmethod
    def _analyse(model):
        from ..model.gat import gat2_edge
        spec = _check_model(model, gat2_edge, "FusedEdgeFineTuneStep")
        cnx = model.pretrain.layers[-1].cnx_attr_transform
        return _trained_set(spec, *_VariantStep._layer_units(model, (cnx.weight, cnx.bias)))

    def _args(self, batch, backward: bool, want_preds: bool):
        from ..model.gat.gat2_edge import CNX_IN
        cnx = _on(batch, "cnx_attr", self.dev, torch.float32)
        if cnx.dim() != 2 or cnx.shape[1] != CNX_IN or cnx.shape[0] != batch["frag_index"].shape[1]:
            raise ValueError(f"FusedEdgeFineTuneStep: cnx_attr must be [n_frag_edges, {CNX_IN}] "
                             f"(cnx_attr_transform = Linear({CNX_IN}, 128)); got {tuple(cnx.shape)}")
        a, loss, preds, keep = super()._args(batch, backward, want_preds)
        pt = ops._ptr
        a.cnx_attr, a.W_cnx, a.b_cnx = pt(cnx), pt(self._cnx.weight), pt(self._cnx.bias)
        a.dW_cnx, a.db_cnx = pt(self._grad_of.get(id(self._cnx.weight))), pt(self._grad_of.get(id(self._cnx.bias)))
        return a, loss, preds, keep + (cnx,)


def finetune_step_class(model):
    """The one-call finetuning step class for a ``FragNetFineTune`` of this package's model versions (gat2 for any
    other model, whose constructor then raises ``NotImplementedError``)."""
    from ..model.gat import gat2_edge, gat2_lite
    return {gat2_lite.FragNetFineTune: FusedLiteFineTuneStep,
            gat2_edge.FragNetFineTune: FusedEdgeFineTuneStep}.get(type(model), FusedFineTuneStep)


class LaggedScalars:
    """Every step's scalar result (the loss) read back to the host WITHOUT stalling the launch of the next step.

    The reference reads ``loss.item()`` right after ``optimizer.step()`` (pretrain_utils.py:28): the host then waits
    for the whole step and the GPU idles while the next step is being enqueued.  Here the 4-byte device-to-host copy
    of step ``i`` is queued behind step ``i`` into a pinned slot, and collected once step ``i + lag`` has been enqueued
    (``push`` returns the values that have become due, in step order; ``drain`` returns the rest)."""

    def __init__(self, lag: int = 1):
        import collections
        self.lag = max(0, int(lag))
        n = self.lag + 2
        self._host = torch.empty(n, dtype=torch.float32).pin_memory()
        self._events = [torch.cuda.Event() for _ in range(n)]
        self._ready = [torch.cuda.Event() for _ in range(n)]
        self._side: Optional[torch.cuda.Stream] = None
        self._pending = collections.deque()
        self._count = 0

    def _collect(self, keep: int) -> List[float]:
        out = []
        while len(self._pending) > keep:
            s = self._pending.popleft()
            self._events[s].synchronize()
            out.append(float(self._host[s]))
        return out

    def push(self, value: torch.Tensor) -> List[float]:
        s = self._count % len(self._events)
        self._count += 1
        # the copy runs on a side stream behind the step: in the compute stream the 4-byte DMA would sit between this
        # step's last kernel and the next step's first one (~10 us per step, gpurun_out/r5x)
        cur = torch.cuda.current_stream(value.device)
        if self._side is None:
            self._side = torch.cuda.Stream(value.device)
        src = value.detach().reshape(1)
        self._ready[s].record(cur)
        self._side.wait_event(self._ready[s])
        with torch.cuda.stream(self._side):
            self._host[s:s + 1].copy_(src, non_blocking=True)
        src.record_stream(self._side)
        self._events[s].record(self._side)
        self._pending.append(s)
        return self._collect(self.lag)

    def drain(self) -> List[float]:
        return self._collect(0)
