"""Finetuning loops with the reference's semantics: drop-ins for ``EarlyStopping`` (fragnet/train/utils.py:13-56),
``test_fn`` (:59-76) and ``TrainerFineTune`` (:307-520; ``target_type`` ``regr`` and ``clsf``), the callers of the GAT2
path in train/finetune/finetune_gat2.py:119-288.

Same signatures, same returned quantities (epoch loss = sum of the per-batch losses / dataset size; ``test`` returns
``(mse, targets, predictions)`` resp. ``(roc_auc, targets, predictions)``).  What differs underneath: host batches are
staged by ``DevicePrefetcher`` (pinned, double-buffered copies on a side stream, only the tensors the model reads)
instead of 16 blocking ``batch[k].to(device)`` calls per step (utils.py:335-336), and the per-batch losses are summed
on the device and read back once per epoch instead of one ``loss.item()`` synchronisation per step (utils.py:344).

``TrainerFineTune(..., fused=True)`` runs each training batch of this package's ``FragNetFineTune`` (gat2, gat2_lite or
gat2_edge) as one library call (``FusedFineTuneStep`` and its ``FusedLiteFineTuneStep`` / ``FusedEdgeFineTuneStep``:
collate, encoder, readout, head, loss, backward, then Adam over flat buffers) when the
optimizer is a plain ``torch.optim.Adam`` holding every trained tensor in its one parameter group and the model is one
the library covers, frozen parameters included (the lower encoder layers or the whole encoder, any head linear);
anything else silently takes the generic loop below.  A model wrapped in ``DistributedDataParallel`` trains
data-parallel over the wrapper's process group (the step's ``group``; DDP semantics, collective construction); an
un-wrapped model under an initialised process group keeps the generic loop.  A change of ``requires_grad`` between
epochs (unfreezing the encoder after a warm-up) rebuilds the fused step, on every rank in the same epoch.  Validation
and test always call ``model(batch)``, through the wrapper if there is one.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn as nn


class EarlyStopping:
    """Stops when the validation loss has not improved by ``delta`` for ``patience`` epochs; checkpoints the best
    ``state_dict`` to ``chkpoint_name`` (utils.py:13-56)."""

    def __init__(self, patience=7, verbose=False, delta=0, chkpoint_name="gnn_best.pt"):
        self.patience, self.verbose, self.delta, self.chkpoint_name = patience, verbose, delta, chkpoint_name
        self.counter, self.best_score, self.early_stop, self.val_loss_min = 0, None, False, np.inf

    def __call__(self, val_loss, model):
        score = -val_loss
        improved = self.best_score is None or score >= self.best_score + self.delta
        if improved:
            self.best_score, self.counter = score, 0
            self.save_checkpoint(val_loss, model)
            return
        self.counter += 1
        print(f"EarlyStopping counter: {self.counter} out of {self.patience}")
        self.early_stop = self.counter >= self.patience

    def save_checkpoint(self, val_loss, model):
        if self.verbose:
            print(f"Validation loss decreased ({self.val_loss_min:.6f} --> {val_loss:.6f}).  Saving model ...")
        torch.save(model.state_dict(), self.chkpoint_name)
        self.val_loss_min = val_loss


def _extra_keys(model):
    """Batch entries a model of this package reads beyond the GAT2 hot path: gat2_edge reads ``cnx_attr``."""
    from ..model.gat import gat2_edge
    return ("cnx_attr",) if isinstance(model, (gat2_edge.FragNetFineTune, gat2_edge.FragNet)) else ()


def _batches(loader, device, model=None):
    """Device-resident batch dicts of ``loader``: prefetched for CUDA devices, moved key by key otherwise.  For this
    package's own models only the tensors their path reads are moved."""
    device = torch.device(device)
    if device.type == "cuda":
        from ..dataset.prefetch import DevicePrefetcher
        ours = model is not None and type(model).__module__.startswith("fragnet_b200.")
        keep = _extra_keys(model) if ours else ()
        yield from DevicePrefetcher(loader, device, depth=2, hot_path_only=ours, keep=keep)
    else:
        for batch in loader:
            yield {k: v.to(device) for k, v in batch.items()}


def compute_bce_loss(prediction, target):
    """Masked BCE-with-logits: labels < -0.5 are missing (utils.py:296-303)."""
    is_valid = target > -0.5
    loss_mat = nn.BCEWithLogitsLoss(reduction="none")(prediction, target)
    loss_mat = torch.where(is_valid, loss_mat, torch.zeros_like(loss_mat))
    return torch.sum(loss_mat) / torch.sum(is_valid)


def test_fn(loader, model, device):
    """utils.py:59-76: ``(mse, targets, predictions)`` over a loader."""
    model.eval()
    target, predicted = [], []
    with torch.no_grad():
        for batch in _batches(loader, device, model):
            predicted.append(model(batch).reshape(-1))
            target.append(batch["y"].reshape(-1))
    t = torch.cat(target).cpu().numpy() if target else np.zeros(0, dtype=np.float32)
    p = torch.cat(predicted).cpu().numpy() if predicted else np.zeros(0, dtype=np.float32)
    return float(np.mean((t - p) ** 2)) if t.size else float("nan"), t, p


test_fn.__test__ = False      # not a pytest test


class TrainerFineTune:
    """utils.py:307-520 for ``target_type`` ``regr`` (MSE) and ``clsf`` (masked BCE, ROC-AUC validation)."""

    def __init__(self, target_pos=None, target_type="regr", n_multi_task_heads=0, fused: bool = False):
        self.target_pos = target_pos
        self.n_multi_task_heads = n_multi_task_heads
        self.fused = fused
        # [(weakref(model), weakref(optimizer), FusedFineTuneStep | None, requires_grad of the model's parameters)]
        self._fused_steps = []
        if target_type == "regr":
            self.train, self.validate, self.test = self.train_regr, self.validate_regr, self.test_regr
            self.loss_fn = nn.MSELoss()
        elif target_type == "clsf":
            self.train, self.validate, self.test = self.train_clsf_bce, self.validate_clsf_bce, self.test_clsf_bce
            self.loss_fn = nn.BCEWithLogitsLoss(reduction="none")
        else:
            raise NotImplementedError(f"target_type {target_type!r}: only 'regr' and 'clsf' drive the gat2 path here")

    # ---- one pass over a loader: per-batch losses summed on the device, read back once
    def _epoch(self, model, loader, device, loss_of, optimizer=None):
        total = torch.zeros((), dtype=torch.float64, device=device)
        for batch in _batches(loader, device, model):
            if optimizer is not None:
                optimizer.zero_grad()
            loss = loss_of(batch)
            if optimizer is not None:
                loss.backward()
                optimizer.step()
            total += loss.detach().double()
        return float(total) / len(loader.dataset)

    # ---- fused path (fused=True): one library call per training batch
    def _fused_for(self, model, optimizer, device, loss):
        """The ``FusedFineTuneStep`` bound to (model, optimizer), or None when the fused path does not apply.  ``model``
        may be a ``DistributedDataParallel`` wrapper: the step is built for its module over its process group, and
        cached under the wrapper."""
        if not self.fused or torch.device(device).type != "cuda" or optimizer is None:
            return None
        from .pretrain_utils import _plain_adam
        if loss == "mse":
            ok = type(self.loss_fn) is nn.MSELoss and self.loss_fn.reduction == "mean"
        else:
            ok = type(self.loss_fn) is nn.BCEWithLogitsLoss and self.loss_fn.reduction == "none" and \
                self.loss_fn.weight is None and self.loss_fn.pos_weight is None
        p0 = next(model.parameters(), None)
        if not (ok and _plain_adam(optimizer) and torch.is_tensor(p0) and p0.is_cuda):
            return None
        import weakref
        frozen = tuple(p.requires_grad for p in model.parameters())
        # a step is built for one set of trained tensors: after a requires_grad change it is rebuilt
        self._fused_steps = [e for e in self._fused_steps if e[0]() is not None and e[1]() is not None and
                             not (e[0]() is model and e[1]() is optimizer and e[3] != frozen)]
        g = optimizer.param_groups[0]
        owned = {id(p) for p in g["params"]}
        for wm, wo, fs, _ in self._fused_steps:
            if wm() is model and wo() is optimizer:
                ok = fs is not None and fs.bound_to_model() and all(id(p) in owned for p in fs.live)
                return fs if ok else None
        from torch.nn.parallel import DistributedDataParallel
        from .fused import finetune_step_class
        inner, group = (model.module, model.process_group) if isinstance(model, DistributedDataParallel) else (model, None)
        step_class = finetune_step_class(inner)
        fs = None
        try:
            # every trained tensor must be the optimizer's: the generic loop's Adam updates nothing else (frozen or
            # gradient-less tensors in the optimizer are skipped by both paths)
            if all(id(p) in owned for p in step_class.trained_parameters(inner)):
                fs = step_class(inner, lr=g["lr"], betas=g["betas"], eps=g["eps"], weight_decay=g["weight_decay"],
                                loss=loss, group=group)
                fs.attach_optimizer(optimizer)      # optimizer.state_dict() keeps checkpointing the real moments
        except NotImplementedError:
            fs = None
        self._fused_steps.append((weakref.ref(model), weakref.ref(optimizer), fs, frozen))
        return fs

    @staticmethod
    def _fused_epoch(fs, loader, device, optimizer):
        """One training epoch through ``fs``; the next batch's collate is queued underneath every step."""
        from ..dataset.prefetch import DevicePrefetcher
        staged = DevicePrefetcher(loader, device, depth=2, hot_path_only=True, keep=fs._EXTRA_KEYS)
        feed = iter(staged)
        total = torch.zeros((), dtype=torch.float64, device=device)
        batch = next(feed, None)
        while batch is not None:
            g = optimizer.param_groups[0]            # LR schedulers / edited hyper-parameters are honoured per step
            fs.lr, fs.betas, fs.eps, fs.weight_decay = float(g["lr"]), g["betas"], float(g["eps"]), float(g["weight_decay"])
            loss = fs.step(batch)
            batch = next(feed, None)
            if batch is not None:
                fs.prefetch_plan(batch, staged.last_event)
            total += loss.double()
        return float(total) / len(loader.dataset)

    # ---- regression (utils.py:330-385)
    def train_regr(self, model, loader, optimizer, scheduler, device, val_loader):
        model.train()
        fs = self._fused_for(model, optimizer, device, "mse")
        if fs is not None:
            mean = self._fused_epoch(fs, loader, device, optimizer)
        else:
            mean = self._epoch(model, loader, device, lambda b: self.loss_fn(model(b).view(-1), b["y"]), optimizer)
        if scheduler:
            self.validate(model, val_loader, device)
            scheduler.step()
        return mean

    def validate_regr(self, model, loader, device):
        model.eval()
        with torch.no_grad():
            return self._epoch(model, loader, device, lambda b: self.loss_fn(model(b).view(-1), b["y"]))

    def test_regr(self, model, loader, device):
        return test_fn(loader, model, device)

    # ---- binary / multi-label classification with missing labels (utils.py:406-470)
    def _bce(self, out, y):
        labels = y.view(out.shape)
        is_valid = labels > -0.5
        loss_mat = torch.where(is_valid, self.loss_fn(out, labels), torch.zeros_like(out))
        return torch.sum(loss_mat) / torch.sum(is_valid)

    def train_clsf_bce(self, model, loader, optimizer, scheduler, device, val_loader):
        model.train()
        fs = self._fused_for(model, optimizer, device, "bce")
        if fs is not None:
            mean = self._fused_epoch(fs, loader, device, optimizer)
        else:
            mean = self._epoch(model, loader, device, lambda b: self._bce(model(b), b["y"]), optimizer)
        if scheduler:
            scheduler.step(self.validate(model, val_loader, device))
        return mean

    def _scores(self, model, loader, device):
        """Targets and RAW model outputs (logits) of a loader, as the reference collects them (utils.py:466-476,
        :519-531: ``predicted.append(pred)`` with ``pred = model(batch)``; ROC-AUC is rank based, so no sigmoid)."""
        model.eval()
        target, predicted = [], []
        with torch.no_grad():
            for batch in _batches(loader, device, model):
                out = model(batch)
                predicted.append(out)
                target.append(batch["y"].view(out.shape))
        return torch.cat(target).cpu().numpy(), torch.cat(predicted).cpu().numpy()

    @staticmethod
    def _neg_mean_auc(target, predicted):
        """-mean ROC-AUC over the label columns that hold at least one 1 and one 0 (utils.py:477-486, :532-542).
        NEGATIVE because the callers minimise it (``early_stopping(val_loss, model)``, finetune_gat2.py:268-274)."""
        from sklearn.metrics import roc_auc_score
        rocs = []
        for c in range(target.shape[1]):
            if np.sum(target[:, c] == 1) > 0 and np.sum(target[:, c] == 0) > 0:
                valid = target[:, c] > -0.5
                rocs.append(roc_auc_score(target[valid, c], predicted[valid, c]))
        return -(sum(rocs) / len(rocs))      # ZeroDivisionError without a scorable column, as upstream

    def validate_clsf_bce(self, model, loader, device):
        return self._neg_mean_auc(*self._scores(model, loader, device))

    def test_clsf_bce(self, model, loader, device):
        """Returns ``(-roc_auc, targets, raw outputs)`` exactly as the reference (utils.py:519-544)."""
        target, predicted = self._scores(model, loader, device)
        return self._neg_mean_auc(target, predicted), target, predicted
