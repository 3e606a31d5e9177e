"""Finetuning step on the GPU: the one-call ``FusedFineTuneStep`` against ``TrainerFineTune``'s autograd loop.

Model: ``FragNetFineTune`` per exps/ft/esol/e1pt4.yaml (4 layers, FTHead3 128/1024/1024/512, dropout 0.1, ReLU) in
training mode; loss ``nn.MSELoss`` and Adam (lr 1e-4).  Batches: ESOL-shaped synthetic molecules, resident in device
memory, rotated so that the batches of one pass exceed the 126 MB of L2.  Both paths train twin copies of the same
model on the same batches; the autograd leg is the loop body of ``TrainerFineTune.train_regr`` (zero_grad,
``MSELoss(model(b).view(-1), y)``, backward, ``optimizer.step()``) with the per-batch losses summed on the device.
The legs alternate, ``--rounds`` times each.

``--variant`` picks the model versions: ``gat2`` (default), ``lite`` (``gat2_lite``) and ``edge`` (``gat2_edge``), each
with the same FTHead3 and the one-call step of its version (``FusedLiteFineTuneStep`` / ``FusedEdgeFineTuneStep``).
The edge batches' connection attributes get two random columns: ``cnx_attr_transform`` is ``Linear(8, 128)`` and the
featuriser emits 6.

``--freeze`` also times the usual finetuning set-ups with frozen parameters (``requires_grad = False``): ``lower2``
freezes encoder layers 0 and 1, ``encoder`` the whole encoder.  Both legs then train the same tensors: the autograd leg's
Adam holds the trainable ones, and the fused step stops its backward below the lowest trained layer.

Per leg and batch size: ms per step (host clock around the timed steps, ending in a device synchronise),
molecules/s, host enqueue ms per step (the same clock before the synchronise) and library launches per step
(``fnb_launch_count``).  Prints one JSON line, with the card's name and power limit read in the same run."""
from __future__ import annotations

import argparse
import copy
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

FT_KW = dict(n_classes=1, num_layer=4, drop_ratio=0.1, num_heads=4, emb_dim=128, h1=128, h2=1024, h3=1024, h4=512,
             act="relu", fthead="FTHead3")
LR = 1e-4
L2_BYTES = 126 * 2 ** 20
FREEZE = {"none": 0, "lower2": 2, "encoder": FT_KW["num_layer"]}     # encoder layers frozen from the bottom


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"] = out or None
    except OSError:
        info["power_limit"] = None
    return info


VARIANTS = ("gat2", "lite", "edge")


def model_class(variant):
    from fragnet_b200.model.gat import gat2, gat2_edge, gat2_lite
    return {"gat2": gat2, "lite": gat2_lite, "edge": gat2_edge}[variant].FragNetFineTune


def make_batches(batch, pool, seed, variant="gat2"):
    """Collated ESOL-shaped batches on the device, as many as it takes for one pass to exceed L2 (at least 4)."""
    import random

    from fragnet_b200 import synth
    from fragnet_b200.dataset.data import collate_fn
    mols = synth.make_dataset("esol", pool, seed=seed, with_pretrain_targets=False)
    rng = random.Random(seed)
    out, total = [], 0
    while len(out) < 4 or total < 2 * L2_BYTES:
        b = collate_fn([mols[rng.randrange(len(mols))] for _ in range(batch)])
        gen = torch.Generator().manual_seed(seed + len(out))
        b["y"] = torch.randn(b["y"].shape, generator=gen)
        if variant == "edge":
            b["cnx_attr"] = torch.cat((b["cnx_attr"], torch.rand(b["cnx_attr"].shape[0], 2, generator=gen)), dim=1)
        b = {k: v.cuda() for k, v in b.items()}
        out.append(b)
        total += sum(v.numel() * v.element_size() for v in b.values())
    return out, total


def timed(run, steps, warmup):
    """``run(i) -> loss`` for step i; returns (ms/step, host enqueue ms/step, library launches/step)."""
    from fragnet_b200 import ops
    lib = ops._lib()
    for i in range(warmup):
        run(i)
    torch.cuda.synchronize()
    n0 = lib.fnb_launch_count()
    t0 = time.perf_counter()
    total = torch.zeros((), dtype=torch.float64, device="cuda")
    for i in range(steps):
        total += run(warmup + i).detach().double()
    t1 = time.perf_counter()
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    loss = float(total) / steps
    if loss != loss:
        raise RuntimeError("non-finite loss")
    return (t2 - t0) * 1e3 / steps, (t1 - t0) * 1e3 / steps, (lib.fnb_launch_count() - n0) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="128,1024", help="molecules per step, comma separated")
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=2, help="alternations of the two legs per batch size")
    ap.add_argument("--pool", type=int, default=1128, help="distinct synthetic molecules (ESOL has 1 128)")
    ap.add_argument("--freeze", default="none", help=f"comma separated, of {', '.join(FREEZE)}")
    ap.add_argument("--variant", default="gat2", help=f"comma separated, of {', '.join(VARIANTS)}")
    args = ap.parse_args()
    modes = args.freeze.split(",")
    if any(m not in FREEZE for m in modes):
        raise SystemExit(f"--freeze: expected names from {sorted(FREEZE)}, got {args.freeze!r}")
    variants = args.variant.split(",")
    if any(v not in VARIANTS for v in variants):
        raise SystemExit(f"--variant: expected names from {list(VARIANTS)}, got {args.variant!r}")
    if not torch.cuda.is_available():
        raise SystemExit("finetune_bench.py needs a CUDA device")
    from fragnet_b200.train.fused import finetune_step_class
    result = {"workload": "FragNetFineTune exps/ft/esol/e1pt4.yaml training step (fwd + MSE + bwd + Adam), "
                          "ESOL-shaped synthetic batches resident in HBM", "card": card(), "steps": args.steps,
              "warmup": args.warmup, "rounds": args.rounds, "legs": {}}
    for variant, batch, mode in ((v, int(x), m) for v in variants for x in args.batches.split(",") for m in modes):
        batches, nbytes = make_batches(batch, args.pool, seed=7, variant=variant)
        torch.manual_seed(0)
        kw = dict(FT_KW, edge_features=batches[0]["node_features_bonds"].shape[1])
        m_fused = model_class(variant)(**kw).cuda().train()
        for layer in m_fused.pretrain.layers[:FREEZE[mode]]:
            for p in layer.parameters():
                p.requires_grad_(False)
        m_auto = copy.deepcopy(m_fused)
        fused = finetune_step_class(m_fused)(m_fused, lr=LR)
        opt = torch.optim.Adam([p for p in m_auto.parameters() if p.requires_grad], lr=LR)
        loss_fn = torch.nn.MSELoss()
        nb = len(batches)

        def run_fused(i):
            return fused.step(batches[i % nb], next_batch=batches[(i + 1) % nb])

        def run_auto(i):
            b = batches[i % nb]
            opt.zero_grad()
            loss = loss_fn(m_auto(b).view(-1), b["y"])
            loss.backward()
            opt.step()
            return loss

        legs = {"fused": [], "autograd": []}
        for _ in range(args.rounds):
            legs["fused"].append(timed(run_fused, args.steps, args.warmup))
            legs["autograd"].append(timed(run_auto, args.steps, args.warmup))
        out = {"rotated_batches": nb, "rotated_bytes": nbytes}
        for name, runs in legs.items():
            ms, enq, launches = min(runs)
            out[name] = {"ms_per_step": round(ms, 3), "molecules_per_s": round(batch / ms * 1e3, 1),
                         "host_enqueue_ms_per_step": round(enq, 3), "fnb_launches_per_step": round(launches, 1),
                         "ms_per_step_all_rounds": [round(r[0], 3) for r in runs]}
        out["speedup"] = round(out["autograd"]["ms_per_step"] / out["fused"]["ms_per_step"], 2)
        prefix = "" if variant == "gat2" else f"{variant}_"
        result["legs"][f"{prefix}batch_{batch}" + ("" if mode == "none" else f"_freeze_{mode}")] = out
        del batches, fused, m_fused, m_auto, opt
        torch.cuda.empty_cache()
    result["card_after"] = card()
    print(json.dumps(result))


if __name__ == "__main__":
    main()
