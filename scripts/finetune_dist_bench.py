#!/usr/bin/env python
"""Data-parallel finetuning step on N GPUs: ``FusedFineTuneStep(group=...)`` against the DDP autograd loop.  Launch with
torchrun, one process per GPU::

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29512 \\
        scripts/finetune_dist_bench.py

Model and batches as ``scripts/finetune_bench.py`` (gat2 ``FragNetFineTune`` of exps/ft/esol/e1pt4.yaml, ESOL-shaped
synthetic batches resident in HBM, different batches on every rank, Adam lr 1e-4).  Legs, per batch size (molecules
per rank):

- ``fused``: ``FusedFineTuneStep(model, group=WORLD)``: one library call for the step, then the gradient exchange and
  Adam (``fnb_allreduce_adam_runs`` over NVLink peer memory on NCCL, one kernel);
- ``ddp``: ``DistributedDataParallel(model, find_unused_parameters=True)`` (87 parameters never get a gradient) with
  the loop body of ``TrainerFineTune.train_regr`` and ``torch.optim.Adam``, i.e. what Fabric DDP runs.

The legs alternate ``--rounds`` times; ms per step is the slowest rank's (host clock around the timed steps, ending in
a device synchronise).  A separate ``torch.profiler`` run of the fused leg gives the exchange kernel's device time per
step on rank 0; it includes the wait for the slowest rank at the kernel's entry barrier.  ``exchange_bytes_per_rank``
is what the kernel reads per rank and step (every rank's whole gradient buffer).  The card's name and power limit are
read in the same run.  Rank 0 merges its result into ``--out`` under the world size."""
from __future__ import annotations

import argparse
import copy
import json
import os
import sys
import time

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from finetune_bench import FT_KW, LR, card, make_batches  # noqa: E402


def timed(run, steps, warmup):
    """ms per step of ``run(i)`` on the slowest rank."""
    for i in range(warmup):
        run(i)
    torch.cuda.synchronize()
    dist.barrier()
    t0 = time.perf_counter()
    total = torch.zeros((), dtype=torch.float64, device="cuda")
    for i in range(steps):
        total += run(warmup + i).detach().double()
    torch.cuda.synchronize()
    ms = torch.tensor([(time.perf_counter() - t0) * 1e3 / steps], device="cuda")
    if not torch.isfinite(total):
        raise RuntimeError("non-finite loss")
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms)


def exchange_us_per_step(run, steps, rank, out_dir):
    """Device time per step of the exchange kernel (``k_allreduce_adam_runs``) on rank 0, from a profiler run."""
    from torch.profiler import ProfilerActivity, profile
    for i in range(3):
        run(i)
    torch.cuda.synchronize()
    dist.barrier()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(steps):
            run(i)
        torch.cuda.synchronize()
    dist.barrier()
    if rank != 0:
        return None
    us = sum(e.device_time_total for e in prof.key_averages() if "allreduce_adam" in e.key)
    total = sum(e.device_time_total for e in prof.key_averages() if e.device_time_total > 0 and not e.is_user_annotation)
    if out_dir:
        prof.export_chrome_trace(os.path.join(out_dir, f"finetune_dist_trace_w{dist.get_world_size()}.json"))
    return {"exchange_us_per_step": round(us / steps, 2), "device_us_per_step_all_kernels": round(total / steps, 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="128,1024", help="molecules per step and rank, comma separated")
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--pool", type=int, default=1128)
    ap.add_argument("--profile-steps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r9_finetune_dist_bench.json"))
    ap.add_argument("--trace-dir", default="", help="where to write the profiler traces (none by default)")
    args = ap.parse_args()
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    from torch.nn.parallel import DistributedDataParallel as DDP
    from fragnet.model.gat.gat2 import FragNetFineTune
    from fragnet_b200.train.fused import FusedFineTuneStep
    result = {"world": world, "card": card(), "steps": args.steps, "warmup": args.warmup, "rounds": args.rounds,
              "legs": {}}
    for batch in (int(x) for x in args.batches.split(",")):
        batches, _ = make_batches(batch, args.pool, seed=7 + 101 * rank)
        torch.manual_seed(0)
        kw = dict(FT_KW, edge_features=batches[0]["node_features_bonds"].shape[1])
        m_fused = FragNetFineTune(**kw).cuda().train()
        m_ddp = copy.deepcopy(m_fused)
        fused = FusedFineTuneStep(m_fused, lr=LR, group=dist.group.WORLD)
        ddp = DDP(m_ddp, device_ids=[local], find_unused_parameters=True)
        opt = torch.optim.Adam(ddp.parameters(), lr=LR)
        loss_fn = torch.nn.MSELoss()
        nb = len(batches)

        def run_fused(i):
            return fused.step(batches[i % nb], next_batch=batches[(i + 1) % nb])

        def run_ddp(i):
            b = batches[i % nb]
            opt.zero_grad()
            loss = loss_fn(ddp(b).view(-1), b["y"])
            loss.backward()
            opt.step()
            return loss

        legs = {"fused": [], "ddp": []}
        for _ in range(args.rounds):
            legs["fused"].append(timed(run_fused, args.steps, args.warmup))
            legs["ddp"].append(timed(run_ddp, args.steps, args.warmup))
        out = {name: {"ms_per_step": round(min(v), 3), "ms_per_step_all_rounds": [round(x, 3) for x in v],
                      "molecules_per_s_all_ranks": round(world * batch / min(v) * 1e3, 1)} for name, v in legs.items()}
        out["speedup"] = round(out["ddp"]["ms_per_step"] / out["fused"]["ms_per_step"], 2)
        out["fused_exchange"] = "fnb_allreduce_adam_runs" if fused._peers is not None else (
            "none (one rank)" if world == 1 else "dist.all_reduce + fnb_adam_step")
        out["gradient_bytes"] = fused.flat_g.numel() * 4
        out["exchange_bytes_per_rank"] = world * fused.flat_g.numel() * 4 if fused._peers is not None else 0
        prof = exchange_us_per_step(run_fused, args.profile_steps, rank, args.trace_dir)
        if prof is not None:
            out.update(prof)
            out["exchange_share_of_step"] = round(prof["exchange_us_per_step"] / 1e3 / out["fused"]["ms_per_step"], 4)
        result["legs"][f"batch_{batch}"] = out
        del batches, fused, ddp, m_fused, m_ddp, opt
        torch.cuda.empty_cache()
    result["card_after"] = card()
    if rank == 0:
        print(json.dumps(result))
        merged = {}
        if os.path.isfile(args.out):
            with open(args.out) as f:
                merged = json.load(f)
        merged[f"world_{world}"] = result
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(merged, f, indent=1)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
