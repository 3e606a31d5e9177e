#!/usr/bin/env python
"""Benchmark of the FragNet GAT2 hot path (BASELINE.json: molecules/s, fwd+bwd GAT2 message passing).

Workload (``config.workload``, BASELINE configs[1] at the per-GPU batch of configs[3]): the reference's pretraining step
-- ``FragNetPreTrain`` per ``exps/pt/unimol_exp1s4/config.yaml`` (4 layers, 4 heads, emb 128, drop 0.2, Adam lr 1e-4,
loss of ``train/pretrain/pretrain_utils.py``) on UniMol-shaped synthetic molecules, per-GPU batch ``--batch`` (1024;
weak scaling).  A step = on-device collate + forward + loss + backward + gradient all-reduce (N > 1) + Adam on one batch;
``--rotate`` distinct pre-collated batches are cycled so the working set exceeds the 126 MB L2.

``value`` is measured in the ``fp32`` precision mode -- the mode whose outputs are within 1e-5 of the reference (dense
projections on tcgen05 tensor cores with the 3xTF32 split); ``value_tf32`` is the same step with single-TF32 products
(stated tolerance 2e-3).  The JSON line also carries, from the same run: ``e2e`` (host batches in, loss out),
``e2e_arena`` (molecule ids in), ``roofline`` (whole step + the four dominant kernels timed cold), ``cpu_baseline`` (the
reference on the host cores) and ``extra`` (BASELINE configs[0], [2], [4]: ESOL finetuning on the CPU arm, inference
screening at batch 4096, skewed-degree stress at batch 1024).

  python bench.py --gpus N --steps K --warmup W             (torchrun launches N ranks for N > 1)
  python bench.py ... --dump-outputs DIR                    also write the last timed step's results as DIR/*.npy
  python bench.py --impl reference ...                      the reference itself on the host cores, same metric
"""
from __future__ import annotations

import argparse
import contextlib
import io
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

PT_KW = dict(num_layer=4, drop_ratio=0.2, num_heads=4, emb_dim=128, atom_features=167, frag_features=167,
             edge_features=17, fedge_in=6, fbond_edge_in=6)
FT_KW = dict(n_classes=1, num_layer=4, drop_ratio=0.1, num_heads=4, emb_dim=128, h1=128, h2=1024, h3=1024, h4=512,
             act="relu", fthead="FTHead3")          # exps/ft/esol/e1pt4.yaml: finetune.model
LR = 1e-4
METRIC = "molecules/s fwd+bwd GAT2 msg-passing (FragNetPreTrain step)"
D, H = 128, 4


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=1024, help="molecules per GPU per step")
    ap.add_argument("--shape", default="unimol", choices=["esol", "unimol", "stress"])
    ap.add_argument("--rotate", type=int, default=4, help="distinct batches cycled through")
    ap.add_argument("--pool", type=int, default=512, help="distinct synthetic molecules generated")
    ap.add_argument("--precision", default="fp32", choices=["fp32", "tf32", "fp32_simt"],
                    help="arithmetic of the dense projections for `value` (everything else is fp32)")
    ap.add_argument("--autograd", action="store_true",
                    help="drive the step through nn.Module / autograd / FlatAdam instead of the one-call fused step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the configs[0]/[2]/[4] legs")
    ap.add_argument("--pack", action="store_true",
                    help="host batches packed into one pinned buffer (one copy per batch; measured no faster: r5x)")
    ap.add_argument("--no-arena", action="store_true", help="skip the arena-fed leg")
    ap.add_argument("--no-plan-prefetch", action="store_true",
                    help="collate every batch at the head of its own step instead of underneath the previous one")
    ap.add_argument("--no-tf32", action="store_true", help="skip the second timed region (value_tf32)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps of `value`, write what their last step returned to its caller (loss, "
                         "updated parameters, their gradients) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs is supported for --impl ours only")
    return args


def make_batches(shape, batch, rotate, pool, seed, pretrain=True):
    """``rotate`` collated batches of ``batch`` molecules drawn (with replacement) from a pool of distinct
    synthetic molecules; deterministic per seed."""
    import random

    from fragnet_b200 import synth
    from fragnet_b200.dataset.data import collate_fn, collate_fn_pt
    mols = synth.make_dataset(shape, min(pool, batch * rotate), seed=seed, with_pretrain_targets=pretrain)
    rng = random.Random(seed)
    col = collate_fn_pt if pretrain else collate_fn
    return [col([mols[rng.randrange(len(mols))] for _ in range(batch)]) for _ in range(rotate)]


def batch_counts(b):
    return dict(G=int(b["y"].shape[0]), Na=b["x_atoms"].shape[0], Ea=b["edge_index"].shape[1],
                Eb=b["edge_index_bonds_graph"].shape[1], Nf=b["x_frags"].shape[0], Ef=b["frag_index"].shape[1],
                Efb=b["edge_index_fbonds"].shape[1])


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (every 20 ms)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "20"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
            time.sleep(0.15)            # nvidia-smi needs a moment before its first sample
            self.rows.clear()           # samples from before the timed region do not count
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.03)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
# Algorithmic bytes (SURVEY.md section 8d: compulsory traffic, every operand counted once per kernel, fp32 = 4 B,
# int32 indices).  ``step_bytes`` is the contract's whole-step figure on the actual counts of a batch.
def att_fwd_bytes(N, E, X, train=True):
    return 2 * N * D * 4 + X + E * 4 + (N + 1) * 4 + (E * H * 4 if train else 0)


def att_bwd_bytes(N, E, X, dX):
    return 3 * N * D * 4 + E * H * 4 + 3 * E * 4 + 2 * (N + 1) * 4 + dX


def step_bytes(c, n_layers=4, K0=(17, 167, 6), live_only=False):
    """(fwd, fwd+bwd) bytes of the encoder for one batch with counts ``c`` (batch_counts).  ``live_only`` drops the
    fragment-graph block and the pooling of the layers whose fragment output is overwritten unread (gat2.py:234; the
    reference executes them, this library does not): the contract figure keeps them."""
    Na, Ea, Eb, Nf, Ef, Efb, G = c["Na"], c["Ea"], c["Eb"], c["Nf"], c["Ef"], c["Efb"], c["G"]
    Nb, Nfb = Ea, Ef
    fwd = bwd = 0
    for l in range(n_layers):
        Kb, Ka, Kfb = K0 if l == 0 else (D, D, D)
        gemm = (Nb * Kb + Nb * D + Na * Ka + Na * D + Nfb * Kfb + Nfb * D) * 4
        blocks = [(Nb, Eb, Eb * 4, 0), (Na, Ea + Na, Ea * D * 4, Ea * D * 4), (Nfb, Efb, Efb * 24, 0)]
        pool_f, pool_b = (Na + Nf) * D * 4 + Na * 4, (Na + Nf) * D * 4
        if not live_only or l == n_layers - 1:
            blocks.append((Nf, Ef, Ef * D * 4, Ef * D * 4))
        else:
            pool_f = pool_b = 0
        fwd += gemm + pool_f + sum(att_fwd_bytes(N, E, X) for N, E, X, _ in blocks)
        bwd += 2 * gemm + pool_b + sum(att_bwd_bytes(N, E, X, dX) for N, E, X, dX in blocks)
    readout = (Na + Nf) * D * 4 + 2 * G * D * 4
    return fwd + readout, fwd + bwd + 2 * readout


def _cold_time(launch, sets, iters):
    """Average microseconds per launch over back-to-back launches that cycle ``sets`` operand sets (no launch finds its
    operands in L2), CUDA events on the launch stream."""
    for i in range(sets):
        launch(i)
    times = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
        e0.record()
        for i in range(sets):
            launch(i)
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1) / sets * 1e3)
    return statistics.mean(times)


# Share of the summed kernel time of one fp32-mode step per kernel, and the DRAM traffic of one captured launch of each:
# both come from the committed profiles of this state (scripts/summarize_launches.py, scripts/summarize_ncu_full.py
# write profiles/r5_kernel_shares.json next to the markdown tables they are taken from).
KERNEL_SHARE = {"source": "profiles/r5_launch_list.md"}
NCU_TRAFFIC = {"source": "profiles/r5_ncu_full.md", "per_kernel": {}}
try:
    _p = os.path.join(ROOT, "profiles", "r5_kernel_shares.json")
    if os.path.isfile(_p):
        _d = json.load(open(_p))
        KERNEL_SHARE.update(_d.get("share", {}))
        NCU_TRAFFIC["per_kernel"] = _d.get("traffic", {})
except (OSError, ValueError):
    pass


def roofline_kernels(batch_dev, peaks, iters=6, sets=8):
    """Live, cold timings of the four dominant kernels on the bond graph of the bench batch (the bond graph is ~60 % of
    the gathered rows of a step): attention forward in its training configuration, destination pass and source pass of
    its backward (timed separately through an event recorded between the two launches), and the 3xTF32 projection."""
    from fragnet_b200 import ops
    b = batch_dev
    dev = b["x_atoms"].device
    Nb, Eb = b["node_features_bonds"].shape[0], b["edge_index_bonds_graph"].shape[1]
    eb = b["edge_index_bonds_graph"]
    g = ops.csr_build(eb[0].contiguous(), eb[1].contiguous(), Nb)
    g.attr = ops.gather_rows(b["edge_attr_bonds"].reshape(-1, 1), g.eid, Eb)
    alpha = torch.randn(4, 96, device=dev) * 0.1
    nxt = torch.randn(4, 192, device=dev) * 0.1
    We, be = torch.randn(32, 1, device=dev), torch.randn(32, device=dev)
    W, bias = torch.randn(128, 128, device=dev) * 0.1, torch.randn(128, device=dev)
    hs = [torch.randn(Nb, 128, device=dev) for _ in range(sets)]
    gos = [torch.randn(Nb, 128, device=dev) for _ in range(sets)]
    Ss = [ops.node_scalars(h, alpha, 96, 0, 64) for h in hs]
    peak = peaks.get("hbm_gbs")
    out = []

    def entry(name, us, nbytes, note, launches):
        gbs = nbytes / us / 1e3
        e = {"kernel": name, "us_per_launch": round(us, 2), "bytes_per_launch": int(nbytes), "achieved": round(gbs, 1),
             "frac": round(gbs / peak, 4) if peak else None, "launches_per_step": launches,
             "share_of_kernel_time": KERNEL_SHARE.get(name), "bytes_model": note,
             "traffic": NCU_TRAFFIC["per_kernel"].get(name)}
        out.append(e)
        return e

    # --- forward, training configuration (pre + post activation rows, saved p, consumer edge term)
    def fwd(i):
        return ops.gat_fwd_tiled(g, hs[i], Ss[i], ops.EDGE_AFFINE1, We=We, be=be, alpha_e=alpha[:, 32:], alpha_stride=96,
                                 post=(0.2, 1, 1, 1234, 0), next_alpha=nxt[:, 32:], next_alpha_stride=192)
    us = _cold_time(fwd, sets, iters)
    contract = att_fwd_bytes(Nb, Eb, Eb * 4)
    fused = Nb * 128 * 4 + Nb * 32 + (Nb + 1) * 4 + 3 * Eb * 4 + 2 * Nb * 128 * 4 + Eb * 16 + Nb * 16
    e = entry("k_gat_fwd_tiled<AFFINE1>", us, fused,
              "reads h, S, rowptr, col, row, cos; writes pre- and post-activation rows, p, consumer edge term "
              "(section 8d B_att_fwd + the fused epilogue outputs)", 4)
    e["bytes_contract"] = int(contract)
    e["frac_contract"] = round(contract / us / 1e3 / peak, 4) if peak else None

    # --- backward: destination pass | source pass
    ps = [fwd(i)[2] for i in range(sets)]
    d_alpha = torch.zeros(4, 96, device=dev)
    bufs = [(torch.empty(Eb, 4, device=dev), torch.empty(Nb, 4, device=dev), torch.empty(Nb, 128, device=dev))
            for _ in range(sets)]
    mark = torch.cuda.Event(enable_timing=True)
    mark.record()

    def bwd(i, ev=None):
        ops.gat_bwd_tiled(g, hs[i], gos[i], ps[i], ops.EDGE_AFFINE1, alpha, 96, 0, 32, 64, d_alpha, We=We, be=be,
                          want_bias_grad=True, mark=ev, out=bufs[i])
    for i in range(sets):
        bwd(i)
    t_dst, t_src = [], []
    for _ in range(iters):
        for i in range(sets):
            e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
            e0.record()
            bwd(i, mark)
            e1.record()
            e1.synchronize()
            t_dst.append(e0.elapsed_time(mark) * 1e3)
            t_src.append(mark.elapsed_time(e1) * 1e3)
    dst_b = 2 * Nb * D * 4 + 2 * Eb * H * 4 + Eb * 4 + (Nb + 1) * 4 + Nb * H * 4
    src_b = 3 * Nb * D * 4 + 2 * Eb * H * 4 + 2 * Eb * 4 + (Nb + 1) * 4 + Nb * H * 4
    entry("k_gat_bwd_dst_tiled<AFFINE1>", statistics.mean(t_dst), dst_b,
          "reads h, g, p, rowptr, col; writes dz, dSt (in the step the FUSE variant also assembles g)", 4)
    entry("k_gat_bwd_src_tiled", statistics.mean(t_src), src_b,
          "reads g, own h row, p, dz, dSt, reverse CSR; writes dh (13 launches per step over the four graphs; this "
          "is the bond graph's)", 13)
    pair_contract = att_bwd_bytes(Nb, Eb, Eb * 4, 0)
    pair_us = statistics.mean(t_dst) + statistics.mean(t_src)

    # --- 3xTF32 projection (forward / dX)
    def proj(i):
        ops.proj_fwd(hs[i], W, bias, alpha, 96, 0, 64, precision=ops.PRECISION_TF32X3)
    us = _cold_time(proj, sets, iters)
    entry("k_tc_proj3r", us, (Nb * 128 + Nb * 128 + Nb * 8) * 4,
          "reads x [N,128]; writes h [N,128] and the logit scalars S [N,8] (W resident in shared memory)", 24)
    # a plain device copy of the forward kernel's byte count, timed the same way: what the memory system delivers at
    # this problem size (launch ramp and tail included)
    n_copy = max(1, fused // 8)
    srcs = [torch.empty(n_copy, dtype=torch.float32, device=dev) for _ in range(sets)]
    dsts = [torch.empty(n_copy, dtype=torch.float32, device=dev) for _ in range(sets)]
    copy_us = _cold_time(lambda i: dsts[i].copy_(srcs[i]), sets, iters)
    extra = {"bwd_pair_bytes_contract": int(pair_contract), "bwd_pair_us": round(pair_us, 2),
             "bwd_pair_frac_contract": round(pair_contract / pair_us / 1e3 / peak, 4) if peak else None,
             "same_size_copy_gbs": round(2 * n_copy * 4 / copy_us / 1e3, 1), "nodes": Nb, "edges": Eb,
             "cache": f"{sets} operand sets cycled per kernel (> 126 MB L2)"}
    return out, extra


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return {"hbm_gbs": d.get("hbm_gbs"), "source": "MEASURED_PEAKS.json (of measured)"}
    return {"hbm_gbs": 6650.0, "source": "B200_PROFILING.md fallback (of fallback)"}


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference itself (oracle/_ref or the checkout, through oracle/shims.py) or, if neither is there, the port
def _reference_modules():
    from oracle import ref_import
    if ref_import.available():
        with ref_import.quiet():
            ns = ref_import.load()
        return ns, ("reference", f"unmodified reference modules ({ref_import.kind()}) + third-party shims")
    return None, ("port", "oracle port (no reference build under oracle/_ref)")


def _time_cpu_steps(one, batches, steps, warmup):
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        one(batches[i % len(batches)])
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    return statistics.mean(times)


def cpu_pretrain_rate(shape, n_mols, steps, warmup, seed=0):
    """The reference's pretraining step (FragNetPreTrain.forward + the loss and update of Trainer.train,
    pretrain_utils.py:9-31) on the host cores: (molecules/s, seconds per step, kind, description)."""
    torch.set_num_threads(os.cpu_count() or 1)
    torch.manual_seed(seed)
    ns, (kind, how) = _reference_modules()
    batches = make_batches(shape, n_mols, 2, 256, seed + 1)
    loss_fn = torch.nn.MSELoss()
    if ns is not None:
        from oracle import ref_import
        model = ns.pretrain_heads.FragNetPreTrain(**PT_KW).train()
        opt = torch.optim.Adam(model.parameters(), lr=LR)

        def one(b):
            opt.zero_grad()
            with ref_import.quiet():          # the layer prints on every forward (gat2.py:172)
                bl, ba, da, e = model(b)
            # pretrain_utils.py:22-26 (the bond-length term is overwritten by the dihedral term)
            loss_l = loss_fn(da, b["dh_angl"])
            loss = loss_l + loss_fn(ba, b["bnd_angl"]) + loss_l + loss_fn(e.view(-1), b["y"])
            loss.backward()
            loss.item()
            opt.step()
    else:
        from fragnet.model.gat.gat2_pretrain import FragNetPreTrain
        from oracle import gat2_oracle as O
        P = O.params_from_module(FragNetPreTrain(**PT_KW))
        opt = torch.optim.Adam([v for v in P.values() if v.requires_grad], lr=LR)

        def one(b):
            opt.zero_grad()
            loss = O.pretrain_loss(O.pretrain_forward(P, b, drop_ratio=PT_KW["drop_ratio"], training=True), b)
            loss.backward()
            loss.item()
            opt.step()
    sec = _time_cpu_steps(one, batches, steps, warmup)
    return n_mols / sec, sec, kind, how


def cpu_esol_finetune_rate(steps=5, warmup=1, batch=128):
    """BASELINE configs[0]: FragNetFineTune per exps/ft/esol/e1pt4.yaml (FTHead3 128/1024/1024/512, drop 0.1), ESOL-shaped
    molecules, batch 128, fwd + MSE + bwd + Adam on the host cores (train/utils.py:331-351)."""
    torch.set_num_threads(os.cpu_count() or 1)
    torch.manual_seed(0)
    ns, (kind, how) = _reference_modules()
    batches = make_batches("esol", batch, 2, 256, seed=7, pretrain=False)
    loss_fn = torch.nn.MSELoss()
    if ns is not None:
        from oracle import ref_import
        model = ns.gat2.FragNetFineTune(**FT_KW).train()
        opt = torch.optim.Adam(model.parameters(), lr=LR)

        def one(b):
            opt.zero_grad()
            with ref_import.quiet():
                out = model(b)
            loss = loss_fn(out.view(-1), b["y"])
            loss.backward()
            loss.item()
            opt.step()
    else:
        from fragnet.model.gat.gat2 import FragNetFineTune
        from oracle import gat2_oracle as O
        P = O.params_from_module(FragNetFineTune(**FT_KW))
        opt = torch.optim.Adam([v for v in P.values() if v.requires_grad], lr=LR)

        def one(b):
            opt.zero_grad()
            loss = loss_fn(O.finetune_forward(P, b).view(-1), b["y"])
            loss.backward()
            loss.item()
            opt.step()
    sec = _time_cpu_steps(one, batches, steps, warmup)
    return {"workload": "FragNetFineTune exps/ft/esol/e1pt4.yaml step (fwd + MSE + bwd + Adam), ESOL-shaped molecules, "
                        f"batch {batch}, host cores (BASELINE configs[0])",
            "value": round(batch / sec, 2), "unit": "molecules/s", "ms_per_step": round(sec * 1e3, 1),
            "cores": os.cpu_count() or 1, "kind": kind, "how": how, "steps": steps, "warmup": warmup,
            "batch0_counts": batch_counts(batches[0])}


def workload_name(shape):
    """``config.workload`` of both arms (BASELINE.json configs[1])."""
    return f"FragNetPreTrain exps/pt/unimol_exp1s4 step (4 layers, 4 heads, emb 128, drop 0.2, Adam), {shape}-shaped molecules"


# Steps between the launch of a step and the host's read of its loss in the host-fed legs (every loss is read inside the
# timed region either way).  FNB_BENCH_LAG overrides for measurements.
LOSS_LAG = int(os.environ.get("FNB_BENCH_LAG", "1"))


def bench_config(args, world):
    """``config`` of the JSON line -- the same dict in both arms (the driver compares them)."""
    return {"workload": workload_name(args.shape), "per_gpu_batch": args.batch, "global_batch": args.batch * world,
            "parallelism": f"dp{world}",
            "cache": f"GPU arm: {args.rotate} distinct batches rotated, fwd+bwd working set > 126 MB L2, CSR plans rebuilt "
                     "every step; CPU arm: a bounded sample of the same workload per step (see cpu_baseline.sample)"}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path, all host threads, on a bounded sample of
    the workload (the full per-GPU batch when it fits the time budget)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    budget = 150.0 / max(1, args.steps + args.warmup)            # seconds per step
    n_mols = int(max(32, min(args.batch, 150 * budget)))
    with contextlib.redirect_stdout(io.StringIO()):
        rate, sec, kind, how = cpu_pretrain_rate(args.shape, n_mols, args.steps, args.warmup)
    cores = os.cpu_count() or 1
    sample = f"{n_mols} {args.shape}-shaped molecules per step (fwd+bwd+Adam, train mode, drop 0.2); {how}"
    line = {"metric": METRIC, "value": round(rate, 2), "unit": "molecules/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(sec * 1e3, 2),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "impl": "reference",
            "config": bench_config(args, args.gpus),
            "cpu_baseline": {"value": round(rate, 2), "unit": "molecules/s", "cores": cores, "kind": kind,
                             "sample": sample},
            "e2e": {"value": round(rate, 2), "unit": "molecules/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
def make_step(batch=1024, shape="unimol", rotate=4, pool=512, precision="fp32", rank=0, world=1, dev=None,
              return_host=False, autograd_path=False, pack=False, return_model=False):
    """The timed unit: ``step(batch_dict)`` = on-device collate + forward + loss + backward + gradient all-reduce
    (world > 1) + Adam on one batch.  Returns (step, device batches[, pinned host batches in the compact wire format]
    [, the model the step trains])."""
    from fragnet.model.gat.gat2_pretrain import FragNetPreTrain
    from fragnet_b200 import config, ops
    from fragnet_b200.dataset.data import compact_batch, pack_batch
    from fragnet_b200.dist import FlatGradSync
    from fragnet_b200.train.optim import FlatAdam
    from fragnet_b200.train.pretrain_utils import pretrain_loss
    dev = dev or torch.device("cuda", torch.cuda.current_device())
    config.set_precision(precision)
    torch.manual_seed(1234)                      # identical initial weights on every rank
    model = FragNetPreTrain(**PT_KW).to(dev).train()
    loss_fn = torch.nn.MSELoss()
    wide = make_batches(shape, batch, rotate, pool, seed=100 + rank)
    dev_batches = [{k: v.to(dev) for k, v in b.items()} for b in wide]
    # what a DataLoader with collate_fn_pt_compact + pin_memory hands over: uint8 one-hot matrices, int32 indices
    # (pack: collate_fn_pt_packed, the tensors of the hot path as views of one pinned buffer per batch)
    host_batches = [(pack_batch(compact_batch(b), pin=True) if pack else compact_batch(b, pin=True)) for b in wide] \
        if return_host else None
    if autograd_path:
        # the unchanged reference loop: model(batch) -> loss -> backward -> (all-reduce) -> Adam, through nn.Module
        sync = FlatGradSync(model.parameters())
        opt = None

        def step(b):
            nonlocal opt
            ops.clear_plan_cache()       # every step is a new batch to the model: the on-device collate is always timed
            sync.zero()
            loss = pretrain_loss(loss_fn, model(b), b)
            loss.backward()
            sync.sync()
            if opt is None:          # Adam over the live parameters (grad-less ones are skipped by torch's Adam too)
                opt = FlatAdam(sync.live_parameters(), lr=LR)
            opt.step(sync.flat if world > 1 else None)
            return loss
    else:
        # the same arithmetic as ONE library call per step (+ gradient all-reduce + one Adam launch)
        from fragnet_b200.train.fused import FusedPretrainStep
        step = FusedPretrainStep(model, lr=LR).step

    out = (step, dev_batches, host_batches) if return_host else (step, dev_batches)
    return out + (model,) if return_model else out


class Timer:
    """K steps bracketed by barrier + synchronize, CUDA events on the launch stream, max over ranks."""

    def __init__(self, dev, world, lib):
        self.dev, self.world, self.lib = dev, world, lib

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def __call__(self, run_step, n_steps):
        self.barrier()
        e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
        l0 = self.lib.fnb_launch_count()
        e0.record()
        for i in range(n_steps):
            run_step(i)
        e1.record()
        self.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=self.dev)
        if self.world > 1:
            import torch.distributed as dist
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms), self.lib.fnb_launch_count() - l0


def dump_outputs(path, model, loss):
    """``--dump-outputs``: what a training step hands its caller -- the loss, and the model's parameters after the
    Adam update with the gradients they were updated from -- one float32 ``.npy`` per array (~6 MB in all at PT_KW),
    so that two builds run with the same arguments can be compared array by array.  Returns the file names."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    arrays = {"loss": loss}
    for name, p in model.named_parameters():
        arrays[f"param.{name}"] = p
        if p.grad is not None:
            arrays[f"grad.{name}"] = p.grad
    for name, t in arrays.items():
        np.save(os.path.join(path, name + ".npy"), t.detach().float().cpu().numpy())
    return sorted(arrays)


# ------------------------------------------------------------------------------------------------
def extra_inference(dev, timed, world, rank, steps=24, warmup=3, batch=4096):
    """BASELINE configs[2]: inference screening, batch 4096 per GPU, eval mode, the last layer's attention sums returned
    (the arrangement of vizualize/model.py).  Resident: batches in HBM, outputs left on the device; e2e: the screening
    pipeline on the packed arena -- molecule ids in, predictions + four attention tensors copied to pinned host memory."""
    import numpy as np

    from fragnet.vizualize.model import FragNetFineTuneViz
    from fragnet_b200 import ops, synth
    from fragnet_b200.dataset.arena import MoleculeArena
    from fragnet_b200.screen import screen
    torch.manual_seed(7)
    viz = FragNetFineTuneViz(num_layer=4, drop_ratio=0.1, n_classes=1, edge_features=17).to(dev).eval()
    pool = synth.make_dataset("unimol", 512, seed=300 + rank, with_pretrain_targets=False)
    arena = MoleculeArena(pool, dev, pretrain=False)
    rng = np.random.default_rng(300 + rank)
    ids = [rng.integers(0, len(pool), size=batch) for _ in range(4)]
    dev_batches = [{k: v.clone() for k, v in arena.batch(i).items()} for i in ids]
    sink = [None]

    def resident(i):
        with torch.no_grad():
            ops.clear_plan_cache()
            sink[0] = viz(dev_batches[i % 4])
    for i in range(warmup):
        resident(i)
    ms_res, _ = timed(resident, steps)
    d2h = sum(int(t.numel()) * t.element_size() for t in sink[0])
    all_ids = np.concatenate([ids[j % 4] for j in range(steps + warmup)])
    state = {"n": 0}

    def e2e(i):            # one timed call = the whole pipelined screen of (steps + warmup) batches
        for _bid, outs in screen(viz, arena, batch_size=batch, ids=all_ids):
            state["n"] += int(outs[0].shape[0])
    for _ in screen(viz, arena, batch_size=batch, ids=all_ids[:2 * batch]):
        pass
    ms_e2e, _ = timed(e2e, 1)
    assert state["n"] == all_ids.shape[0]
    n_e2e = all_ids.shape[0]
    out = {"workload": f"inference screening (BASELINE configs[2]): FragNetFineTuneViz eval, batch {batch} per GPU, "
                       "prediction + last-layer attention sums of the four graphs returned, UniMol-shaped molecules",
           "value": round(batch * steps * world / (ms_res * 1e-3), 1), "unit": "molecules/s",
           "ms_per_batch": round(ms_res / steps, 3),
           "e2e": {"value": round(n_e2e * world / (ms_e2e * 1e-3), 1), "unit": "molecules/s",
                   "h2d_bytes_per_step": batch * 8, "d2h_bytes_per_step": d2h,
                   "seconds_per_1M_molecules": round(1e6 / (n_e2e * world / (ms_e2e * 1e-3)), 3),
                   "how": "fragnet_b200.screen on a MoleculeArena: molecule ids in; on-device batch assembly, forward and "
                          "the pinned device-to-host copy of predictions + attention sums in flight together; every "
                          "batch's results are on the host inside the timed region"},
           "n_gpus": world, "steps": steps, "warmup": warmup, "precision": "fp32"}
    del arena
    return out


def extra_stress(dev, timed, world, rank, steps=8, warmup=3, batch=1024):
    """BASELINE configs[4]: skewed-degree stress (~100 atoms, ~20 fragments, 3 components, ~20 k fragment-connection
    edges per molecule), per-GPU batch 1024, the same pretraining step."""
    step, dev_batches = make_step(batch, "stress", rotate=2, pool=64, precision="fp32", rank=rank, world=world, dev=dev)
    for i in range(warmup):
        step(dev_batches[i % 2])
    ms, launches = timed(lambda i: step(dev_batches[i % 2]), steps)
    c = {k: int(v) for k, v in batch_counts(dev_batches[0]).items()}
    _, all_b = step_bytes(c)
    peak = load_peaks()["hbm_gbs"]
    sec = ms * 1e-3 / steps
    return {"workload": workload_name("stress") + f", per-GPU batch {batch} (BASELINE configs[4])",
            "value": round(batch * world / sec, 1), "unit": "molecules/s", "ms_per_step": round(ms / steps, 3),
            "n_gpus": world, "steps": steps, "warmup": warmup, "precision": "fp32", "batch0_counts": c,
            "roofline_step": {"bytes_contract": int(all_b), "achieved": round(all_b / sec / 1e9, 1), "peak": peak,
                              "frac": round(all_b / sec / 1e9 / peak, 4)},
            "gpu_launches": int(launches)}


# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist

    from fragnet_b200 import _abi, config

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl ours) needs a CUDA device: there is no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    lib = _abi.load()
    step, dev_batches, host_batches, model = make_step(args.batch, args.shape, args.rotate, args.pool, args.precision,
                                                       rank, world, dev, return_host=True, autograd_path=args.autograd,
                                                       pack=args.pack, return_model=True)
    timed = Timer(dev, world, lib)
    barrier = timed.barrier
    # a training loop knows its next batch: its on-device collate is queued underneath the running step
    # (FusedPretrainStep.prefetch_plan; --no-plan-prefetch collates at the head of every step instead)
    fs = getattr(step, "__self__", None)
    prefetch = fs.prefetch_plan if (fs is not None and hasattr(fs, "prefetch_plan") and not args.no_plan_prefetch) else None

    last_loss = [None]

    def resident(i):
        loss = last_loss[0] = step(dev_batches[i % args.rotate])
        if prefetch is not None:
            prefetch(dev_batches[(i + 1) % args.rotate])
        return loss

    # ---- kernel-resident throughput: inputs already in HBM
    for i in range(args.warmup):
        resident(i)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_total, launches = timed(resident, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    mols = args.batch * world * args.steps
    value = mols / (ms_total * 1e-3)
    if args.dump_outputs and rank == 0:
        # before the legs below take further steps on the same model
        dump_outputs(args.dump_outputs, model, last_loss[0])

    # ---- the same step with single-TF32 products (stated tolerance 2e-3): value_tf32
    tf32 = None
    if not args.no_tf32 and args.precision == "fp32" and not args.autograd:
        config.set_precision("tf32")
        for i in range(max(3, args.warmup)):
            resident(i)
        ms_tf, _ = timed(resident, args.steps)
        tf32 = {"value": round(mols / (ms_tf * 1e-3), 1), "ms_per_step": round(ms_tf / args.steps, 4)}
        config.set_precision(args.precision)
        step(dev_batches[0])

    # ---- end to end through the public API with HOST (pinned) batches: H2D + step + loss read back
    e2e = None
    if not args.no_e2e:
        from fragnet_b200.dataset.prefetch import DevicePrefetcher, staged_bytes
        from fragnet_b200.train.fused import LaggedScalars
        h2d = staged_bytes(host_batches[0])
        reader = LaggedScalars(lag=LOSS_LAG)     # pinned floats, allocated once (cudaHostAlloc synchronises the device)

        def e2e_run(n):
            staged = DevicePrefetcher((host_batches[i % args.rotate] for i in range(n)), dev, depth=2, hot_path_only=True)
            feed = iter(staged)
            state = {"b": next(feed), "sum": 0.0, "read": 0}

            def one(i):
                loss = step(state["b"])
                state["b"] = next(feed, None)     # stage batch i+2 while step i runs on the GPU
                if prefetch is not None and state["b"] is not None:
                    prefetch(state["b"], staged.last_event)   # collate of batch i+1 underneath step i
                # every step's loss is copied device -> host (pinned) behind its step and collected once the next
                # step has been enqueued; the last one is collected inside the timed region too
                vals = reader.push(loss) + (reader.drain() if i == n - 1 else [])
                state["sum"] += sum(vals)
                state["read"] += len(vals)
                if i == n - 1:
                    assert state["read"] == n and state["sum"] == state["sum"]
            return one

        # (the first pinned-memory transfers of a fresh process run slower for some tens of milliseconds: the host-fed legs
        # warm up for at least 24 steps, whatever --warmup says for the resident leg)
        # One epoch-like run: the same DevicePrefetcher feeds the warm-up steps and the timed steps.  (A prefetcher
        # created inside the timed region allocates its device slots there; depending on the state of the caching
        # allocator that is a cudaMalloc / cudaFree round -- a 100-300 ms device-synchronising stall that showed up as
        # 1.45-2.3 ms per step in one run out of three, gpurun_out/r5w..r6b -- which an epoch of thousands of steps pays once.)
        n_warm = max(24, args.warmup)
        run = e2e_run(n_warm + args.steps)
        for i in range(n_warm):
            run(i)
        barrier()
        ms_e2e, _ = timed(lambda i: run(n_warm + i), args.steps)
        e2e = {"value": round(mols / (ms_e2e * 1e-3), 1), "unit": "molecules/s", "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": 4, "ms_per_step": round(ms_e2e / args.steps, 3),
               "batch_dict_bytes": sum(v.numel() * v.element_size() for v in dev_batches[0].values()),
               "staging": "pinned host batches in the compact wire format of collate_fn_pt_compact (one-hot feature "
                          "matrices uint8, indices int32: exact" + ("; packed into one buffer per batch" if args.pack else "")
                          + ") -> DevicePrefetcher(hot_path_only=True) copies the tensors FragNet.forward reads and "
                          "widens them on the device (fnb_widen_batch)",
               "loss_read": "every step's loss is copied to pinned host memory behind its step and collected one step "
                            "later (after the next step has been enqueued); all reads inside the timed region"}

    # ---- the same loop fed by the device-resident packed arena (SURVEY 8(f).1): the per-step host -> device traffic
    # is the list of molecule ids; the batch dict is assembled on the device inside the timed region
    e2e_arena = None
    if not args.no_e2e and not args.autograd and not args.no_arena:
        import numpy as np

        from fragnet_b200 import synth
        from fragnet_b200.dataset.arena import MoleculeArena
        from fragnet_b200.train.fused import LaggedScalars
        pool = synth.make_dataset(args.shape, min(args.pool, args.batch * args.rotate), seed=100 + rank)
        arena = MoleculeArena(pool, dev)
        rng = np.random.default_rng(100 + rank)
        id_lists = [rng.integers(0, len(pool), size=args.batch) for _ in range(args.rotate)]
        reader = LaggedScalars(lag=LOSS_LAG)

        def arena_run(n):
            state = {"b": arena.batch_overlapped(id_lists[0]), "read": 0}

            def one(i):
                loss = step(state["b"])
                # assembled on a side stream underneath step i, its collate queued behind it
                state["b"] = arena.batch_overlapped(id_lists[(i + 1) % args.rotate])
                if prefetch is not None:
                    prefetch(state["b"], arena.last_event)
                vals = reader.push(loss) + (reader.drain() if i == n - 1 else [])
                state["read"] += len(vals)
                if i == n - 1:
                    assert state["read"] == n
            return one

        n_warm = max(24, args.warmup)
        run_a = arena_run(n_warm + args.steps)
        for i in range(n_warm):
            run_a(i)
        barrier()
        ms_a, _ = timed(lambda i: run_a(n_warm + i), args.steps)
        e2e_arena = {"value": round(mols / (ms_a * 1e-3), 1), "unit": "molecules/s",
                     "h2d_bytes_per_step": int(args.batch * 8), "d2h_bytes_per_step": 4,
                     "ms_per_step": round(ms_a / args.steps, 3),
                     "batch_dict_bytes": int(arena.batch_nbytes(id_lists[0])), "arena_bytes": int(arena.nbytes),
                     "note": "dataset resident in HBM (MoleculeArena); per step: molecule ids H2D, on-device batch "
                             "assembly (fnb_arena_assemble), step, loss read back"}
        del arena

    # ---- roofline legs use the bench batch: take them before the extras free it
    roofline = None
    counts = batch_counts(dev_batches[0])
    if rank == 0 and not args.no_roofline:
        peaks = load_peaks()
        peak = peaks["hbm_gbs"]
        kernels, kextra = roofline_kernels(dev_batches[0], peaks)
        _, all_b = step_bytes(counts)
        _, live_b = step_bytes(counts, live_only=True)
        sec = ms_total * 1e-3 / args.steps
        step_r = {"bytes_contract": int(all_b), "bytes_live": int(live_b), "ms": round(sec * 1e3, 4),
                  "achieved": round(all_b / sec / 1e9, 1), "peak": peak, "frac": round(all_b / sec / 1e9 / peak, 4),
                  "frac_live": round(live_b / sec / 1e9 / peak, 4),
                  "note": "encoder fwd+bwd bytes by SURVEY 8d on batch 0's counts (every block of every layer, as the "
                          "reference executes them; `live` drops the fragment blocks / pooling whose output is "
                          "overwritten unread and which this library skips); the heads, loss and Adam are in the time "
                          "but not in the bytes"}
        shares = [(k.get("share_of_kernel_time") or 0.0, i) for i, k in enumerate(kernels)]
        top = kernels[max(shares)[1]] if any(s for s, _ in shares) else kernels[2]
        roofline = {"bound": "hbm", "kernel": top["kernel"] + " (bond graph; largest share of the step's kernel time)",
                    "achieved": top["achieved"], "peak": peak, "unit": "GB/s", "frac": top["frac"],
                    "traffic": top.get("traffic"), "bytes_per_launch": top["bytes_per_launch"],
                    "us_per_launch": top["us_per_launch"], "peak_source": peaks.get("source"),
                    "share_source": KERNEL_SHARE["source"], "traffic_source": NCU_TRAFFIC["source"],
                    "step": step_r, "kernels": kernels, **kextra}

    # ---- BASELINE configs[4] and [2] on every rank (weak scaling / replicas), configs[0] on rank 0's host cores
    extra = {}
    if not args.no_extras and not args.autograd:
        del step, dev_batches, model
        torch.cuda.empty_cache()
        config.set_precision("fp32")
        for name, fn in (("stress_b1024", extra_stress), ("infer_b4096", extra_inference)):
            try:
                extra[name] = fn(dev, timed, world, rank)
            except Exception as ex:      # an extra leg must never take the headline down with it
                if world > 1:
                    raise                # (a rank that skips a collective would hang the others)
                extra[name] = {"error": f"{type(ex).__name__}: {ex}"[:300]}
            torch.cuda.empty_cache()

    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            with contextlib.redirect_stdout(io.StringIO()):
                rate, _sec, kind, how = cpu_pretrain_rate(args.shape, 512, 8, 1)        # ~10-15 s of host work
            cpu = {"value": round(rate, 2), "unit": "molecules/s", "cores": os.cpu_count() or 1, "kind": kind,
                   "sample": f"512 {args.shape}-shaped molecules per step, 1 warm-up + 8 timed steps "
                             f"(fwd+bwd+Adam, train mode, all host threads); {how}"}
            if not args.no_extras:
                try:
                    with contextlib.redirect_stdout(io.StringIO()):
                        extra["esol_ft_cpu"] = cpu_esol_finetune_rate()
                except Exception as ex:
                    extra["esol_ft_cpu"] = {"error": f"{type(ex).__name__}: {ex}"[:300]}
        line = {"metric": METRIC, "value": round(value, 1), "unit": "molecules/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_total / args.steps, 4),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": {"fp32": "f32 (projections: 3xTF32 split on tcgen05, f32-grade; the 1e-5 parity mode)",
                          "fp32_simt": "f32", "tf32": "f32 (tf32-in/f32-acc tensor-core projections)"}[args.precision],
                "precision": args.precision,
                "value_tf32": tf32["value"] if tf32 else None, "ms_per_step_tf32": tf32["ms_per_step"] if tf32 else None,
                "data": "synthetic",
                "config": bench_config(args, world),
                "run": {"batch0_counts": counts,
                        "collate": "on the device, every step" + (" (the collate of batch i+1 is queued underneath step i, "
                                   "as a prefetching loader allows)" if prefetch is not None else ""),
                        "driver": "nn.Module + autograd + FlatAdam" if args.autograd else
                                  "FusedPretrainStep (fnb_pretrain_step + fnb_adam_step)"},
                "e2e": e2e, "e2e_arena": e2e_arena, "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
                "cpu_baseline": cpu, "extra": extra or None}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
