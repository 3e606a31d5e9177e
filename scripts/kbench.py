#!/usr/bin/env python
"""Kernel micro-benchmark on the bench batch: every message-passing kernel, L2 flushed before each launch, CUDA events
on the launch stream; prints microseconds and achieved algorithmic GB/s (DESIGN.md section 3 byte model).

usage (GPU box): python scripts/kbench.py [--batch 1024] [--shape unimol] [--iters 20] [--json out.json]
"""
import argparse
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--shape", default="unimol")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--json", default=None)
    ap.add_argument("--no-flush", action="store_true")
    args = ap.parse_args()
    from bench import make_batches
    from fragnet_b200 import ops
    dev = torch.device("cuda", 0)
    b = {k: v.to(dev) for k, v in make_batches(args.shape, args.batch, 1, 512, seed=100)[0].items()}
    Na, Nb = b["x_atoms"].shape[0], b["node_features_bonds"].shape[0]
    Nf, Nfb = b["x_frags"].shape[0], b["node_features_fbonds"].shape[0]
    plan = ops.build_layer_plan(b["edge_index"], b["frag_index"], b["atom_to_frag_ids"], b["edge_index_bonds_graph"],
                                b["edge_attr_bonds"], b["edge_index_fbonds"], b["edge_attr_fbonds"], Na, Nf, Nb, Nfb, dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    results = []

    def timeit(name, fn, nbytes):
        ts = []
        for i in range(args.iters + 3):
            if not args.no_flush:
                flush.zero_()
            e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            if i >= 3:
                ts.append(e0.elapsed_time(e1) * 1e3)
        us = statistics.median(ts)
        gbs = nbytes / us / 1e3
        results.append(dict(kernel=name, us=round(us, 2), min_us=round(min(ts), 2), MB=round(nbytes / 1e6, 2),
                            GBs=round(gbs, 1)))
        print(f"{name:44s} {us:9.2f} us  (min {min(ts):8.2f})  {nbytes / 1e6:9.2f} MB  {gbs:8.1f} GB/s", flush=True)

    gen = torch.Generator(device=dev).manual_seed(0)
    rnd = lambda *s: torch.randn(*s, device=dev, generator=gen)
    a96, a192 = rnd(4, 96) * 0.1, rnd(4, 192) * 0.1
    We1, be1, We6, be6 = rnd(32, 1), rnd(32), rnd(32, 6), rnd(32)
    graphs = [("bond", plan.bond, ops.EDGE_AFFINE1, a96, 96, 64), ("atom", plan.atom, ops.EDGE_TABLE, a192, 192, 160),
              ("fbond", plan.fbond, ops.EDGE_AFFINE6, a96, 96, 64), ("frag", plan.frag, ops.EDGE_TABLE, a192, 192, 160)]
    for name, g, mode, alpha, stride, off_s in graphs:
        N, E = g.n_nodes, g.n_edges
        h, go = rnd(N, 128), rnd(N, 128)
        S = ops.node_scalars(h, alpha, stride, 0, off_s)
        X = {ops.EDGE_AFFINE1: E * 4, ops.EDGE_AFFINE6: E * 24, ops.EDGE_TABLE: E * 16 + E * 4}[mode]
        fwd_bytes = 2 * N * 512 + X + 2 * E * 4 + (N + 1) * 4 + E * 16 + 2 * N * 32
        kw_b = {}
        if mode == ops.EDGE_AFFINE1:
            kw_new = dict(We=We1, be=be1, alpha_e=alpha[:, 32:], alpha_stride=stride)
            kw_b = dict(We=We1, be=be1)
        elif mode == ops.EDGE_AFFINE6:
            kw_new = dict(We=We6, be=be6, alpha_e=alpha[:, 32:], alpha_stride=stride)
            kw_b = dict(We=We6, be=be6)
        else:
            kw_new = dict(table=rnd(g.n_real, 4))
        timeit(f"{name}: gat_fwd tiled (N={N},E={E})", lambda: ops.gat_fwd_tiled(g, h, S, mode, **kw_new), fwd_bytes)
        timeit(f"{name}: gat_fwd tiled +y(drop .2)+nextSe",
               lambda: ops.gat_fwd_tiled(g, h, S, mode, post=(0.2, 1, 1, 1, 0), next_alpha=a192[:, 32:],
                                         next_alpha_stride=192, **kw_new), fwd_bytes + N * 512 + N * 16)
        timeit(f"{name}: gat_fwd tiled inference (y only)",
               lambda: ops.gat_fwd_tiled(g, h, S, mode, save_p=False, want_out=False, post=(0.0, 0, 1, 0, 0), **kw_new),
               fwd_bytes - E * 16)
        _, _, p, _ = ops.gat_fwd_tiled(g, h, S, mode, **kw_new)
        d_alpha = torch.zeros(4, stride, device=dev)
        bwd_bytes = 5 * N * 512 + 4 * E * 16 + 3 * E * 4 + 2 * N * 16 + 2 * (N + 1) * 4
        timeit(f"{name}: gat_bwd dst+src tiled",
               lambda: ops.gat_bwd_tiled(g, h, go, p, mode, alpha, stride, 0, 32, off_s, d_alpha, want_bias_grad=True,
                                         **kw_b), bwd_bytes)
        if mode == ops.EDGE_TABLE:
            dz = rnd(E, 4)
            feat, dy = rnd(g.n_real, 128), rnd(g.n_real, 128)
            y = torch.relu(feat)
            timeit(f"{name}: edge_table_bwd fused dropout-relu bwd",
                   lambda: ops.edge_table_bwd_fused(g, dz, feat, alpha, stride, 32, d_alpha, dy=dy, y=y, post_scale=1.25),
                   4 * g.n_real * 512)
    # dense projections
    for N, K, label in ((Nb, 128, "bond"), (Na, 128, "atom")):
        x, W, bb, dh = rnd(N, K), rnd(128, K) * 0.1, rnd(128), rnd(N, 128)
        for prec, pn in ((0, "fp32"), (1, "tf32")):
            timeit(f"proj_fwd {label} {N}x{K} {pn}", lambda: ops.proj_fwd(x, W, bb, a96, 96, 0, 64, precision=prec),
                   (N * K + N * 128 + N * 8) * 4)
            timeit(f"proj_bwd {label} {N}x{K} {pn} (dx+dW)", lambda: ops.proj_bwd(x, W, dh, True, prec, want_db=False),
                   4 * N * 128 * 4)
    x = rnd(Nb, 128)
    timeit("dropout_relu_fwd bond", lambda: ops.dropout_relu_fwd(x, 0.2, True, True, 1, 0), 2 * Nb * 512)
    timeit("copy (torch) bond [N,128]", lambda: x.clone(), 2 * Nb * 512)
    big = torch.empty(1 << 28, dtype=torch.float32, device=dev)
    big2 = torch.empty_like(big)
    timeit("copy (torch) 1 GiB", lambda: big2.copy_(big), 2 * big.numel() * 4)
    if args.json:
        json.dump(results, open(args.json, "w"), indent=1)


if __name__ == "__main__":
    main()
