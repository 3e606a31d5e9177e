#!/usr/bin/env python
"""Projection GEMMs alone, per precision mode (0 FFMA, 1 TF32, 2 3xTF32): cold (L2 flushed) and back-to-back timings
with CUDA events; algorithmic GB/s = (N*K + N*128 + N*8)*4 bytes (forward), (2*N*128 + 2*N*K)*4 (dX + dW).  K is the
weight's input width: 128 for the attention projections, 167 / 17 / 6 for the raw input features of layer 0, 256 for
the energy head's readout.

usage (GPU box): python scripts/gemm_bench.py [--rows 53940,26000,10000] [--k 128] [--iters 20]
"""
import argparse
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", default="53940,26000,10000,215000")
    ap.add_argument("--k", type=int, default=128, help="input width K of the [128, K] weight")
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    from fragnet_b200 import ops
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def timeit(fn, cold):
        ts = []
        for i in range(args.iters + 3):
            if cold:
                flush.zero_()
            e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            if i >= 3:
                ts.append(e0.elapsed_time(e1) * 1e3)
        return statistics.median(ts)

    a96 = torch.randn(4, 96, device=dev) * 0.1
    K = args.k
    for N in [int(r) for r in args.rows.split(",")]:
        x, W, b, dh = (torch.randn(N, K, device=dev), torch.randn(128, K, device=dev) * 0.1,
                       torch.randn(128, device=dev), torch.randn(N, 128, device=dev))
        fb, bb = (N * K + N * 128 + N * 8) * 4, (2 * N * 128 + 2 * N * K) * 4
        for prec, name in ((0, "ffma"), (1, "tf32"), (2, "3xtf32")):
            f = lambda: ops.proj_fwd(x, W, b, a96, 96, 0, 64, precision=prec)
            g = lambda: ops.proj_bwd(x, W, dh, True, prec, want_db=False)
            w = lambda: ops.proj_bwd(x, W, dh, False, prec, want_db=False)
            fc, fw, gc, gw, wc = timeit(f, True), timeit(f, False), timeit(g, True), timeit(g, False), timeit(w, True)
            print(f"N={N:7d} K={K:3d} {name:7s} fwd cold {fc:7.2f} us ({fb / fc / 1e3:6.0f} GB/s) warm {fw:7.2f} us | "
                  f"dX+dW cold {gc:7.2f} us ({bb / gc / 1e3:6.0f} GB/s) warm {gw:7.2f} us | dW only cold {wc:7.2f} us",
                  flush=True)


if __name__ == "__main__":
    main()
