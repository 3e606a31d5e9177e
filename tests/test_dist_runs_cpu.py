"""Argument checks of ``fnb_allreduce_adam_runs`` (the data-parallel exchange with per-run Adam step counts): every
malformed run table returns its documented code from the host-side checks, before anything is launched (CPU only)."""
import ctypes as C

import pytest
import torch

N = 64          # floats of the flat buffer in these calls


@pytest.fixture(scope="module")
def call():
    from fragnet_b200 import _abi
    lib = _abi.load()
    bufs = [torch.zeros(N) for _ in range(5)]            # 64-byte aligned host memory: never touched, no launch
    p, m, v, g, flags = (C.c_void_p(t.data_ptr()) for t in bufs)
    done = C.c_void_p(bufs[4].data_ptr())
    peers = _abi.CPeerSet()
    peers.grads[0], peers.flags[0], peers.world, peers.rank = g, flags, 1, 0

    def run(table, n_runs=None, n=N, runs_ptr=True):
        arr = (_abi.CAdamRun * max(1, len(table)))(*table)
        return lib.fnb_allreduce_adam_runs(C.byref(peers), p, m, v, n, arr if runs_ptr else None,
                                           len(table) if n_runs is None else n_runs, 1e-3, 0.9, 0.999, 1e-8, 0.0, 1,
                                           done, None)
    run.keep = bufs
    return run


def test_null_run_table(call):
    assert call([(0, N, 1)], runs_ptr=False) == -1


@pytest.mark.parametrize("table", [[(0, 6, 1), (6, N, 1)], [(2, N, 1)], [(0, N - 2, 1)]],
                         ids=["end", "first", "last-end"])
def test_boundaries_that_are_not_multiples_of_4(call, table):
    assert call(table) == -5


@pytest.mark.parametrize("table", [
    [(0, 16, 1), (8, N, 2)],            # overlapping
    [(0, 16, 1), (20, N, 2)],           # gap
    [(0, 32, 1)],                       # does not reach n
    [(0, 32, 1), (32, N + 4, 1)],       # past n
    [(4, N, 1)],                        # does not start at 0
    [(0, 16, 1), (16, 16, 1), (16, N, 1)],   # empty run
    [(0, 16, 2), (16, N, 0)],           # step < 1
], ids=["overlap", "gap", "short", "long", "offset", "empty", "step0"])
def test_run_tables_that_do_not_tile_the_buffer(call, table):
    assert call(table) == -2


def test_run_count_limits(call):
    from fragnet_b200 import _abi
    assert call([], n_runs=0) == -2
    k = _abi.MAX_ADAM_RUNS + 1
    assert call([(4 * i, 4 * i + 4, 1) for i in range(k)], n=4 * k) == -2
    assert call([(0, N, 1)], n=N + 2) == -2               # n itself not a multiple of 4, as fnb_allreduce_adam_step


def test_limit_matches_the_header():
    import os
    import re
    from conftest import ROOT
    from fragnet_b200 import _abi
    text = open(os.path.join(ROOT, "include", "fragnet_b200.h")).read()
    assert int(re.search(r"#define FNB_MAX_ADAM_RUNS (\d+)", text).group(1)) == _abi.MAX_ADAM_RUNS
    assert C.sizeof(_abi.CAdamRun) == 24
