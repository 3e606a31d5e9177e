"""bench.py end to end on a small batch: ``--steps`` sets the number of timed steps, and ``--dump-outputs`` writes what
the last of them returned to its caller, the same from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT


def _bench(out, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "2",
           "--batch", "64", "--rotate", "2", "--pool", "64", "--no-cpu-baseline", "--no-e2e", "--no-roofline",
           "--no-extras", "--no-tf32", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def _load(d):
    return {f[:-len(".npy")]: np.load(d / f) for f in os.listdir(d)}


@pytest.mark.gpu
def test_bench_steps_and_dumped_outputs(tmp_path):
    import bench
    from fragnet.model.gat.gat2_pretrain import FragNetPreTrain
    two, again, four = (_bench(tmp_path / n, s) for n, s in (("two", 2), ("again", 2), ("four", 4)))
    # the two batches alternate: four timed steps launch exactly twice what two do
    assert two["gpu_launches"] > 0 and four["gpu_launches"] == 2 * two["gpu_launches"]
    params = [f"param.{k}" for k, _ in FragNetPreTrain(**bench.PT_KW).named_parameters()]
    dumps = [_load(tmp_path / n) for n in ("two", "again", "four")]
    for arrays in dumps:
        assert set(arrays) >= {"loss", *params}
        grads = [k for k in arrays if k.startswith("grad.")]
        assert grads and all("param." + k[len("grad."):] in params for k in grads)
        assert len(arrays) == 1 + len(params) + len(grads)
        assert all(a.dtype == np.float32 and np.isfinite(a).all() for a in arrays.values())
        assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
        assert arrays["loss"].size == 1 and float(arrays["loss"]) > 0
    # same arguments, same inputs, same results: the step's float reductions do not depend on the order in which
    # blocks finish (its only atomics are integer counters), so two runs agree bit for bit
    assert sorted(dumps[0]) == sorted(dumps[1])
    assert all(np.array_equal(dumps[0][k], dumps[1][k]) for k in dumps[0])
    # the dump is taken after the last timed step: two more Adam steps have moved the parameters
    assert any(not np.array_equal(dumps[0][k], dumps[2][k]) for k in params)
