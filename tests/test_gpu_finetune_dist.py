"""Data-parallel fused finetuning: ``FusedFineTuneStep(model, group=...)``, ``TrainerFineTune(fused=True)`` on a
``DistributedDataParallel`` model, and the exchange kernel with per-run Adam step counts (``fnb_allreduce_adam_runs``).

Ranks are processes started with ``torch.multiprocessing`` (spawn); every one is joined with a timeout and killed if it
is still alive, so no process outlives a test.  On one GPU two ranks share the device over ``gloo``: the exchange then
takes the ``dist.all_reduce`` + ``_adam()`` path.  With two or more GPUs the ranks use NCCL and the symmetric-memory
exchange kernel."""
import copy
import os
import socket
import traceback

import pytest
import torch
import torch.distributed as dist

from conftest import rel_err
from test_gpu_finetune_step import W_ODD, _case_batch, _model

pytestmark = pytest.mark.gpu

TIMEOUT = 600          # seconds per spawned group of ranks
SEED0 = 100            # rank r's model is seeded SEED0 + r: the broadcast has to make them equal


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _entry(worker, rank, world, port, out, backend):
    """Child process: one rank.  Results go to ``out/res{rank}.pt``, a failure's traceback to ``out/err{rank}.txt``."""
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dev = torch.device("cuda", rank if backend == "nccl" else 0)
    torch.cuda.set_device(dev)
    try:
        kw = {"device_id": dev} if backend == "nccl" else {}
        dist.init_process_group(backend, rank=rank, world_size=world, **kw)
        try:
            res = globals()[worker](rank, world)
            torch.cuda.synchronize()
            torch.save(res, os.path.join(out, f"res{rank}.pt"))
        finally:
            dist.destroy_process_group()
    except BaseException:
        with open(os.path.join(out, f"err{rank}.txt"), "w") as f:
            f.write(traceback.format_exc())
        raise


def _spawn(worker, world, out, backend):
    ctx = torch.multiprocessing.get_context("spawn")
    port = _free_port()
    procs = [ctx.Process(target=_entry, args=(worker, r, world, port, str(out), backend)) for r in range(world)]
    for p in procs:
        p.start()
    try:
        for p in procs:
            p.join(TIMEOUT)
    finally:
        for p in procs:
            if p.is_alive():
                p.kill()
                p.join(30)
    errs = [open(out / f"err{r}.txt").read() for r in range(world) if (out / f"err{r}.txt").exists()]
    assert not errs and all(p.exitcode == 0 for p in procs), "\n".join(errs) or [p.exitcode for p in procs]
    return [torch.load(out / f"res{r}.pt", weights_only=False) for r in range(world)]


def _batches(rank, n=3, seed=500):
    """Different batches on every rank."""
    return [_case_batch(1, "mse", seed + 10 * rank + i) for i in range(n)]


def _resume(m, opt_seed=7):
    """An Adam state as a resumed run with gradual unfreezing leaves it: the encoder 3 steps in, the head 7 steps in
    (two runs of the flat buffer), moments from a fixed generator."""
    opt = torch.optim.Adam(m.parameters(), lr=1e-3)
    gen = torch.Generator().manual_seed(opt_seed)
    for name, p in m.named_parameters():
        steps = 7 if name.startswith("fthead.") else 3
        opt.state[p] = {"step": torch.tensor(float(steps)),
                        "exp_avg": (1e-3 * torch.randn(p.shape, generator=gen)).to(p.device),
                        "exp_avg_sq": (1e-6 * torch.rand(p.shape, generator=gen)).to(p.device)}
    return opt


def _state(m):
    return {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}


# ---- ranks: one GPU, gloo (the dist.all_reduce + _adam() exchange) -------------------------------------------------------
def _w_gloo(rank, world):
    from torch.nn.parallel import DistributedDataParallel as DDP
    from fragnet_b200.train.fused import FusedFineTuneStep
    from fragnet_b200.train.utils import TrainerFineTune
    from test_gpu_finetune_freeze import _freeze, _loader
    res = {}
    wg = dist.group.WORLD
    # an un-wrapped model without group= under a process group keeps refusing
    try:
        FusedFineTuneStep(_model("FTHead3", "celu", 1, 0.0, W_ODD, 2, SEED0))
        res["no_group"] = None
    except NotImplementedError as ex:
        res["no_group"] = str(ex)
    # broadcast, then three steps on different batches per rank
    m = _model("FTHead3", "celu", 1, 0.0, W_ODD, 2, SEED0 + rank)
    fs = FusedFineTuneStep(m, lr=1e-3, group=wg)
    res["init"], res["peers"] = _state(m), fs._peers is not None
    for hb in _batches(rank):
        fs.step({k: v.cuda() for k, v in hb.items()})
    res["final"] = _state(m)
    # the same from a resumed optimizer whose step counts differ (two runs)
    m = _model("FTHead3", "celu", 1, 0.0, W_ODD, 2, SEED0 + rank)
    fs = FusedFineTuneStep(m, lr=1e-3, group=wg)
    opt = _resume(m)
    fs.attach_optimizer(opt)
    res["runs"] = list(fs._adam_runs)
    for hb in _batches(rank, seed=600):
        fs.step({k: v.cuda() for k, v in hb.items()})
    res["final_runs"] = _state(m)
    res["steps_runs"] = sorted({int(opt.state[p]["step"]) for p in fs.live})
    # a differently frozen model on rank 1: ValueError on every rank, before anything is re-homed
    m = _freeze(_model("FTHead3", "celu", 1, 0.0, W_ODD, 2, SEED0), 1 if rank == 1 else 0)
    try:
        FusedFineTuneStep(m, lr=1e-3, group=wg)
        res["layout"] = None
    except ValueError as ex:
        res["layout"] = str(ex)
    # TrainerFineTune(fused=True) on DDP-wrapped models against the DDP generic loop (p = 0), and validation through
    # the wrapper once the parameters live in the flat buffers
    m1 = _model("FTHead3", "celu", 1, 0.0, W_ODD, 2, 14)
    m2 = copy.deepcopy(m1)
    d1, d2 = DDP(m1, find_unused_parameters=True), DDP(m2, find_unused_parameters=True)
    o1, o2 = torch.optim.Adam(d1.parameters(), lr=1e-3), torch.optim.Adam(d2.parameters(), lr=1e-3)
    t1, t2 = TrainerFineTune(fused=True), TrainerFineTune()
    loader = _loader(20 + rank)
    res["trainer_losses"] = [(t1.train(d1, loader, o1, None, "cuda", loader), t2.train(d2, loader, o2, None, "cuda", loader))
                             for _ in range(2)]
    fs = t1._fused_for(d1, o1, "cuda", "mse")
    res["trainer_fused"] = fs is not None and fs.world_size == world and fs.model is m1 and not t2._fused_steps
    res["trainer_params"] = (_state(m1), _state(m2))
    res["trainer_val"] = (t1.validate(d1, loader, "cuda"), t2.validate(d2, loader, "cuda"))
    res["trainer_step"] = sorted({int(s["step"]) for s in o1.state_dict()["state"].values()})
    return res


@pytest.fixture(scope="module")
def gloo(tmp_path_factory):
    return _spawn("_w_gloo", 2, tmp_path_factory.mktemp("gloo"), "gloo")


def _reference(hbs_per_rank, opt_seed=None):
    """Single process: ``forward_backward`` on each rank's batch, mean of the flat gradients, ``_adam()``."""
    from fragnet_b200.train.fused import FusedFineTuneStep
    m = _model("FTHead3", "celu", 1, 0.0, W_ODD, 2, SEED0)
    fs = FusedFineTuneStep(m, lr=1e-3)
    if opt_seed is not None:
        fs.attach_optimizer(_resume(m, opt_seed))
    for step_batches in zip(*hbs_per_rank):
        grads = []
        for hb in step_batches:
            fs.forward_backward({k: v.cuda() for k, v in hb.items()})
            grads.append(fs.flat_g.clone())
        fs.flat_g.copy_(sum(grads) * (1.0 / len(grads)))
        fs.t += 1
        fs._adam()
    return _state(m)


def _max_rel(a, b):
    return max(rel_err(a[k], b[k]) for k in a if a[k].is_floating_point())


def _differ(a, b):
    return [k for k in b if not torch.equal(a[k], b[k])]


def test_group_is_opt_in(gloo):
    assert all("process group" in r["no_group"] for r in gloo)


def test_broadcast_makes_differently_seeded_models_identical(gloo):
    want = _state(_model("FTHead3", "celu", 1, 0.0, W_ODD, 2, SEED0))
    for rank, r in enumerate(gloo):
        assert not r["peers"]                       # gloo: the all_reduce path
        assert not _differ(r["init"], want), (rank, _differ(r["init"], want))


def test_three_steps_equal_the_mean_gradient_reference(gloo):
    want = _reference([_batches(r) for r in range(2)])
    for rank, r in enumerate(gloo):
        assert _max_rel(r["final"], want) <= 1e-6, (rank, _differ(r["final"], want))
    assert not _differ(gloo[0]["final"], gloo[1]["final"])


def test_resumed_optimizer_with_two_step_counts(gloo):
    want = _reference([_batches(r, seed=600) for r in range(2)], opt_seed=7)
    for rank, r in enumerate(gloo):
        assert len(r["runs"]) == 2 and r["steps_runs"] == [6, 10]
        assert _max_rel(r["final_runs"], want) <= 1e-6, (rank, _differ(r["final_runs"], want))


def test_layout_check_raises_on_every_rank(gloo):
    assert all(r["layout"] is not None and "differ between the ranks" in r["layout"] for r in gloo)


def test_trainer_on_ddp_takes_the_fused_path_and_matches_the_ddp_loop(gloo):
    for r in gloo:
        assert r["trainer_fused"]
        assert all(abs(l1 - l2) <= 1e-5 * abs(l2) for l1, l2 in r["trainer_losses"])
        p1, p2 = r["trainer_params"]
        assert _max_rel(p1, p2) <= 5e-4
        v1, v2 = r["trainer_val"]
        assert abs(v1 - v2) <= 1e-3 * abs(v2)
        assert r["trainer_step"] == [6]               # 2 epochs x 3 batches
    assert not _differ(gloo[0]["trainer_params"][0], gloo[1]["trainer_params"][0])


# ---- the run-table kernel on one GPU: a one-rank peer set ----------------------------------------------------------------
def test_run_table_kernel_on_one_rank():
    """World 1: the mean is the rank's own gradient.  One run gives bitwise ``fnb_allreduce_adam_step``; three runs
    give bitwise ``fnb_adam_step`` per run.  The buffer spans two grid sweeps, so threads cross run boundaries."""
    import ctypes as C
    from fragnet_b200 import _abi, ops
    lib = ops._lib()
    n = 4 * 256 * 148 * 2 + 4 * 37
    gen = torch.Generator(device="cuda").manual_seed(3)
    p0, g = torch.randn(n, device="cuda", generator=gen), torch.randn(n, device="cuda", generator=gen)
    m0 = 0.1 * torch.randn(n, device="cuda", generator=gen)
    v0 = 0.01 * torch.rand(n, device="cuda", generator=gen)
    flags, done = torch.zeros(2, dtype=torch.int32, device="cuda"), torch.zeros(1, dtype=torch.int32, device="cuda")
    ps = _abi.CPeerSet()
    ps.grads[0], ps.flags[0], ps.world, ps.rank = g.data_ptr(), flags.data_ptr(), 1, 0
    hp = (1e-3, 0.9, 0.999, 1e-8, 0.01)
    epoch = [0]

    def runs(table):
        p, m, v = p0.clone(), m0.clone(), v0.clone()
        arr = (_abi.CAdamRun * len(table))(*table)
        epoch[0] += 1
        _abi.check(lib.fnb_allreduce_adam_runs(C.byref(ps), ops._p(p), ops._p(m), ops._p(v), n, arr, len(table), *hp,
                                               epoch[0], ops._p(done), ops._stream()), "runs")
        return p, m, v

    one = runs([(0, n, 5)])
    p, m, v = p0.clone(), m0.clone(), v0.clone()
    epoch[0] += 1
    _abi.check(lib.fnb_allreduce_adam_step(C.byref(ps), ops._p(p), ops._p(m), ops._p(v), n, *hp, 5, epoch[0],
                                           ops._p(done), ops._stream()), "step")
    assert all(torch.equal(a, b) for a, b in zip(one, (p, m, v)))
    table = [(0, 4 * 256 * 148 + 12, 3), (4 * 256 * 148 + 12, n - 40, 1), (n - 40, n, 9)]
    three = runs(table)
    p, m, v = p0.clone(), m0.clone(), v0.clone()
    for lo, hi, step in table:
        _abi.check(lib.fnb_adam_step(ops._p(p[lo:]), ops._p(g[lo:]), ops._p(m[lo:]), ops._p(v[lo:]), hi - lo, *hp, step,
                                     ops._stream()), "adam")
    assert all(torch.equal(a, b) for a, b in zip(three, (p, m, v)))
    assert not torch.equal(three[0], one[0])
    assert int(done) == 0 and flags.tolist() == [epoch[0], epoch[0]]


# ---- ranks: one GPU each, NCCL + the symmetric-memory exchange kernel ----------------------------------------------------
def _gather(t):
    out = [torch.empty_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(out, t)
    return out


def _rank_mean(g):
    """The kernel's mean: sum in rank order from zero, times 1/W in fp32."""
    acc = torch.zeros_like(g)
    for x in _gather(g):
        acc += x
    return acc * (1.0 / dist.get_world_size())


def _w_nccl(rank, world):
    from fragnet_b200.train.fused import FusedFineTuneStep, FusedPretrainStep, finetune_step_class
    from test_gpu_finetune_freeze import _freeze
    from test_gpu_finetune_variants import _batch as _vbatch, _model as _vmodel
    res = {"identical": [], "vs_nccl": [], "runs_bitwise": [], "pretrain_runs_bitwise": [], "variants": {}}
    wg = dist.group.WORLD
    cuda = lambda hb: {k: v.cuda() for k, v in hb.items()}

    def twins(make, step_class, opt=None, **kw):
        m1 = make()
        m2 = copy.deepcopy(m1)
        f1 = step_class(m1, lr=1e-3, group=wg, **kw)
        os.environ["FNB_FUSED_ALLREDUCE"] = "0"
        try:
            f2 = step_class(m2, lr=1e-3, group=wg, **kw)
        finally:
            os.environ["FNB_FUSED_ALLREDUCE"] = "1"
        if opt is not None:
            f1.attach_optimizer(opt(m1))
            f2.attach_optimizer(opt(m2))
        return f1, f2

    # fused exchange against the NCCL path: rank-identical bits after every step, agreement to fp32 rounding
    f1, f2 = twins(lambda: _model("FTHead3", "celu", 1, 0.0, W_ODD, 2, SEED0 + rank), FusedFineTuneStep)
    res["peers"] = (f1._peers is not None, f2._peers is None)
    for hb in _batches(rank):
        f1.step(cuda(hb))
        f2.step(cuda(hb))
        res["identical"].append(all(torch.equal(x, f1.flat_p) for x in _gather(f1.flat_p)))
        res["vs_nccl"].append(rel_err(f1.flat_p, f2.flat_p))
    # two runs: the kernel against _adam() fed the same mean gradient, bit for bit
    f3, f4 = twins(lambda: _model("FTHead3", "celu", 1, 0.0, W_ODD, 2, SEED0), FusedFineTuneStep, opt=_resume)
    res["n_runs"] = len(f3._adam_runs)
    for hb in _batches(rank, seed=600):
        f3.step(cuda(hb))
        f4.flat_g.copy_(_rank_mean(f3.flat_g))
        f4.t += 1
        f4._adam()
        res["runs_bitwise"].append(torch.equal(f3.flat_p, f4.flat_p) and torch.equal(f3.exp_avg_sq, f4.exp_avg_sq))
    # the other model versions and a frozen encoder take a step on the fused exchange
    makers = {"lite": lambda: _vmodel("lite", "FTHead3", "relu", 1, 0.0, W_ODD, 2, SEED0 + rank),
              "edge": lambda: _vmodel("edge", "FTHead3", "relu", 1, 0.0, W_ODD, 2, SEED0 + rank),
              "frozen_encoder": lambda: _freeze(_model("FTHead3", "celu", 1, 0.0, W_ODD, 2, SEED0 + rank), 2)}
    for name, make in makers.items():
        m = make()
        fs = finetune_step_class(m)(m, lr=1e-3, group=wg)
        hb = _vbatch("edge" if name == "edge" else "lite", 1, "mse", 700 + rank)
        loss = fs.step(cuda(hb))
        flat = torch.cat([p.detach().reshape(-1) for p in m.parameters()])
        res["variants"][name] = (fs._peers is not None, bool(torch.isfinite(loss)),
                                 all(torch.equal(x, flat) for x in _gather(flat)))
    # pretraining with two runs: per-run step counts on the fused path too
    import bench
    from fragnet.model.gat.gat2_pretrain import FragNetPreTrain
    torch.manual_seed(1234 + rank)
    pt_batches = [cuda(b) for b in bench.make_batches("unimol", 64, 3, 32, seed=50 + rank)]

    def pt_opt(m):
        opt = torch.optim.Adam(m.parameters(), lr=1e-3)
        for name, p in m.named_parameters():
            if name.startswith("head."):
                opt.state[p] = {"step": torch.tensor(4.0), "exp_avg": torch.zeros_like(p),
                                "exp_avg_sq": torch.zeros_like(p)}
        return opt
    f5, f6 = twins(lambda: FragNetPreTrain(**bench.PT_KW).cuda().train(), FusedPretrainStep, opt=pt_opt)
    res["pretrain_runs"] = len(f5._adam_runs)
    for b in pt_batches:
        torch.manual_seed(9)
        f5.step(b)
        f6.flat_g.copy_(_rank_mean(f5.flat_g))
        f6.t += 1
        f6._adam()
        res["pretrain_runs_bitwise"].append(torch.equal(f5.flat_p, f6.flat_p))
    return res


@pytest.fixture(scope="module")
def nccl(tmp_path_factory):
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs 2 GPUs")
    return _spawn("_w_nccl", min(n, 8), tmp_path_factory.mktemp("nccl"), "nccl")


def test_fused_exchange_is_active_and_rank_identical(nccl):
    for r in nccl:
        assert r["peers"] == (True, True)
        assert all(r["identical"])
        assert max(r["vs_nccl"]) <= 2e-5


def test_run_table_equals_adam_runs_on_the_same_mean_gradient(nccl):
    """Bitwise: the kernel's mean is summed in rank order from zero and scaled by 1/W in fp32, and ``_rank_mean``
    forms the same; the Adam arithmetic is that of ``fnb_adam_step``."""
    for r in nccl:
        assert r["n_runs"] == 2 and all(r["runs_bitwise"])


def test_variants_and_frozen_encoder_take_a_data_parallel_step(nccl):
    for r in nccl:
        assert r["variants"] == {k: (True, True, True) for k in ("lite", "edge", "frozen_encoder")}


def test_pretraining_honours_two_step_counts(nccl):
    for r in nccl:
        assert r["pretrain_runs"] == 2 and all(r["pretrain_runs_bitwise"])
