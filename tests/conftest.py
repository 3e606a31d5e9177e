import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden", "gat2_golden.pt")
# north_star: "Embeddings, attention weights and predictions must match within 1e-5 relative in fp32"
# measured as max|a-b| / max|b| per tensor (SURVEY.md section 8c).
FP32_REL_TOL = 1e-5


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")
    # The CPU oracle's fp32 reductions are partitioned over the intra-op threads: pin their number so that the
    # reference values do not depend on how many cores the box running the tests happens to have.
    torch.set_num_threads(min(8, torch.get_num_threads()))


@pytest.fixture(autouse=True)
def deterministic_cpu_accumulation(request):
    """CPU tests run with ``torch.use_deterministic_algorithms``: otherwise the fp32 ``index_put_(accumulate=True)`` in
    the oracle's backward (gradients of indexed gathers) adds with parallel atomics, and the order in which colliding
    adds land changes from process to process -- enough, in gradients that cancel to rounding noise, to leave the
    golden vectors (generated with the sequential order) by ~1e-5 relative in about one run out of ten.  GPU tests keep
    the default: several CUDA ops refuse to run in deterministic mode."""
    if "gpu" in request.keywords:
        yield
        return
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev)


def pytest_collection_modifyitems(config, items):
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


def rel_err(a: torch.Tensor, b: torch.Tensor) -> float:
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    assert a.shape == b.shape, (a.shape, b.shape)
    if b.numel() == 0:
        return 0.0
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def grad_errs(pairs, floor=1e-3):
    """Gradient parity metric: per tensor, max|a-b| / max(max|b|, floor * largest gradient entry of the model).

    Some GAT2 gradients are sums that cancel to rounding noise (softmax is shift invariant, so e.g. the bias of the
    edge-attribute embedding only gets the LeakyReLU slope residual: entries ~1e-9 next to ~1e-2 elsewhere); for
    those tensors a pure per-tensor relative error compares noise with noise, hence the floor tied to the model's
    overall gradient scale (1e-3 of it: at 1e-4 the layer-0 edge-embedding weight of the 21-molecule pretraining
    test, max entry 6e-5 in a model whose gradients reach 0.5, sat at 3-7e-5 = 2-4e-9 absolute and crossed the
    tolerance from run to run).  ``pairs``: iterable of (name, got, want).  Returns {name: err}."""
    pairs = [(k, a.detach().double().cpu(), b.detach().double().cpu()) for k, a, b in pairs]
    scale = max((float(b.abs().max()) for _, _, b in pairs if b.numel()), default=0.0)
    out = {}
    for k, a, b in pairs:
        assert a.shape == b.shape, (k, a.shape, b.shape)
        den = max(float(b.abs().max()) if b.numel() else 0.0, floor * scale, 1e-30)
        out[k] = float((a - b).abs().max()) / den if b.numel() else 0.0
    return out


@pytest.fixture(scope="session")
def golden():
    return torch.load(GOLDEN)


@pytest.fixture(scope="session")
def golden_batch():
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    from make_golden import golden_batch as gb
    return gb()
