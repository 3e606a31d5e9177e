"""Per-kernel parity of the CUDA path (through the C ABI) against the CPU oracle / plain torch fp32."""
import pytest
import torch
import torch.nn.functional as F

from conftest import FP32_REL_TOL, rel_err

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("n,K", [(1, 128), (77, 128), (1000, 167), (333, 17), (65, 6), (4097, 128), (9000, 128),
                                 (9000, 167)])
def test_projection_forward_backward(n, K):
    from fragnet_b200 import ops
    g = torch.Generator().manual_seed(n * 1000 + K)
    x = torch.randn(n, K, generator=g)
    W = torch.randn(128, K, generator=g) * 0.2
    b = torch.randn(128, generator=g)
    alpha = torch.randn(4, 96, generator=g)
    h, S = ops.proj_fwd(x.cuda(), W.cuda(), b.cuda(), alpha.cuda(), 96, 0, 64)
    href = F.linear(x, W, b)
    assert rel_err(h, href) <= FP32_REL_TOL
    hv = href.view(n, 4, 32)
    Sref = torch.cat([(hv * alpha[:, 0:32]).sum(-1), (hv * alpha[:, 64:96]).sum(-1)], dim=1)
    assert rel_err(S, Sref) <= FP32_REL_TOL
    dh = torch.randn(n, 128, generator=g)
    dx, dW, db = ops.proj_bwd(x.cuda(), W.cuda(), dh.cuda(), True)
    assert rel_err(dx, dh @ W) <= FP32_REL_TOL
    assert rel_err(dW, dh.t() @ x) <= FP32_REL_TOL
    assert rel_err(db, dh.sum(0)) <= FP32_REL_TOL
    assert rel_err(ops.node_scalars(h, alpha.cuda(), 96, 0, 64), Sref) <= FP32_REL_TOL


def test_projection_forward_beyond_65535_row_tiles():
    # 65 538 tiles of 64 rows: more than a grid's y dimension holds, so the GEMM's row tiles must be on x
    from fragnet_b200 import ops
    n, K, m = 4_194_400, 128, 3000
    g = torch.Generator(device="cuda").manual_seed(11)
    x = torch.randn(n, K, device="cuda", generator=g)
    W = torch.randn(128, K, device="cuda", generator=g) * 0.2
    b = torch.randn(128, device="cuda", generator=g)
    alpha = torch.randn(4, 96, device="cuda", generator=g)
    h, S = ops.proj_fwd(x, W, b, alpha, 96, 0, 64)
    for rows in (slice(0, m), slice(n - m, n)):
        href = F.linear(x[rows].double(), W.double(), b.double())
        assert rel_err(h[rows], href) <= FP32_REL_TOL
        hv = href.view(m, 4, 32)
        ad = alpha.double()
        Sref = torch.cat([(hv * ad[:, 0:32]).sum(-1), (hv * ad[:, 64:96]).sum(-1)], dim=1)
        assert rel_err(S[rows], Sref) <= FP32_REL_TOL


def test_segment_sum_and_gather():
    from fragnet_b200 import ops
    gen = torch.Generator().manual_seed(4)
    ids = torch.randint(0, 50, (700,), generator=gen)
    ids[:50] = torch.arange(50)
    x = torch.randn(700, 128, generator=gen)
    pool = ops.csr_build(ids.cuda(), None, 50, reverse=False)
    alpha = torch.randn(4, 192, generator=gen)
    out, S = ops.segment_sum(pool.rowptr, pool.col, 50, x.cuda(), alpha=alpha.cuda(), alpha_stride=192, off_t=0, off_s=160)
    ref = torch.zeros(50, 128).index_add_(0, ids, x)
    assert rel_err(out, ref) <= FP32_REL_TOL
    rv = ref.view(50, 4, 32)
    Sref = torch.cat([(rv * alpha[:, 0:32]).sum(-1), (rv * alpha[:, 160:192]).sum(-1)], 1)
    assert rel_err(S, Sref) <= FP32_REL_TOL
    base = torch.randn(700, 128, generator=gen)
    got = ops.segment_gather(out, 128, ops.narrow_index(ids.cuda()), 700, base.cuda())
    assert rel_err(got, base + ref[ids]) <= FP32_REL_TOL
    # contiguous (readout) form writing into a strided [G,256] buffer
    sorted_ids = torch.sort(ids).values
    ptr = ops.segment_offsets(sorted_ids.cuda(), 50)
    wide = torch.zeros(50, 256, device="cuda")
    ops.segment_sum(ptr, None, 50, x.cuda(), out=wide[:, 128:], out_stride=256)
    assert rel_err(wide[:, 128:], torch.zeros(50, 128).index_add_(0, sorted_ids, x)) <= FP32_REL_TOL
    assert float(wide[:, :128].abs().max()) == 0.0


def test_dropout_relu_statistics_and_backward():
    from fragnet_b200 import ops
    x = torch.randn(1000, 128, device="cuda")
    y_eval = ops.dropout_relu_fwd(x, 0.2, False, True, 0, 0)
    assert torch.equal(y_eval, torch.relu(x))
    y = ops.dropout_relu_fwd(x, 0.2, True, True, 123, 0)
    y2 = ops.dropout_relu_fwd(x, 0.2, True, True, 123, 0)
    y3 = ops.dropout_relu_fwd(x, 0.2, True, True, 123, 32000)
    assert torch.equal(y, y2) and not torch.equal(y, y3)
    pos = x > 0
    kept = (y > 0)[pos].float().mean().item()
    assert abs(kept - 0.8) < 0.01
    assert torch.allclose(y[y > 0], (x / 0.8)[y > 0])
    dy = torch.randn_like(x)
    dx = ops.dropout_relu_bwd(dy, y, 0.2, True)
    assert torch.allclose(dx, torch.where(y > 0, dy / 0.8, torch.zeros_like(dy)))
    odd = torch.randn(333, 167, device="cuda")[:, :167].contiguous()
    d = ops.dropout_relu_fwd(odd, 0.5, True, False, 9, 0)
    frac = (d != 0).float().mean().item()
    assert abs(frac - 0.5) < 0.02 and torch.allclose(d[d != 0], (odd * 2)[d != 0])


@pytest.mark.parametrize("n,K", [(5000, 167), (9001, 17), (777, 6), (3, 167)])
def test_rowsparse_projection_on_one_hot_features(n, K):
    """Layer-0 inputs are one-hot groups (features.py:43-139): the row-sparse kernels must equal the dense fp32 result."""
    from fragnet_b200 import ops
    g = torch.Generator().manual_seed(n + K)
    x = torch.zeros(n, K)
    for _ in range(min(K, 9)):                       # ~9 non-zeros per row, some of them not 1.0
        x[torch.arange(n), torch.randint(0, K, (n,), generator=g)] = 1.0
    x[:, K - 1] = torch.randint(0, 5, (n,), generator=g).float()
    W = torch.randn(128, K, generator=g) * 0.2
    b = torch.randn(128, generator=g)
    alpha = torch.randn(4, 192, generator=g)
    h, S = ops.proj_fwd(x.cuda(), W.cuda(), b.cuda(), alpha.cuda(), 192, 0, 160)
    href = F.linear(x, W, b)
    assert rel_err(h, href) <= FP32_REL_TOL
    hv = href.view(n, 4, 32)
    Sref = torch.cat([(hv * alpha[:, 0:32]).sum(-1), (hv * alpha[:, 160:192]).sum(-1)], dim=1)
    assert rel_err(S, Sref) <= FP32_REL_TOL
    dh = torch.randn(n, 128, generator=g)
    _, dW, _ = ops.proj_bwd(x.cuda(), W.cuda(), dh.cuda(), False, want_db=False)
    assert rel_err(dW, dh.t() @ x) <= 2e-5
    _, dW2, _ = ops.proj_bwd(x.cuda(), W.cuda(), dh.cuda(), False, want_db=False)
    assert torch.equal(dW, dW2)                      # deterministic


def test_segment_sum_and_gather_with_empty_segments_over_several_grid_sweeps():
    """Readouts have segments without members (leading, interior runs, trailing), and batches have more segments than
    one grid sweep covers: k_segment_sum runs one warp per segment on at most 148 x 8 CTAs of 8 warps (9 472 segments
    per sweep), k_segment_gather one thread per float4 on at most 148 x 16 CTAs (18 944 rows per sweep)."""
    from fragnet_b200 import ops
    gen = torch.Generator().manual_seed(12)
    n_seg, n_rows = 3 * 9472 + 17, 2 * 18944 + 9
    empty = torch.zeros(n_seg, dtype=torch.bool)
    empty[:5] = True
    empty[1000:1100] = True
    empty[::7] = True
    empty[-20:] = True
    members = (~empty).nonzero().flatten()
    ids = members[torch.randint(0, members.numel(), (n_rows,), generator=gen)]
    x = torch.randn(n_rows, 128, generator=gen)
    alpha = torch.randn(4, 192, generator=gen)
    ref = torch.zeros(n_seg, 128, dtype=torch.float64).index_add_(0, ids, x.double())
    assert torch.equal(ref[empty].abs().sum(1) == 0, torch.ones(int(empty.sum()), dtype=torch.bool))
    rv = ref.view(n_seg, 4, 32)
    a64 = alpha.double()
    Sref = torch.cat([(rv * a64[:, 0:32]).sum(-1), (rv * a64[:, 160:192]).sum(-1)], 1)

    pool = ops.csr_build(ids.cuda(), None, n_seg, reverse=False)
    out, S = ops.segment_sum(pool.rowptr, pool.col, n_seg, x.cuda(), alpha=alpha.cuda(), alpha_stride=192, off_t=0,
                             off_s=160)
    assert rel_err(out, ref) <= FP32_REL_TOL and rel_err(S, Sref) <= FP32_REL_TOL
    assert float(out[empty.cuda()].abs().max()) == 0.0 and float(S[empty.cuda()].abs().max()) == 0.0
    base = torch.randn(n_rows, 128, generator=gen)
    got = ops.segment_gather(out, 128, ops.narrow_index(ids.cuda()), n_rows, base.cuda())
    assert torch.equal(got, base.cuda() + out[ids.cuda()])
    assert rel_err(got, base.double() + ref[ids]) <= FP32_REL_TOL
    # contiguous (readout) form, offsets built over the gaps
    sorted_ids = torch.sort(ids).values
    ptr = ops.segment_offsets(sorted_ids.cuda(), n_seg)
    assert torch.equal(ptr.cpu().long(), torch.cat([torch.zeros(1, dtype=torch.long),
                                                    torch.bincount(ids, minlength=n_seg).cumsum(0)]))
    out2, _ = ops.segment_sum(ptr, None, n_seg, x[torch.sort(ids).indices].cuda())
    assert rel_err(out2, ref) <= FP32_REL_TOL and float(out2[empty.cuda()].abs().max()) == 0.0


@pytest.mark.parametrize("n,K", [(2 * 9472 + 5, 167), (2 * 18944 + 3, 17)])
def test_rowsparse_projection_over_several_grid_sweeps(n, K):
    """k_proj_rowsparse_fwd covers 4 rows per warp and at most 148 x 2 CTAs of 8 warps at K = 167 (86 KB of staged
    weights: 9 472 rows per sweep), 148 x 4 at K = 17 (18 944 rows per sweep): these row counts make every warp loop."""
    from fragnet_b200 import ops
    g = torch.Generator().manual_seed(n + K)
    x = torch.zeros(n, K)
    for _ in range(9):
        x[torch.arange(n), torch.randint(0, K, (n,), generator=g)] = 1.0
    x[:, K - 1] = torch.randint(0, 5, (n,), generator=g).float()
    x[n // 3] = 0.0                                  # a row without non-zeros: the bias alone
    W = torch.randn(128, K, generator=g) * 0.2
    b = torch.randn(128, generator=g)
    alpha = torch.randn(4, 192, generator=g)
    h, S = ops.proj_fwd(x.cuda(), W.cuda(), b.cuda(), alpha.cuda(), 192, 0, 160)
    href = F.linear(x.double(), W.double(), b.double())
    assert rel_err(h, href) <= FP32_REL_TOL
    assert torch.equal(h[n // 3].cpu(), b)
    hv = href.view(n, 4, 32)
    a64 = alpha.double()
    Sref = torch.cat([(hv * a64[:, 0:32]).sum(-1), (hv * a64[:, 160:192]).sum(-1)], dim=1)
    assert rel_err(S, Sref) <= FP32_REL_TOL
