"""GPU: pairwise SOT distances (`sot_b200.pairwise.wasserstein_cdist`) against the oracle on the materialised pairs.

Gates (DESIGN §2): without the cutoff every entry within rel 1e-5 of the reference's formula in float64, or within
1.5 x the reference's own float32 deviation from it (P3, per entry as for the split-frame path); with the cutoff the
mean over all entries as close to the float64 value as the reference's own float32 value is, x 1.5 (P4); gradients of
(G * D).sum() through `_assert_grad_gate` at ratio 3, the small-fixture setting.
"""
import pytest
import torch

from oracle import sot_oracle as O
from tests import golden_io as G
from tests.test_gpu_parity import _assert_grad_gate

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


@pytest.fixture(scope="module")
def PW():
    from sot_b200 import pairwise
    return pairwise


def _materialised(x, y):
    """(P, n), (R, m) -> the P * R pairs as rows, pair (i, j) at i * R + j."""
    P, R = x.shape[0], y.shape[0]
    return (x[:, None].expand(P, R, x.shape[1]).reshape(-1, x.shape[1]),
            y[None].expand(P, R, y.shape[1]).reshape(-1, y.shape[1]))


def _opts(kw):
    return dict(p=kw["p"], square_dist=kw["square"], dont_normalize=kw["cut_scale"],
                limit_quantile_range=kw["limit"])


def _check_values(mine, x, y, px, py, kw):
    X, Y = _materialised(x, y)
    ref = O.sot_per_frame(X, Y, px, py, stable=True, **kw).reshape(mine.shape)
    r64 = O.sot_per_frame(X.double(), Y.double(), px.double(), py.double(), stable=True, **kw).reshape(mine.shape)
    mine = mine.cpu()
    if not kw["limit"]:
        # every entry within 1e-5 of the float64 value, or as close to it as the reference's own float32 value is
        # (the per-frame gate of the split-frame path, whose CDF stage the pre-pass runs)
        tol = torch.maximum(torch.full_like(r64, 1e-5), 1.5 * (ref.double() - r64).abs() / r64.abs())
        err = (mine.double() - r64).abs()
        assert (err <= tol * r64.abs() + 1e-12).all(), (err / r64.abs()).max().item()
        return
    ref64 = r64.mean().item()
    tol = max(1e-5, 1.5 * abs(ref.mean().item() - ref64) / abs(ref64))
    assert abs(mine.double().mean().item() - ref64) <= tol * abs(ref64), (mine.mean().item(), ref64)


def _case(name):
    g = G.load(name)
    F = g["x"].shape[-1]
    kw = G.oracle_kwargs(g["meta"]["ctor"])
    kw.pop("require_sort")
    return g["x"].reshape(-1, F), g["y"].reshape(-1, F), g["pos_x"], g["pos_y"], kw


@pytest.mark.parametrize("name", G.MODULE_CASES)
@pytest.mark.parametrize("limit", [False, True])
def test_values_on_the_fixtures(PW, name, limit):
    x, y, px, py, kw = _case(name)
    kw["limit"] = limit
    mine = PW.wasserstein_cdist(x.to(DEV), y.to(DEV), px.to(DEV), py.to(DEV), **_opts(kw))
    assert mine.shape == (x.shape[0], y.shape[0]) and mine.dtype == torch.float32
    _check_values(mine, x, y, px, py, kw)


@pytest.mark.parametrize("cut", [False, True])
def test_values_with_different_bin_counts(PW, cut):
    from sot_b200 import synthetic as S
    x, _ = S.sot_batch(1, 512, seed=3)
    _, y = S.sot_batch(1, 1024, seed=4)
    x, y = x.reshape(-1, 257)[:12], y.reshape(-1, 513)[:10]
    px, py = S.linear_positions(512), S.linear_positions(1024)
    kw = dict(p=2, square=True, cut_scale=cut, limit=cut)
    mine = PW.wasserstein_cdist(x.to(DEV), y.to(DEV), px.to(DEV), py.to(DEV), **_opts(kw))
    _check_values(mine, x, y, px, py, kw)


@pytest.mark.parametrize("cut", [False, True])
@pytest.mark.parametrize("square", [False, True])
@pytest.mark.parametrize("name", ["sot512_nocut", "sot2048_nocut"])
def test_gradients_vs_fp64_oracle(PW, name, cut, square):
    x, y, px, py, kw = _case(name)
    x, y = x[:10], y[:12]
    kw.update(square=square, cut_scale=cut, limit=cut)
    Gm = torch.rand(x.shape[0], y.shape[0], generator=torch.Generator().manual_seed(5), dtype=torch.float64)
    xd, yd = x.to(DEV).requires_grad_(True), y.to(DEV).requires_grad_(True)
    D = PW.wasserstein_cdist(xd, yd, px.to(DEV), py.to(DEV), **_opts(kw))
    (Gm.float().to(DEV) * D).sum().backward()
    X, Y = _materialised(x, y)
    up = Gm.reshape(-1)
    _, gx32, gy32 = O.sot_loss_and_grads(X, Y, px, py, upstream=up.float(), stable=True, **kw)
    _, gx64, gy64 = O.sot_loss_and_grads(X.double(), Y.double(), px.double(), py.double(), upstream=up, stable=True,
                                         **kw)
    P, R = x.shape[0], y.shape[0]
    fold_x = lambda g: g.reshape(P, R, -1).sum(1)  # noqa: E731
    fold_y = lambda g: g.reshape(P, R, -1).sum(0)  # noqa: E731
    _assert_grad_gate(xd.grad.cpu(), fold_x(gx32), fold_x(gx64), f"{name} cut={cut} sq={square} dx", ratio=3)
    _assert_grad_gate(yd.grad.cpu(), fold_y(gy32), fold_y(gy64), f"{name} cut={cut} sq={square} dy", ratio=3)


def _sample(seed=0, P=9, R=11, n_fft=512):
    from sot_b200 import synthetic as S
    x, y = S.sot_batch(1, n_fft, seed=seed)
    F = n_fft // 2 + 1
    return x.reshape(-1, F)[:P].to(DEV), y.reshape(-1, F)[:R].to(DEV), S.linear_positions(n_fft).to(DEV)


@pytest.mark.parametrize("cut", [False, True])
def test_identical_rows_have_an_exactly_zero_diagonal(PW, cut):
    x, _, g = _sample()
    D = PW.wasserstein_cdist(x, x, g, g, p=2, square_dist=True, dont_normalize=cut, limit_quantile_range=cut)
    assert torch.all(torch.diagonal(D) == 0)
    assert torch.all(D + torch.eye(D.shape[0], device=DEV) > 0)


def test_scaling_x_by_a_power_of_two_is_bit_identical(PW):
    x, y, g = _sample()
    D = PW.wasserstein_cdist(x, y, g, g, p=2, square_dist=True)
    for k in (-7, 5):
        assert torch.equal(PW.wasserstein_cdist(x * 2.0 ** k, y, g, g, p=2, square_dist=True), D)


@pytest.mark.parametrize("cut", [False, True])
def test_batched_call_equals_per_batch_calls_and_runs_repeat_bitwise(PW, cut):
    from sot_b200 import synthetic as S
    x, y = S.sot_batch(3, 512, seed=11)
    x, y = x.to(DEV), y[:, :13].contiguous().to(DEV)  # (3, 16, 257) x (3, 13, 257)
    g = S.linear_positions(512).to(DEV)
    opts = dict(p=2, square_dist=True, dont_normalize=cut, limit_quantile_range=cut)
    Gm = torch.rand(3, 16, 13, device=DEV)

    def run(a, b, up):
        a, b = a.clone().requires_grad_(True), b.clone().requires_grad_(True)
        D = PW.wasserstein_cdist(a, b, g, g, **opts)
        (up * D).sum().backward()
        return D.detach(), a.grad, b.grad

    full = run(x, y, Gm)
    assert all(torch.equal(s, t) for s, t in zip(full, run(x, y, Gm)))  # two runs, same bits
    for b in range(3):
        one = run(x[b], y[b], Gm[b])
        assert all(torch.equal(s[b], t) for s, t in zip(full, one)), b


@pytest.mark.parametrize("cut", [False, True])
def test_nan_rows_poison_like_the_materialised_path(PW, cut):
    from sot_b200 import losses
    x, y, g = _sample(P=6, R=7)
    x[2, 40] = float("nan")
    y[4, 3] = float("nan")
    kw = dict(p=2, square=True, cut_scale=cut, limit=cut)
    Gm = torch.rand(6, 7, device=DEV)
    xd, yd = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
    D = PW.wasserstein_cdist(xd, yd, g, g, **_opts(kw))
    (Gm * D).sum().backward()
    xm, ym = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
    X, Y = _materialised(xm, ym)
    Dm = losses.sot_frames(X, Y, g, g, **kw).reshape(6, 7)
    (Gm * Dm).sum().backward()
    for mine, ref in ((D, Dm), (xd.grad, xm.grad), (yd.grad, ym.grad)):
        assert torch.equal(torch.isnan(mine), torch.isnan(ref))


def test_empty_sides(PW):
    x, y, g = _sample(P=4, R=5)
    for a, b in ((x[:0], y), (x, y[:0])):
        a, b = a.clone().requires_grad_(True), b.clone().requires_grad_(True)
        D = PW.wasserstein_cdist(a, b, g, g, p=2, square_dist=True)
        assert D.shape == (a.shape[0], b.shape[0])
        D.sum().backward()
        assert torch.equal(a.grad, torch.zeros_like(a)) and torch.equal(b.grad, torch.zeros_like(b))
    assert PW.wasserstein_cdist(x[None, :0], y[None], g, g).shape == (1, 0, 5)


@pytest.mark.parametrize("cut", [False, True])
def test_cuda_graph_replays_forward_and_backward_to_the_eager_bits(PW, cut):
    x, y, g = _sample(P=12, R=10)
    opts = dict(p=2, square_dist=True, dont_normalize=cut, limit_quantile_range=cut)
    Gm = torch.rand(12, 10, device=DEV)
    xs, ys = x.clone().requires_grad_(True), y.clone().requires_grad_(True)

    def step():
        D = PW.wasserstein_cdist(xs, ys, g, g, **opts)
        gx, gy = torch.autograd.grad((Gm * D).sum(), (xs, ys))
        return D.detach(), gx, gy

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        eager = [t.clone() for t in step()]
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = step()
    with torch.no_grad():
        xs.zero_()
        ys.zero_()
    graph.replay()
    with torch.no_grad():
        xs.copy_(x)
        ys.copy_(y)
    graph.replay()
    torch.cuda.synchronize()
    assert all(torch.equal(s, t) for s, t in zip(out, eager))


def test_scale_4096_by_4096_at_1025_bins(PW):
    from sot_b200 import losses, synthetic as S
    x, y = S.sot_batch(256, 2048, seed=42, device=DEV)
    x, y = x.reshape(-1, 1025), y.reshape(-1, 1025)  # 4096 rows each: 2 x 68.8 GB of inputs if materialised
    g = S.linear_positions(2048).to(DEV)
    xd, yd = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
    D = PW.wasserstein_cdist(xd, yd, g, g, p=2, square_dist=True)
    (torch.rand_like(D) * D).sum().backward()
    torch.cuda.synchronize()
    assert D.shape == (4096, 4096) and torch.isfinite(D).all()
    assert torch.isfinite(xd.grad).all() and torch.isfinite(yd.grad).all()
    gen = torch.Generator().manual_seed(1)
    i, j = torch.randint(0, 4096, (256,), generator=gen), torch.randint(0, 4096, (256,), generator=gen)
    ref = losses.sot_frames(x[i.to(DEV)], y[j.to(DEV)], g, g, p=2, square=True)
    assert torch.allclose(D[i.to(DEV), j.to(DEV)], ref, rtol=1e-5, atol=0)
