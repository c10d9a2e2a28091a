"""GPU: exact radius search (`sot_b200.pairwise.wasserstein_radius`) against `(wasserstein_cdist(...) <= r).nonzero()`
with the same options -- values bit for bit, indices exactly -- and `cluster.wasserstein_dbscan` against the dense
oracle of its definition on `wasserstein_cdist(x, x) <= eps`."""
import ctypes
import math

import numpy as np
import pytest
import torch

from tests.dbscan_oracle import oracle

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


@pytest.fixture(scope="module")
def PW():
    from sot_b200 import pairwise
    return pairwise


def _spectra(P, R, n_fft=512, seed=0, n_fft_y=None):
    from sot_b200 import synthetic as S
    Fx, Fy = n_fft // 2 + 1, (n_fft_y or n_fft) // 2 + 1
    x, _ = S.sot_batch((P + 15) // 16, n_fft, seed=seed)
    _, y = S.sot_batch((R + 15) // 16, n_fft_y or n_fft, seed=seed + 1)
    return (x.reshape(-1, Fx)[:P].contiguous().to(DEV), y.reshape(-1, Fy)[:R].contiguous().to(DEV),
            S.linear_positions(n_fft).to(DEV), S.linear_positions(n_fft_y or n_fft).to(DEV))


def _check(PW, x, y, px, py, r, **opts):
    got = PW.wasserstein_radius(x, y, r, px, py, **opts)
    D = PW.wasserstein_cdist(x, y, px, py, **opts)
    mask = D <= torch.tensor(r, dtype=torch.float32)
    assert got.values.dtype == torch.float32 and got.indices.dtype == torch.int64
    assert torch.equal(got.indices, mask.nonzero())
    assert torch.equal(got.values.view(torch.int32), D[mask].view(torch.int32))
    return got


def _radii(PW, x, y, px, py, **opts):
    """0, the median distance to the nearest and to the 10th nearest row of y, and +inf"""
    v = PW.wasserstein_knn(x, y, 10, px, py, **opts).values.reshape(-1, 10)
    return [0.0, v[:, 0].nanmedian().item(), v[:, 9].nanmedian().item(), math.inf]


@pytest.mark.parametrize("limit", [False, True])
@pytest.mark.parametrize("cut", [False, True])
@pytest.mark.parametrize("p,square", [(1, False), (1, True), (2, False), (2, True), (3, False), (3, True)])
def test_contract_against_masked_cdist(PW, p, square, cut, limit):
    x, y, px, py = _spectra(37, 300, seed=3)
    opts = dict(p=p, square_dist=square, dont_normalize=cut, limit_quantile_range=limit)
    for r in _radii(PW, x, y, px, py, **opts):
        _check(PW, x, y, px, py, r, **opts)


@pytest.mark.parametrize("cut", [False, True])
def test_different_bin_counts_and_batches(PW, cut):
    x, y, px, py = _spectra(48, 160, n_fft=512, n_fft_y=1024, seed=5)
    opts = dict(p=2, square_dist=True, dont_normalize=cut)
    r = _radii(PW, x, y, px, py, **opts)[2]
    _check(PW, x, y, px, py, r, **opts)
    xb, yb = x.reshape(3, 16, -1), y.reshape(2, 80, -1)[:1].expand(3, 80, -1).contiguous()
    r = _radii(PW, xb, yb, px, py, **opts)[2]
    got = _check(PW, xb, yb, px, py, r, **opts)
    assert got.indices.shape[1] == 3 and got.values.numel() > 0
    for b in range(3):
        one = PW.wasserstein_radius(xb[b], yb[b], r, px, py, **opts)
        sel = got.indices[:, 0] == b
        assert torch.equal(one.indices, got.indices[sel][:, 1:]) and torch.equal(one.values, got.values[sel])


def test_duplicates_and_queries_in_the_database(PW):
    x, y, px, py = _spectra(20, 200, seed=7)
    y[50:60] = y[10:20]        # exact duplicates of rows 10..19
    y[100:120] = x             # the queries themselves: zero distances
    y[150:160] = x[:10]        # and again, at higher indices
    got = _check(PW, x, y, px, py, 0.0, p=2, square_dist=True)
    pairs = set(map(tuple, got.indices.tolist()))
    assert {(i, 100 + i) for i in range(20)} <= pairs and {(i, 150 + i) for i in range(10)} <= pairs
    for r in _radii(PW, x, y, px, py, p=1)[1:3]:
        _check(PW, x, y, px, py, r, p=1)


def test_zero_mass_and_nan_rows(PW):
    x, y, px, py = _spectra(24, 180, seed=9)
    y[5] = 0.0                 # no mass: no bound, always walked
    y[77] = 0.0
    x[3] = 0.0
    y[40, 17] = float("nan")   # NaN distances are never within the radius
    y[120, 3] = float("nan")
    x[6, 2] = float("nan")
    for opts in (dict(p=2, square_dist=True), dict(p=1), dict(p=2, square_dist=True, dont_normalize=True)):
        for r in _radii(PW, x, y, px, py, **opts):
            got = _check(PW, x, y, px, py, r, **opts)
            assert not torch.any(got.indices[:, 0] == 6) and not torch.any(got.indices[:, 1] == 40)


def test_repeated_calls_give_the_same_bits(PW):
    x, y, px, py = _spectra(64, 2048, seed=11)
    r = _radii(PW, x, y, px, py, p=2, square_dist=True)[2]
    a = PW.wasserstein_radius(x, y, r, px, py, p=2, square_dist=True)
    for _ in range(2):
        b = PW.wasserstein_radius(x, y, r, px, py, p=2, square_dist=True)
        assert torch.equal(a.values, b.values) and torch.equal(a.indices, b.indices)


def _c_radius(u, v, px, py, p, flags, radius, capacity, guard=0):
    """The C entry point on buffers of capacity + guard entries filled with sentinels."""
    from sot_b200 import _capi
    prob = _capi.pairwise_problem(u, v, px, py, p, flags)
    rows = torch.full((capacity + guard,), -5, dtype=torch.int64, device=DEV)
    cols = torch.full((capacity + guard,), -5, dtype=torch.int64, device=DEV)
    values = torch.full((capacity + guard,), -5.0, device=DEV)
    count = torch.full((1,), 7, dtype=torch.int64, device=DEV)
    walked = torch.full((1,), 7, dtype=torch.int64, device=DEV)
    rc = _capi.load().sot_pairwise_radius_device(ctypes.byref(prob), radius, capacity, _capi._ptr(rows),
                                                 _capi._ptr(cols), _capi._ptr(values), _capi._ptr(count),
                                                 _capi._ptr(walked), _capi._stream(u.device))
    assert rc == 0, _capi.load().sot_last_error()
    torch.cuda.synchronize()
    return rows, cols, values, count, walked


def test_count_only_and_short_capacity_calls(PW):
    from sot_b200 import _capi
    x, y, px, py = _spectra(40, 500, seed=13)
    u, v = x[None].contiguous(), y[None].contiguous()
    r = _radii(PW, x, y, px, py, p=2, square_dist=True)[2]
    D = PW.wasserstein_cdist(x, y, px, py, p=2, square_dist=True)
    mask = D <= torch.tensor(r, dtype=torch.float32)
    E = int(mask.sum())
    assert E > 10
    rows, _, _, count, walked = _c_radius(u, v, px, py, 2.0, _capi.SOT_SQUARE, r, 0, guard=16)
    assert count.item() == E and 0 < walked.item() <= 40 * 500
    assert torch.all(rows == -5)  # nothing written
    rows, cols, values, count, _ = _c_radius(u, v, px, py, 2.0, _capi.SOT_SQUARE, r, E - 3, guard=64)
    assert count.item() == E  # counted in full, nothing written at or past the capacity
    assert torch.all(rows[E - 3:] == -5) and torch.all(cols[E - 3:] == -5) and torch.all(values[E - 3:] == -5.0)
    rows, cols, values, count, _ = _c_radius(u, v, px, py, 2.0, _capi.SOT_SQUARE, r, E + 40, guard=8)
    hits = mask.nonzero()
    assert count.item() == E and torch.equal(rows[:E], hits[:, 0]) and torch.equal(cols[:E], hits[:, 1])
    assert torch.equal(values[:E], D[mask]) and torch.all(rows[E + 40:] == -5)


def test_empty_problems_set_the_count_to_zero(PW):
    from sot_b200 import _capi
    x, y, px, py = _spectra(4, 20)
    before = _capi.launch_count()
    for u, v in ((x[None, :0], y[None]), (x[None], y[None, :0]), (x[None][:0], y[None][:0])):
        _, _, _, count, walked = _c_radius(u.contiguous(), v.contiguous(), px, py, 1.0, 0, 1.0, 0)
        assert count.item() == 0 and walked.item() == 0
    assert _capi.launch_count() == before
    r = PW.wasserstein_radius(x[:0], y, 1.0, px, py)
    assert r.values.shape == (0,) and r.indices.shape == (0, 2)
    r = PW.wasserstein_radius(x[None], y[None, :0], 1.0, px, py)
    assert r.values.shape == (0,) and r.indices.shape == (0, 3)


def test_cuda_graph_replay_of_the_c_entry_point(PW):
    from sot_b200 import _capi
    x, y, px, py = _spectra(40, 500, seed=13)
    u, v = x[None].contiguous(), y[None].contiguous()
    r = _radii(PW, x, y, px, py, p=2, square_dist=True)[2]
    eager = _capi.pairwise_radius(u, v, px, py, 2.0, _capi.SOT_SQUARE, r, 4096)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        _capi.pairwise_radius(u, v, px, py, 2.0, _capi.SOT_SQUARE, r, 4096)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = _capi.pairwise_radius(u, v, px, py, 2.0, _capi.SOT_SQUARE, r, 4096, want_walked=True)
    graph.replay()
    torch.cuda.synchronize()
    E = eager[3].item()
    assert 0 < E <= 4096 and out[3].item() == E
    for a, b in zip(out[:3], eager[:3]):
        assert torch.equal(a[:E], b[:E])
    assert 0 < out[4].item() <= 40 * 500


def test_pruning_is_active_on_spectra(PW):
    from sot_b200 import _capi, synthetic as S
    x, _ = S.sot_batch(16, 2048, seed=1, device=DEV)
    y1, y2 = S.sot_batch(256, 2048, seed=2, device=DEV)
    x = x.reshape(-1, 1025)[:256].contiguous()
    y = torch.cat([y1.reshape(-1, 1025), y2.reshape(-1, 1025)])[:8192].contiguous()
    g = S.linear_positions(2048).to(DEV)
    r = _radii(PW, x, y, g, g, p=2, square_dist=True)[1]
    _, _, _, count, walked = _capi.pairwise_radius(x[None], y[None], g, g, 2.0, _capi.SOT_SQUARE, r, 1 << 16,
                                                   want_walked=True)
    D = PW.wasserstein_cdist(x, y, g, g, p=2, square_dist=True)
    assert count.item() == int((D <= torch.tensor(r, dtype=torch.float32)).sum())
    frac = walked.item() / (256 * 8192)
    assert 0 < frac < 0.10, frac
    _, _, _, _, walked = _capi.pairwise_radius(x[None], y[None], g, g, 2.0, _capi.SOT_SQUARE, math.inf, 0,
                                               want_walked=True)
    assert walked.item() == 256 * 8192  # +inf never prunes
    # cut mode: no bound, every pair walked
    _, _, _, _, walked = _capi.pairwise_radius(x[None], y[None], g, g, 2.0, _capi.SOT_SQUARE | _capi.SOT_CUT_SCALE, r,
                                               0, want_walked=True)
    assert walked.item() == 256 * 8192


def test_1024_queries_against_65536_frames(PW):
    from sot_b200 import synthetic as S
    x, _ = S.sot_batch(64, 2048, seed=21, device=DEV)
    _, y = S.sot_batch(4096, 2048, seed=22, device=DEV)
    x, y = x.reshape(-1, 1025), y.reshape(-1, 1025)
    g = S.linear_positions(2048).to(DEV)
    assert x.shape[0] == 1024 and y.shape[0] == 65536
    r = _radii(PW, x, y, g, g, p=2, square_dist=True)[2]
    got = _check(PW, x, y, g, g, r, p=2, square_dist=True)
    assert got.values.numel() >= 1024 * 5


@pytest.mark.parametrize("p,square", [(2, False), (1, True)])
def test_dbscan_matches_the_dense_oracle(PW, p, square):
    from sot_b200 import cluster, synthetic as S
    x, y = S.sot_batch(128, 512, seed=31, device=DEV)
    x = torch.cat([x.reshape(-1, 257), y.reshape(-1, 257)[:1000]])  # 3048 rows, two populations
    x[17] = float("nan")
    pos = S.linear_positions(512).to(DEV)
    eps = PW.wasserstein_knn(x, x, 20, pos, pos, p=p, square_dist=square).values[:, 19].nanmedian().item()
    got = cluster.wasserstein_dbscan(x, eps, 12, pos, p=p, square_dist=square)
    D = PW.wasserstein_cdist(x, x, pos, pos, p=p, square_dist=square)
    labels, core, n = oracle((D <= torch.tensor(eps, dtype=torch.float32)).cpu().numpy(), 12)
    assert np.array_equal(got.core.cpu().numpy(), core) and np.array_equal(got.labels.cpu().numpy(), labels)
    assert got.n_clusters == n and n >= 1 and got.labels[17] == -1
    assert 0 < int((got.labels == -1).sum()) < x.shape[0]
