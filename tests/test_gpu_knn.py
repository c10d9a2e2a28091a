"""GPU: exact k nearest neighbours (`sot_b200.pairwise.wasserstein_knn`) against the first k columns of a stable sort
of `wasserstein_cdist` with the same options -- values bit for bit, indices exactly."""
import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
CAP = 128


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


def _check(PW, x, y, px, py, k, **opts):
    got = PW.wasserstein_knn(x, y, k, px, py, **opts)
    D = PW.wasserstein_cdist(x, y, px, py, **opts)
    want_v, want_i = torch.sort(D, dim=-1, stable=True)
    assert got.values.dtype == torch.float32 and got.indices.dtype == torch.int64
    assert got.values.shape == D.shape[:-1] + (k,)
    wv, gv = want_v[..., :k], got.values
    assert torch.equal(torch.isnan(gv), torch.isnan(wv))
    assert torch.equal(gv.nan_to_num(0.0).view(torch.int32), wv.nan_to_num(0.0).view(torch.int32))
    assert torch.equal(got.indices, want_i[..., :k])
    return got


@pytest.mark.parametrize("k", [1, 7, CAP])
@pytest.mark.parametrize("limit", [False, True])
@pytest.mark.parametrize("cut", [False, True])
@pytest.mark.parametrize("p,square", [(1, False), (2, True), (2, False), (3, True)])
def test_contract_against_sorted_cdist(PW, p, square, cut, limit, k):
    x, y, px, py = _spectra(37, 300, seed=3)
    _check(PW, x, y, px, py, k, p=p, square_dist=square, dont_normalize=cut, limit_quantile_range=limit)


@pytest.mark.parametrize("cut", [False, True])
def test_different_bin_counts_and_batches(PW, cut):
    x, y, px, py = _spectra(48, 160, n_fft=512, n_fft_y=1024, seed=5)
    _check(PW, x, y, px, py, 9, p=2, square_dist=True, dont_normalize=cut)
    xb, yb = x.reshape(3, 16, -1), y.reshape(2, 80, -1)[:1].expand(3, 80, -1).contiguous()
    got = _check(PW, xb, yb, px, py, 5, p=2, square_dist=True, dont_normalize=cut)
    for b in range(3):
        one = PW.wasserstein_knn(xb[b], yb[b], 5, px, py, p=2, square_dist=True, dont_normalize=cut)
        assert torch.equal(one.values, got.values[b]) and torch.equal(one.indices, got.indices[b])


def test_duplicates_rank_the_lower_index_first_and_queries_in_the_database(PW):
    x, y, px, py = _spectra(20, 200, seed=7)
    y[50:60] = y[10:20]        # exact duplicates of rows 10..19
    y[100:120] = x            # the queries themselves: zero distances
    y[150:160] = x[:10]       # and again, at higher indices
    got = _check(PW, x, y, px, py, 12, p=2, square_dist=True)
    assert torch.all(got.values[:, 0] == 0) and torch.equal(got.indices[:, 0].cpu(), torch.arange(100, 120))
    _check(PW, x, y, px, py, 3, p=1)


def test_zero_mass_and_nan_rows(PW):
    x, y, px, py = _spectra(24, 180, seed=9)
    y[5] = 0.0                 # no mass: no bound, always walked
    y[77] = 0.0
    x[3] = 0.0
    y[40, 17] = float("nan")   # NaN rows rank last
    y[120, 3] = float("nan")
    x[6, 2] = float("nan")
    for opts in (dict(p=2, square_dist=True), dict(p=1), dict(p=2, square_dist=True, dont_normalize=True)):
        _check(PW, x, y, px, py, 7, **opts)
        _check(PW, x, y, px, py, CAP, **opts)


def test_repeated_calls_give_the_same_bits(PW):
    x, y, px, py = _spectra(64, 2048, seed=11)
    a = PW.wasserstein_knn(x, y, 10, px, py, p=2, square_dist=True)
    for _ in range(2):
        b = PW.wasserstein_knn(x, y, 10, px, py, p=2, square_dist=True)
        assert torch.equal(a.values, b.values) and torch.equal(a.indices, b.indices)


def test_empty_inputs(PW):
    x, y, px, py = _spectra(4, 20)
    r = PW.wasserstein_knn(x[:0], y, 3, px, py)
    assert r.values.shape == (0, 3) and r.indices.shape == (0, 3)
    r = PW.wasserstein_knn(x[None, :0], y[None], 3, px, py)
    assert r.values.shape == (1, 0, 3)
    r = PW.wasserstein_knn(x[None][:0], y[None][:0], 3, px, py)
    assert r.values.shape == (0, 4, 3)


def test_cuda_graph_replay_of_the_c_entry_point(PW):
    from sot_b200 import _capi
    x, y, px, py = _spectra(40, 500, seed=13)
    u, v = x[None].contiguous(), y[None].contiguous()
    eager = _capi.pairwise_knn(u, v, px, py, 2.0, _capi.SOT_SQUARE, 10, want_walked=True)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        _capi.pairwise_knn(u, v, px, py, 2.0, _capi.SOT_SQUARE, 10)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = _capi.pairwise_knn(u, v, px, py, 2.0, _capi.SOT_SQUARE, 10, want_walked=True)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out[0], eager[0]) and torch.equal(out[1], eager[1])
    assert 0 < out[2].item() <= 40 * 500


def test_pruning_is_active_on_spectra(PW):
    from sot_b200 import _capi, synthetic as S
    x, _ = S.sot_batch(16, 2048, seed=1, device=DEV)
    y1, y2 = S.sot_batch(256, 2048, seed=2, device=DEV)
    x = x.reshape(-1, 1025)[:256].contiguous()
    y = torch.cat([y1.reshape(-1, 1025), y2.reshape(-1, 1025)])[:8192].contiguous()
    g = S.linear_positions(2048).to(DEV)
    vals, idx, walked = _capi.pairwise_knn(x[None], y[None], g, g, 2.0, _capi.SOT_SQUARE, 10, want_walked=True)
    D = PW.wasserstein_cdist(x, y, g, g, p=2, square_dist=True)
    wv, wi = torch.sort(D, dim=-1, stable=True)
    assert torch.equal(vals[0], wv[:, :10]) and torch.equal(idx[0], wi[:, :10])
    frac = walked.item() / (256 * 8192)
    assert 0 < frac < 0.10, frac
    # cut mode: no bound, every pair walked
    _, _, walked = _capi.pairwise_knn(x[None], y[None], g, g, 2.0, _capi.SOT_SQUARE | _capi.SOT_CUT_SCALE, 10,
                                      want_walked=True)
    assert walked.item() == 256 * 8192


def test_1024_queries_against_65536_frames(PW):
    from sot_b200 import synthetic as S
    x, _ = S.sot_batch(64, 2048, seed=21, device=DEV)
    _, y = S.sot_batch(4096, 2048, seed=22, device=DEV)
    x, y = x.reshape(-1, 1025), y.reshape(-1, 1025)
    g = S.linear_positions(2048).to(DEV)
    assert x.shape[0] == 1024 and y.shape[0] == 65536
    _check(PW, x, y, g, g, 10, p=2, square_dist=True)
