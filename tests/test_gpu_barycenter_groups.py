"""GPU: grouped barycenters (`sot_b200.barycenter.wasserstein_barycenter_groups`) against the dense call on each group,
bit for bit, and Wasserstein k-means (`sot_b200.cluster.wasserstein_kmeans`)."""
import math

import pytest
import torch

from tests.test_gpu_barycenter import _grids

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


@pytest.fixture(scope="module")
def BC():
    from sot_b200 import barycenter
    return barycenter


def _rows(R, n_fft=512, seed=3):
    from sot_b200 import synthetic as S
    x, y = S.sot_batch(-(-R // 32), n_fft, seed=seed)
    return torch.cat((x, y), 1).reshape(-1, n_fft // 2 + 1)[:R].contiguous(), S.linear_positions(n_fft)


def _labels(sizes, seed=0):
    """Labels of groups of the given sizes, shuffled."""
    lab = torch.repeat_interleave(torch.arange(len(sizes)), torch.tensor(sizes))
    return lab[torch.randperm(lab.shape[0], generator=torch.Generator().manual_seed(seed))]


SIZES = [1, 300, 0, 2, 3, 17, 0, 64, 129, 5, 255, 1, 0, 40]  # 1 .. 300 rows, three empty groups


def _dense_group(BC, x, lab, g, w, pos, op, square, up):
    """Value and gradient rows of the dense call on group g's rows, in increasing row order."""
    idx = (lab == g).nonzero()[:, 0]
    K = idx.shape[0]
    wg = torch.full((K,), 1.0 / K, device=DEV) if w is None else w[idx]
    xs = x[idx].clone().requires_grad_(True)
    out = BC.wasserstein_barycenter(xs, wg, pos, op, square_dist=square)
    (out * up[g]).sum().backward()
    return out.detach(), xs.grad, idx


def _grouped(BC, x, lab, G, w, pos, op, square, up):
    xs = x.clone().requires_grad_(True)
    out = BC.wasserstein_barycenter_groups(xs, lab, G, pos, weights=w, out_pos=op, square_dist=square)
    (out * up).sum().backward()
    return out.detach(), xs.grad


@pytest.mark.parametrize("grid", ["same", "coarse", "fine", "uneven"])
@pytest.mark.parametrize("square", [False, True])
@pytest.mark.parametrize("weights", ["uniform", "per_row"])
def test_every_group_equals_the_dense_call_bitwise(BC, weights, square, grid):
    lab = _labels(SIZES, seed=1).to(DEV)
    x, pos = _rows(lab.shape[0])
    x, pos = x.to(DEV), pos.to(DEV)
    op = _grids(pos.cpu())[grid]
    op = None if op is None else op.to(DEV)
    M = pos.shape[0] if op is None else op.shape[0]
    w = None if weights == "uniform" else torch.rand(lab.shape[0], generator=torch.Generator().manual_seed(2)).to(DEV)
    G = len(SIZES)
    up = torch.randn(G, M, generator=torch.Generator().manual_seed(4)).to(DEV)
    out, grad = _grouped(BC, x, lab, G, w, pos, op, square, up)
    assert out.shape == (G, M)
    for g, K in enumerate(SIZES):
        if K == 0:
            assert torch.isnan(out[g]).all()
            continue
        val, gr, idx = _dense_group(BC, x, lab, g, w, pos, op, square, up)
        assert torch.equal(out[g], val), (g, K)
        assert torch.equal(grad[idx], gr), (g, K)


def test_other_groups_do_not_change_a_group_and_calls_repeat(BC):
    lab = _labels(SIZES, seed=5).to(DEV)
    x, pos = _rows(lab.shape[0], seed=6)
    x, pos = x.to(DEV), pos.to(DEV)
    G = len(SIZES)
    up = torch.rand(G, pos.shape[0], generator=torch.Generator().manual_seed(7)).to(DEV)
    full = _grouped(BC, x, lab, G, None, pos, None, True, up)
    again = _grouped(BC, x, lab, G, None, pos, None, True, up)
    assert torch.equal(full[0].nan_to_num(), again[0].nan_to_num()) and torch.equal(full[1], again[1])
    assert torch.equal(torch.isnan(full[0]), torch.isnan(again[0]))  # (the empty groups' NaN rows)
    keep = (lab != 1) & (lab != 8)  # drop the two largest groups' rows
    part = _grouped(BC, x[keep], lab[keep], G, None, pos, None, True, up)
    for g, K in enumerate(SIZES):
        if K and g not in (1, 8):
            assert torch.equal(part[0][g], full[0][g]), g
    assert torch.equal(part[1], full[1][keep])
    few = _grouped(BC, x[lab == 7], torch.zeros(SIZES[7], dtype=torch.int64, device=DEV), 1, None, pos, None, True,
                   up[7:8])
    assert torch.equal(few[0][0], full[0][7]) and torch.equal(few[1], full[1][lab == 7])


def test_a_bad_row_or_weight_poisons_only_its_group(BC):
    lab = _labels(SIZES, seed=8).to(DEV)
    x, pos = _rows(lab.shape[0], seed=9)
    x, pos = x.to(DEV), pos.to(DEV)
    w = torch.rand(lab.shape[0], generator=torch.Generator().manual_seed(1)).to(DEV)
    G = len(SIZES)
    up = torch.ones(G, pos.shape[0], device=DEV)
    clean = _grouped(BC, x, lab, G, w, pos, None, False, up)
    bad_x, bad_w = x.clone(), w.clone()
    bad_x[(lab == 3).nonzero()[1, 0], 40] = float("nan")
    bad_w[(lab == 9).nonzero()[0, 0]] = -0.5
    out, grad = _grouped(BC, bad_x, lab, G, bad_w, pos, None, False, up)
    for g, K in enumerate(SIZES):
        rows = lab == g
        if g in (3, 9) or K == 0:
            assert torch.isnan(out[g]).all(), g
            assert torch.isnan(grad[rows]).all(), g
        else:
            assert torch.equal(out[g], clean[0][g]) and torch.equal(grad[rows], clean[1][rows]), g


def test_cuda_graph_replays_forward_and_backward_to_the_eager_bits(BC):
    lab = _labels(SIZES, seed=10).to(DEV)
    x, pos = _rows(lab.shape[0], seed=11)
    x, pos = x.to(DEV), pos.to(DEV)
    G = len(SIZES)
    up = torch.rand(G, pos.shape[0], device=DEV)
    xs = x.clone().requires_grad_(True)

    def step():
        out = BC.wasserstein_barycenter_groups(xs, lab, G, pos, square_dist=True)
        return out.detach(), torch.autograd.grad((up * out.nan_to_num()).sum(), xs)[0]

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        eager = [t.clone() for t in step()]
    torch.cuda.current_stream().wait_stream(side)
    # (the labels' range check reads the device: capture the launches behind it)
    from sot_b200 import barycenter as B
    order = torch.argsort(lab, stable=True)
    inverse = torch.argsort(order)
    offsets = torch.zeros(G + 1, dtype=torch.int64, device=DEV)
    offsets[1:] = torch.cumsum(torch.bincount(lab, minlength=G), 0)
    flags = 1
    p = pos.contiguous()

    def captured():
        out = B._Groups.apply(xs, order, inverse, offsets, None, p, p, flags)
        return out.detach(), torch.autograd.grad((up * out.nan_to_num()).sum(), xs)[0]

    with torch.cuda.stream(side):
        captured()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = captured()
    with torch.no_grad():
        xs.zero_()
    graph.replay()
    with torch.no_grad():
        xs.copy_(x)
    graph.replay()
    torch.cuda.synchronize()
    assert all(torch.equal(s, t) for s, t in zip(out[1:], eager[1:]))
    same = ~torch.isnan(eager[0])
    assert torch.equal(out[0][same], eager[0][same]) and torch.isnan(out[0][~same]).all()


def test_empty_inputs_on_the_device(BC):
    x, pos = _rows(4)
    x, pos = x.to(DEV), pos.to(DEV)
    none = torch.zeros(0, dtype=torch.int64, device=DEV)
    xs = x[:0].clone().requires_grad_(True)
    out = BC.wasserstein_barycenter_groups(xs, none, 3, pos)
    assert out.shape == (3, 257) and torch.isnan(out).all()
    out.nan_to_num().sum().backward()
    assert xs.grad.shape == (0, 257)
    assert BC.wasserstein_barycenter_groups(x[:0], none, 0, pos).shape == (0, 257)


# ---- a group past the dense path's 2^24 entries: 20 000 rows x 1025 bins ----------------------------------------------
BIG = 20000


def test_a_big_group_of_one_spectrum_is_that_spectrum(BC):
    x, pos = _rows(8, n_fft=2048, seed=12)
    one = x[3]
    rows = one.to(DEV).expand(BIG, -1).contiguous()
    lab = torch.zeros(BIG, dtype=torch.int64, device=DEV)
    lab[:5] = 1  # a small group in front
    out = BC.wasserstein_barycenter_groups(rows, lab, 2, pos.to(DEV), square_dist=True).double().cpu()
    want = (one.double() ** 2 / (one.double() ** 2).sum()).cumsum(0)
    assert (out[0].cumsum(0) - want).abs().max() <= 1e-6
    assert (out[1].cumsum(0) - want).abs().max() <= 1e-6
    with pytest.raises(ValueError, match="2\\^24"):
        BC.wasserstein_barycenter(rows[5:], torch.full((BIG - 5,), 1.0 / (BIG - 5), device=DEV), pos.to(DEV))


def test_a_big_group_of_diracs_is_one_split_dirac(BC):
    n = 1025
    pos = torch.linspace(0, 1, n)
    at = torch.randint(100, 900, (BIG,), generator=torch.Generator().manual_seed(13))
    rows = torch.zeros(BIG, n)
    rows[torch.arange(BIG), at] = 1.0
    lab = torch.zeros(BIG, dtype=torch.int64)
    out = BC.wasserstein_barycenter_groups(rows.to(DEV), lab.to(DEV), 1, pos.to(DEV))[0].double().cpu()
    z = pos.double()[at].mean().item()
    h = 1.0 / (n - 1)
    b = int(math.floor(z / h))
    want = torch.zeros(n, dtype=torch.float64)
    want[b], want[b + 1] = (b + 1) * h / h - z / h, z / h - b
    # z is rounded to float32 once (an ulp of z near 0.5 is 6e-8, 6e-5 of a bin at 1025 bins)
    assert (out - want).abs().max() <= 2e-4, (out.nonzero(), b, z)
    assert abs(out.sum().item() - 1.0) <= 1e-6 and out.count_nonzero() <= 2


# ---- k-means ------------------------------------------------------------------------------------------------------------
def _planted(per=40, f0s=(180.0, 650.0, 1500.0), seed=14):
    from sot_b200 import synthetic as S
    gen = torch.Generator().manual_seed(seed)
    f0 = torch.tensor(f0s).repeat_interleave(per)[:, None]
    f0 = f0 * (1.0 + 0.04 * (torch.rand(f0.shape, generator=gen) - 0.5))
    audio, _ = S.harmonic_signals(f0.shape[0], gen, n_partials=1, f0=f0)
    spec = S.stft_magnitude(audio, 512)[:, 2]
    truth = torch.arange(len(f0s)).repeat_interleave(per)
    perm = torch.randperm(f0.shape[0], generator=gen)
    return spec[perm].contiguous(), truth[perm], S.linear_positions(512)


def test_kmeans_recovers_planted_clusters_at_a_fixed_point(BC):
    from sot_b200 import cluster, pairwise
    x, truth, pos = _planted()
    x, pos = x.to(DEV), pos.to(DEV)
    r = cluster.wasserstein_kmeans(x, 3, pos, square_dist=True, generator=torch.Generator().manual_seed(0))
    assert r.centroids.shape == (3, 257) and r.labels.shape == (120,) and r.n_iter < 50
    lab = r.labels.cpu()
    for c in range(3):
        assert len(set(lab[truth == c].tolist())) == 1, c
    assert len(set(lab.tolist())) == 3
    w = x * x
    rows = w / w.sum(1, keepdim=True)
    d = pairwise.wasserstein_cdist(rows, r.centroids, pos, pos, p=2)
    assert torch.equal(torch.argmin(d, 1), r.labels)
    assert torch.equal(BC.wasserstein_barycenter_groups(rows, r.labels, 3, pos), r.centroids)
    assert abs(r.inertia - d.min(1).values.double().sum().item()) <= 1e-6 * max(1.0, r.inertia)
    again = cluster.wasserstein_kmeans(x, 3, pos, square_dist=True, generator=torch.Generator().manual_seed(0))
    assert torch.equal(again.centroids, r.centroids) and torch.equal(again.labels, r.labels)
    assert again.inertia == r.inertia and again.n_iter == r.n_iter
