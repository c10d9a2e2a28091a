"""Grouped barycenters and Wasserstein k-means without a GPU: the host layer of
`sot_b200.barycenter.wasserstein_barycenter_groups` and `sot_b200.cluster.wasserstein_kmeans` with recording stand-ins
for the `_capi` wrappers (the oracle's arithmetic), the refusals (all before any launch) and the ABI's argument
checks."""
import ctypes

import pytest
import torch

from oracle import barycenter_oracle as BO
from tests import fake_kernels
from tests.groups_oracle import barycenter_groups as oracle_groups
from tests.test_pairwise_host import _oracle_dist


def _labels_of(offsets):
    return torch.repeat_interleave(torch.arange(offsets.shape[0] - 1), offsets.diff())


@pytest.fixture
def rec(monkeypatch):
    from sot_b200 import _capi, losses
    calls = []

    def barycenter_groups(x, offsets, w, pos, pos_out, flags):
        calls.append(dict(op="fwd", x=x, offsets=offsets, w=w, pos=pos, pos_out=pos_out, flags=flags))
        return oracle_groups(x, _labels_of(offsets), offsets.shape[0] - 1, pos, w, pos_out,
                                    bool(flags & _capi.SOT_SQUARE)).detach()

    def barycenter_groups_backward(x, offsets, w, pos, pos_out, flags, upstream):
        g = torch.arange(x.numel(), dtype=torch.float32).reshape(x.shape)  # distinct rows: the permutation shows
        calls.append(dict(op="bwd", x=x, upstream=upstream, grad=g))
        return g

    def pairwise(u, v, pu, pv, p, flags):
        calls.append(dict(op="cdist", rows=u.shape[1], cols=v.shape[1]))
        return _oracle_dist(u, v, pu, pv, p, flags).detach()

    monkeypatch.setattr(_capi, "barycenter_groups", barycenter_groups)
    monkeypatch.setattr(_capi, "barycenter_groups_backward", barycenter_groups_backward)
    monkeypatch.setattr(_capi, "pairwise", pairwise)
    fake_kernels.allow_cpu_rows(monkeypatch, losses)
    return calls


def _data(R=11, n=9, seed=0):
    gen = torch.Generator().manual_seed(seed)
    x = torch.rand(R, n, generator=gen, dtype=torch.float64) + 0.05
    return x, torch.linspace(0, 1, n)


def test_order_offsets_and_uniform_weights(rec):
    from sot_b200 import barycenter as BC
    x, pos = _data()
    labels = torch.tensor([3, 0, 3, 1, 0, 3, 3, 1, 0, 3, 1])
    out = BC.wasserstein_barycenter_groups(x, labels, 5, pos, square_dist=True)
    assert out.shape == (5, 9) and out.dtype == torch.float32
    c = rec[-1]
    order = torch.tensor([1, 4, 8, 3, 7, 10, 0, 2, 5, 6, 9])  # by group, rows of a group in increasing order
    assert torch.equal(c["x"], x.float()[order]) and c["x"].is_contiguous()
    assert torch.equal(c["offsets"], torch.tensor([0, 3, 6, 6, 11, 11])) and c["offsets"].dtype == torch.int64
    assert c["w"] is None and c["flags"] == 1
    for g in (0, 1, 3):  # weights None: fl32(1 / K_g), the values of torch.full((K,), 1.0 / K)
        rows = x.float()[labels == g]
        K = rows.shape[0]
        want = BO.barycenter(rows[None], torch.full((K,), 1.0 / K), pos, None, True)[0]
        assert torch.equal(out[g], want)
        assert torch.full((K,), 1.0 / K)[0].item() == torch.tensor(1.0 / K, dtype=torch.float32).item()
    assert torch.isnan(out[2]).all() and torch.isnan(out[4]).all()  # empty groups
    w = torch.rand(11, dtype=torch.float64)
    BC.wasserstein_barycenter_groups(x, labels, 5, pos, weights=w, out_pos=torch.linspace(0, 1, 4))
    assert torch.equal(rec[-1]["w"], w.float()[order]) and rec[-1]["pos_out"].shape == (4,)


def test_gradient_rows_go_back_through_the_inverse_permutation(rec):
    from sot_b200 import barycenter as BC
    x, pos = _data()
    labels = torch.tensor([2, 0, 2, 1, 0, 2, 1, 1, 0, 2, 0])
    xs = x.clone().requires_grad_(True)
    out = BC.wasserstein_barycenter_groups(xs, labels, 3, pos)
    out.sum().backward()
    c = rec[-1]
    assert c["op"] == "bwd" and c["upstream"].shape == (3, 9) and c["upstream"].is_contiguous()
    order = torch.argsort(labels, stable=True)
    want = torch.empty_like(c["grad"])
    want[order] = c["grad"]  # sorted row k is x row order[k]
    assert torch.equal(xs.grad.float(), want)


def test_unsorted_grid_and_complex_rows_take_the_dense_prologue(rec):
    from sot_b200 import barycenter as BC
    x, pos = _data()
    labels = torch.tensor([0, 1] * 5 + [0])
    perm = torch.randperm(9, generator=torch.Generator().manual_seed(1))
    out = BC.wasserstein_barycenter_groups(x[:, perm], labels, 2, pos[perm])
    assert torch.equal(rec[-1]["pos"], pos) and torch.equal(out, BC.wasserstein_barycenter_groups(x, labels, 2, pos))
    z = torch.polar(x.float(), torch.rand(x.shape))
    BC.wasserstein_barycenter_groups(z, labels, 2, pos)
    assert torch.allclose(rec[-1]["x"], z.abs()[torch.argsort(labels, stable=True)])


def test_empty_inputs(rec):
    from sot_b200 import barycenter as BC
    x, pos = _data()
    none = torch.zeros(0, dtype=torch.int64)
    assert BC.wasserstein_barycenter_groups(x[:0], none, 0, pos).shape == (0, 9)
    out = BC.wasserstein_barycenter_groups(x[:0], none, 3, pos)
    assert out.shape == (3, 9) and torch.isnan(out).all()
    assert torch.equal(rec[-1]["offsets"], torch.zeros(4, dtype=torch.int64))


def test_refusals_happen_before_any_launch(rec):
    from sot_b200 import _capi, barycenter as BC
    x, pos = _data()
    labels = torch.zeros(11, dtype=torch.int64)
    before = _capi.launch_count()
    for bad in (torch.full((11,), 3), torch.full((11,), -1)):
        with pytest.raises(ValueError, match="labels in"):
            BC.wasserstein_barycenter_groups(x, bad, 3, pos)
    with pytest.raises(ValueError, match="integer"):
        BC.wasserstein_barycenter_groups(x, labels.float(), 3, pos)
    with pytest.raises(ValueError, match="integer"):
        BC.wasserstein_barycenter_groups(x, labels[:5], 3, pos)
    with pytest.raises(ValueError, match="n_groups"):
        BC.wasserstein_barycenter_groups(x, labels, -1, pos)
    with pytest.raises(ValueError, match=r"\(R, n\)"):
        BC.wasserstein_barycenter_groups(x[None], labels, 3, pos)
    with pytest.raises(ValueError, match="weights of shape"):
        BC.wasserstein_barycenter_groups(x, labels, 3, pos, weights=torch.ones(3))
    with pytest.raises(NotImplementedError, match="weights"):
        BC.wasserstein_barycenter_groups(x, labels, 3, pos, weights=torch.ones(11, requires_grad=True))
    with pytest.raises(NotImplementedError, match="`pos`"):
        BC.wasserstein_barycenter_groups(x, labels, 3, pos.clone().requires_grad_(True))
    with pytest.raises(NotImplementedError, match="1-D grid"):
        BC.wasserstein_barycenter_groups(x, labels, 3, pos.expand(11, 9).clone())
    with pytest.raises(ValueError, match="ascending"):
        BC.wasserstein_barycenter_groups(x, labels, 3, pos, out_pos=pos.flip(0))
    assert rec == [] and _capi.launch_count() == before


def test_abi_validation_before_any_launch():
    from sot_b200 import _capi
    lib = _capi.load()
    before = _capi.launch_count()
    fake = ctypes.c_void_p(16)

    def prob(G=2, R=3, n=9, M=9, flags=0, ptr=16, weights=16):
        return _capi.SotBarycenterGroupsProblem(G, R, n, M, ptr, ptr, weights, ptr, ptr, flags)

    def fwd(pr, out=fake):
        return lib.sot_barycenter_groups_device(ctypes.byref(pr), out, None)

    def bwd(pr, up=fake, grad=fake):
        return lib.sot_barycenter_groups_backward_device(ctypes.byref(pr), up, grad, None)

    assert lib.sot_barycenter_groups_device(None, fake, None) == -1
    assert lib.sot_barycenter_groups_backward_device(None, fake, fake, None) == -1
    for flags in (_capi.SOT_CUT_SCALE, _capi.SOT_LIMIT, _capi.SOT_RAW_WEIGHTS, _capi.SOT_COMPLEX_INPUT, 64):
        assert fwd(prob(flags=flags)) == -1 and bwd(prob(flags=flags)) == -1
    assert b"SOT_SQUARE" in lib.sot_last_error()
    for bad in (prob(n=0), prob(M=0), prob(G=-1), prob(R=-1), prob(ptr=0)):
        assert fwd(bad) == -1 and bwd(bad) == -1
    assert fwd(prob(), out=None) == -1
    assert bwd(prob(), up=None) == -1 and bwd(prob(), grad=None) == -1
    assert fwd(prob(R=0), out=None) == -1  # (R == 0: the output rows are still written, NaN)
    # R x n at most 2^31 - 1 per call; no cap per group (2^24 is the dense path's)
    assert fwd(prob(R=(1 << 31) // 1025 + 1, n=1025)) == -2 and b"2^31" in lib.sot_last_error()
    assert bwd(prob(R=1 << 21, n=1024)) == -2
    assert fwd(prob(R=1 << 31, n=1)) == -2
    for empty in (prob(G=0), prob(G=0, R=0, ptr=0)):  # no groups: nothing is launched
        assert fwd(empty, out=None) == 0 and bwd(empty, up=None, grad=None) == 0
    assert bwd(prob(R=0), up=None, grad=None) == 0  # no rows: no gradient to write
    assert _capi.launch_count() == before


# ---- k-means host logic, the kernels replaced by the oracle ------------------------------------------------------
def _clusters(seed=0, per=(5, 4, 3), n=17):
    """Rows that are bumps around C centres, far apart on the grid."""
    gen = torch.Generator().manual_seed(seed)
    rows, truth = [], []
    for c, k in enumerate(per):
        for _ in range(k):
            r = torch.full((n,), 1e-3)
            at = 2 + 6 * c + int(torch.randint(0, 2, (1,), generator=gen))
            r[at:at + 2] += torch.rand(2, generator=gen) + 0.5
            rows.append(r)
            truth.append(c)
    return torch.stack(rows), torch.tensor(truth), torch.linspace(0, 1, n)


def test_kmeans_plus_plus_is_deterministic_under_a_seeded_generator(rec):
    from sot_b200 import cluster
    x, truth, pos = _clusters()
    a = cluster.wasserstein_kmeans(x, 3, pos, generator=torch.Generator().manual_seed(3))
    b = cluster.wasserstein_kmeans(x, 3, pos, generator=torch.Generator().manual_seed(3))
    assert torch.equal(a.centroids, b.centroids) and torch.equal(a.labels, b.labels) and a.n_iter == b.n_iter
    assert a.inertia == b.inertia
    # the planted clusters come back up to a permutation, and the result is the fixed point
    assert all(len(set(a.labels[truth == c].tolist())) == 1 for c in range(3))
    assert len(set(a.labels.tolist())) == 3
    rows = x / x.sum(1, keepdim=True)
    cdist = torch.stack([torch.tensor([float(_oracle_dist(r[None, None], c[None, None], pos, pos, 2.0, 0))
                                       for c in a.centroids]) for r in rows])
    assert torch.equal(torch.argmin(cdist, 1), a.labels)
    assert torch.equal(a.centroids, oracle_groups(rows, a.labels, 3, pos))
    assert abs(a.inertia - cdist.min(1).values.double().sum().item()) <= 1e-5


def test_kmeans_ties_go_to_the_lowest_index_and_it_stops_when_labels_settle(rec):
    from sot_b200 import cluster
    x, truth, pos = _clusters()
    rows = x / x.sum(1, keepdim=True)
    init = torch.stack((rows[0], rows[0], rows[9]))  # clusters 0 and 1 equal: every tie goes to 0
    r = cluster.wasserstein_kmeans(x, 3, pos, init=init, n_iter=1)
    assert r.n_iter == 1
    first = [c for c in rec if c["op"] == "cdist"]
    assert first and all(c["cols"] == 3 for c in first)
    # after the first assignment cluster 1 was empty: it was re-seeded with the farthest row, so the labels changed
    assert (r.labels == 1).any()
    full = cluster.wasserstein_kmeans(x, 3, pos, init=init, n_iter=50)
    assert full.n_iter < 50
    again = cluster.wasserstein_kmeans(x, 3, pos, init=full.centroids, n_iter=50)
    assert again.n_iter == 1 and torch.equal(again.labels, full.labels)  # one update step: the labels did not change


def test_kmeans_reseeds_an_empty_cluster_with_the_farthest_row(rec, monkeypatch):
    from sot_b200 import cluster
    x, truth, pos = _clusters()
    rows = x / x.sum(1, keepdim=True)
    far = torch.zeros(17)
    far[1] = 1.0  # a centroid no row is near
    init = torch.stack((rows[0], far, rows[9]))
    seen = []
    real = cluster.barycenter.wasserstein_barycenter_groups
    monkeypatch.setattr(cluster.barycenter, "wasserstein_barycenter_groups",
                        lambda *a, **k: seen.append(a[1].clone()) or real(*a, **k))
    r = cluster.wasserstein_kmeans(x, 3, pos, init=init, n_iter=2)
    assert not (seen[0] == 1).any()  # cluster 1 empty after the first assignment
    d0 = torch.stack([torch.tensor([float(_oracle_dist(q[None, None], c[None, None], pos, pos, 2.0, 0))
                                    for c in init]) for q in rows])
    m, lab = d0.min(1)
    want = int(torch.argsort(m, descending=True, stable=True)[0])  # the row farthest from its own centroid
    assert (seen[1] == 1).any() and int(seen[1][want]) == 1
    assert r.n_iter == 2


def test_kmeans_refusals(rec):
    from sot_b200 import cluster
    x, _, pos = _clusters()
    with pytest.raises(ValueError, match="8448"):
        cluster.wasserstein_kmeans(torch.rand(4, 8449), 2, torch.linspace(0, 1, 8449))
    with pytest.raises(ValueError, match="n_clusters"):
        cluster.wasserstein_kmeans(x, 0, pos)
    with pytest.raises(ValueError, match="n_clusters"):
        cluster.wasserstein_kmeans(x, 13, pos)
    with pytest.raises(ValueError, match="init"):
        cluster.wasserstein_kmeans(x, 3, pos, init="random")
    with pytest.raises(ValueError, match="init of shape"):
        cluster.wasserstein_kmeans(x, 3, pos, init=x[:2])
    assert rec == []
