"""DBSCAN over spectra without a GPU: `sot_b200.cluster.wasserstein_dbscan` with the radius search replaced by a given
neighbour relation A, against a NumPy / SciPy oracle of its definition (and scikit-learn's DBSCAN where A is
symmetric), and the round count of the connected components on long chains."""
import math

import numpy as np
import pytest
import torch

from tests.dbscan_oracle import oracle


@pytest.fixture
def graph(monkeypatch):
    """Row r of x is the number r; the stand-in radius search returns the edges (i, j) of the current relation, given
    as an edge list sorted by (i, j), for the query rows it is handed, in `wasserstein_radius`'s layout."""
    from sot_b200 import pairwise
    state = {}

    def wasserstein_radius(xq, x, eps, x_pos, y_pos, p=1, square_dist=False, **kw):
        state["calls"].append(dict(P=xq.shape[0], R=x.shape[0], eps=eps, p=p, square_dist=square_dist))
        src, dst = state["edges"]
        rows = xq[:, 0].long()
        if rows.numel() == 0:
            keep = torch.zeros_like(src, dtype=torch.bool)
        else:
            keep = (src >= rows[0]) & (src <= rows[-1])
        ind = torch.stack([src[keep] - (rows[0] if rows.numel() else 0), dst[keep]], 1)
        return pairwise.RadiusResult(torch.zeros(ind.shape[0]), ind)

    monkeypatch.setattr(pairwise, "wasserstein_radius", wasserstein_radius)

    def run(A=None, edges=None, R=None, min_samples=1, **kw):
        from sot_b200 import cluster
        if A is not None:
            R = A.shape[0]
            edges = torch.as_tensor(np.stack(np.nonzero(A)))
        order = torch.argsort(edges[0] * R + edges[1])
        state["edges"] = (edges[0][order], edges[1][order])
        state["calls"] = []
        x = torch.arange(R, dtype=torch.float32)[:, None]
        return cluster.wasserstein_dbscan(x, 0.5, min_samples, torch.zeros(1), **kw)

    run.state = state
    return run


def _check(run, A, min_samples):
    got = run(A, min_samples=min_samples)
    labels, core, n = oracle(A, min_samples)
    assert got.labels.dtype == torch.int64 and got.core.dtype == torch.bool
    assert np.array_equal(got.core.numpy(), core)
    assert np.array_equal(got.labels.numpy(), labels)
    assert got.n_clusters == n
    return got


def _random_relation(R, p, seed, symmetric):
    rng = np.random.default_rng(seed)
    A = rng.random((R, R)) < p
    if symmetric:
        A = A | A.T
    np.fill_diagonal(A, True)
    return A


@pytest.mark.parametrize("seed", range(6))
@pytest.mark.parametrize("min_samples", [1, 2, 4, 7])
def test_random_symmetric_relations_match_the_oracle_and_scikit_learn(graph, seed, min_samples):
    A = _random_relation(120, 0.015 * (seed + 1), seed, symmetric=True)
    got = _check(graph, A, min_samples)
    sklearn = pytest.importorskip("sklearn.cluster")
    D = np.where(A, 0.0, 2.0)
    want = sklearn.DBSCAN(eps=1.0, min_samples=min_samples, metric="precomputed").fit(D)
    assert np.array_equal(got.labels.numpy(), want.labels_)
    core = np.zeros(120, dtype=bool)
    core[want.core_sample_indices_] = True
    assert np.array_equal(got.core.numpy(), core)


@pytest.mark.parametrize("seed", range(6))
def test_asymmetric_relations_match_the_oracle(graph, seed):
    A = _random_relation(150, 0.02 * (seed + 1), seed + 100, symmetric=False)
    A[np.arange(150) % 11 == 3] = False  # some rows that are nobody's neighbour, not even their own (NaN rows)
    _check(graph, A, 3)


def test_all_noise_a_single_cluster_and_min_samples_one(graph):
    R = 50
    A = np.eye(R, dtype=bool)
    got = _check(graph, A, 2)  # every row its own only neighbour: noise
    assert got.n_clusters == 0 and torch.all(got.labels == -1) and not got.core.any()
    got = _check(graph, A, 1)  # min_samples = 1: every row is a cluster of its own
    assert got.n_clusters == R and torch.equal(got.labels, torch.arange(R))
    got = _check(graph, np.ones((R, R), dtype=bool), R)
    assert got.n_clusters == 1 and torch.all(got.labels == 0) and got.core.all()
    got = _check(graph, np.zeros((R, R), dtype=bool), 1)  # no row is its own neighbour (all NaN)
    assert got.n_clusters == 0 and torch.all(got.labels == -1)


def test_a_border_row_between_two_clusters_takes_the_lower_label(graph):
    # two dense groups 0..4 and 6..10 (core at min_samples = 5), row 5 reached by both, row 11 by the second only, and
    # the second group's lowest row listed first by its members: clusters are numbered by their lowest core row
    R = 12
    A = np.eye(R, dtype=bool)
    for grp in (range(0, 5), range(6, 11)):
        for i in grp:
            for j in grp:
                A[i, j] = True
    A[[2, 8], 5] = True
    A[9, 11] = True
    A[5, 11] = True  # (5 is not core: it lends no cluster)
    got = _check(graph, A, 5)
    assert got.labels.tolist() == [0] * 5 + [0] + [1] * 5 + [1]
    A2 = A[::-1, ::-1].copy()  # mirrored: the border row now sits next to the group whose label is higher
    got = _check(graph, A2, 5)
    assert got.labels.tolist() == [0] + [0] * 5 + [0] + [1] * 5


def test_query_blocks_cover_every_row(graph, monkeypatch):
    from sot_b200 import cluster
    monkeypatch.setattr(cluster, "_DBSCAN_BLOCK", 120 * 7)  # seven query rows per radius call
    A = _random_relation(120, 0.03, 5, symmetric=False)
    _check(graph, A, 3)
    calls = graph.state["calls"]
    assert [c["P"] for c in calls] == [7] * 17 + [1] and all(c["R"] == 120 for c in calls)
    assert calls[0]["eps"] == 0.5 and calls[0]["p"] == 2 and calls[0]["square_dist"] is False


@pytest.mark.parametrize("shuffle", [False, True])
def test_a_chain_of_100000_rows_converges_in_logarithmic_rounds(graph, shuffle):
    from sot_b200 import cluster
    R = 100_000
    perm = torch.randperm(R, generator=torch.Generator().manual_seed(3)) if shuffle else torch.arange(R)
    a, b = perm[:-1], perm[1:]  # chain perm[0] - perm[1] - ... in either direction
    src, dst = torch.cat([a, b, torch.arange(R)]), torch.cat([b, a, torch.arange(R)])
    label, rounds = cluster._components(R, src, dst)
    assert torch.all(label == 0)
    assert rounds <= 2 * math.ceil(math.log2(R)), rounds
    got = graph(edges=torch.stack([src, dst]), R=R, min_samples=3)
    # the two ends have two neighbours (themselves and one): border rows of the one cluster
    assert got.n_clusters == 1 and torch.all(got.labels == 0)
    assert int(got.core.sum()) == R - 2 and not got.core[perm[0]] and not got.core[perm[-1]]


def test_refusals():
    from sot_b200 import cluster
    x, pos = torch.rand(5, 4), torch.linspace(0, 1, 4)
    for eps in (float("nan"), "1", None, 1j):
        with pytest.raises(ValueError, match="eps"):
            cluster.wasserstein_dbscan(x, eps, 2, pos)
    for ms in (0, -1, 1.5, True):
        with pytest.raises(ValueError, match="min_samples"):
            cluster.wasserstein_dbscan(x, 0.1, ms, pos)
    with pytest.raises(ValueError, match="must be"):
        cluster.wasserstein_dbscan(x[None], 0.1, 2, pos)
    with pytest.raises(ValueError, match="pos"):
        cluster.wasserstein_dbscan(x, 0.1, 2, pos[:3])


def test_no_rows(graph):
    got = graph(edges=torch.zeros(2, 0, dtype=torch.int64), R=0, min_samples=2)
    assert got.labels.shape == (0,) and got.core.shape == (0,) and got.n_clusters == 0
