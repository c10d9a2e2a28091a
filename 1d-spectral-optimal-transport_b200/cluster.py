"""Clustering of spectra in the geometry of the SOT loss: Wasserstein k-means and DBSCAN.

`wasserstein_kmeans(x, n_clusters, pos)` clusters the rows of `x` by their spectral shape.  The assignment step is
`pairwise.wasserstein_cdist` (W2^2 from every row to every centroid, nothing materialised) and the update step is
`barycenter.wasserstein_barycenter_groups` (the W2 barycenter of each cluster, whatever its size, in one call).  Two
harmonic spectra whose f0 differs average to one peak at the averaged frequency, so a centroid is a spectrum of the
cluster's shape, not a blur of its members.

k-means runs in the mass domain: each row is normalised once to a distribution (of x^2 with `square_dist`), so a
centroid, which is a distribution on `pos`, is compared with the rows as they are.

`wasserstein_dbscan(x, eps, min_samples, pos)` finds the number of clusters itself and labels outliers as noise: it
is host logic over the neighbour lists of `pairwise.wasserstein_radius`, a self-join of the rows, and connected
components of the core rows by hook-and-shortcut on the device.  CUDA only, like the rest of the package.
"""
from __future__ import annotations

import numbers
from typing import NamedTuple

import torch

from . import _capi, barycenter, losses, pairwise

__all__ = ["KMeansResult", "wasserstein_kmeans", "DBSCANResult", "wasserstein_dbscan"]

_BLOCK = 1 << 24  # entries of one (rows x centroids) block of the assignment step
_DBSCAN_BLOCK = 1 << 28  # pairs of one (query rows x rows) block of the DBSCAN self-join: bounds its hit buffer


class KMeansResult(NamedTuple):
    centroids: torch.Tensor  # (C, n) float32 distributions on `pos`
    labels: torch.Tensor     # (R,) int64
    inertia: float           # sum over the rows of W2^2 to their centroid
    n_iter: int              # update steps run


def _assign(rows, cents, pos):
    """(min W2^2, argmin) of every row over the centroids, lowest index on ties, in blocks of at most _BLOCK."""
    step = max(1, _BLOCK // cents.shape[0])
    dmin, lab = [], []
    for r0 in range(0, rows.shape[0], step):
        d = pairwise.wasserstein_cdist(rows[r0:r0 + step], cents, pos, pos, p=2, require_sort=False)
        m, i = torch.min(d, 1)  # (the first minimal index)
        dmin.append(m)
        lab.append(i)
    return torch.cat(dmin), torch.cat(lab)


def _sample(weights, generator):
    """One index drawn with probability proportional to `weights` (uniformly when they have no mass)."""
    w = weights.double().nan_to_num(0.0).clamp_min(0.0).to(generator.device)
    if not bool(w.sum() > 0):
        w = torch.ones_like(w)
    return int(torch.multinomial(w, 1, generator=generator))


def _kmeans_pp(rows, C, pos, generator):
    """k-means++: the first centroid uniformly, each next one with probability proportional to D^2, the W2^2 to the
    nearest centroid chosen so far."""
    picks = [_sample(torch.ones(rows.shape[0]), generator)]
    d2 = None
    for _ in range(1, C):
        d, _ = _assign(rows, rows[picks[-1]][None], pos)
        d2 = d if d2 is None else torch.minimum(d2, d)
        picks.append(_sample(d2, generator))
    return rows[torch.tensor(picks, device=rows.device)].clone()


def wasserstein_kmeans(x, n_clusters, pos, square_dist=False, n_iter=50, init="k-means++",
                       generator=None) -> KMeansResult:
    """Lloyd's algorithm over the rows of `x` (R, n) in the W2 geometry, `pos` (n,) their grid.

    The rows are normalised once to distributions (of x^2 with `square_dist`; complex rows are reduced to |z|, and a
    row needs positive mass); everything after that runs on them without `square_dist`.  `init` is "k-means++" (D^2
    sampling with `generator`, a torch.Generator on the CPU or on the rows' device; the default generator when None)
    or a (C, n) tensor of starting centroids, distributions on `pos`.  Each iteration assigns every row to its
    nearest centroid by W2^2 (`pairwise.wasserstein_cdist`, p = 2; the lowest index wins a tie) and replaces the
    centroids by the barycenters of their clusters (`barycenter.wasserstein_barycenter_groups`).  A cluster left empty
    is re-seeded with the row farthest from its centroid.  It stops when the labels stop changing, or after `n_iter`
    update steps.  On convergence `labels` is the assignment to `centroids`, and `centroids` are the barycenters of
    `labels`.

    The inertia need not decrease at every step: each barycenter is deposited onto the grid by linear split, so a
    centroid is the W2 mean of its cluster only up to that projection.

    Returns `KMeansResult(centroids (C, n), labels (R,), inertia, n_iter)`.  Rows longer than 8448 bins raise
    `ValueError`, as in `pairwise.wasserstein_cdist`.  The result does not carry gradients."""
    if x.ndim != 2:
        raise ValueError(f"sot_b200: `x` must be (R, n), got {tuple(x.shape)}")
    R, n = x.shape
    C = int(n_clusters)
    if not 1 <= C <= R:
        raise ValueError(f"sot_b200: n_clusters must be in [1, {R}], got {n_clusters}")
    if n > _capi.MAX_PAIRWISE_BINS:
        raise ValueError(f"sot_b200: rows of {n} bins: the limit is {_capi.MAX_PAIRWISE_BINS} bins")
    if pos.shape != (n,):
        raise ValueError(f"sot_b200: `pos` of shape {tuple(pos.shape)} for rows of {n} bins")
    generator = torch.default_generator if generator is None else generator
    with torch.no_grad():
        w = losses._magnitude(x).float()
        w = w * w if square_dist else w
        p, perm = torch.sort(pos.detach().to(device=w.device, dtype=torch.float32), stable=True)
        rows = (w / w.sum(1, keepdim=True)).index_select(1, perm).contiguous()
        if isinstance(init, str):
            if init != "k-means++":
                raise ValueError(f"sot_b200: init must be 'k-means++' or a (C, n) tensor, got {init!r}")
            cents = _kmeans_pp(rows, C, p, generator)
        else:
            if tuple(init.shape) != (C, n):
                raise ValueError(f"sot_b200: init of shape {tuple(init.shape)} for {C} clusters of {n} bins")
            cents = init.detach().to(device=rows.device, dtype=torch.float32).index_select(1, perm).contiguous()
        dmin, labels = _assign(rows, cents, p)
        steps = 0
        for steps in range(1, n_iter + 1):
            cents = barycenter.wasserstein_barycenter_groups(rows, labels, C, p, require_sort=False)
            empty = (torch.bincount(labels, minlength=C) == 0).nonzero()[:, 0]
            if empty.numel():
                far = torch.argsort(dmin, descending=True, stable=True)[:empty.numel()]
                cents[empty] = rows[far]
            dmin, new = _assign(rows, cents, p)
            done = torch.equal(new, labels)
            labels = new
            if done:
                break
        inertia = float(dmin.double().sum())
        return KMeansResult(cents.index_select(1, torch.argsort(perm)), labels, inertia, steps)


class DBSCANResult(NamedTuple):
    labels: torch.Tensor  # (R,) int64: cluster 0, 1, ... or -1 for noise
    core: torch.Tensor    # (R,) bool
    n_clusters: int


def _components(n, src, dst):
    """(label, rounds): label[v] = the lowest vertex of v's connected component in the undirected graph with edges
    src[e] -- dst[e], by hook-and-shortcut.  Each round hooks every root onto the lowest root it has an edge to (a
    `scatter_reduce` min over the edges) and then jumps pointers until every vertex points at its root.  Every tree
    with an edge to another one is hooked or hooked onto, so the trees of a component at least halve per round and a
    chain of n vertices takes O(log n) rounds, not O(n)."""
    label = torch.arange(n, device=src.device)
    rounds = 0
    while True:
        rounds += 1
        a, b = label[src], label[dst]
        hooked = label.scatter_reduce(0, torch.maximum(a, b), torch.minimum(a, b), reduce="amin")
        while True:
            jumped = hooked[hooked]
            if torch.equal(jumped, hooked):
                break
            hooked = jumped
        if torch.equal(hooked, label):
            return label, rounds
        label = hooked


def wasserstein_dbscan(x, eps, min_samples, pos, p=2, square_dist=False) -> DBSCANResult:
    """DBSCAN over the rows of `x` (R, n), `pos` (n,) their grid, under `pairwise.wasserstein_cdist(x, x, pos, pos, p=p,
    square_dist=square_dist)` = D.

    With A[i, j] = (D[i, j] <= eps) (the diagonal of D is exactly 0, so a row is its own neighbour unless it is NaN or
    has no mass): row i is a core row when sum_j A[i, j] >= `min_samples`; clusters are the connected components of the
    core rows, with an edge i -- j when A[i, j] or A[j, i], numbered 0, 1, ... in increasing order of their lowest core
    row; a row that is not core takes the lowest cluster label among the core rows c with A[c, i], and is noise (-1)
    when there is none.  On a symmetric A this is what scikit-learn's `DBSCAN(eps, min_samples=min_samples,
    metric="precomputed")` returns for D.

    The neighbour lists come from `pairwise.wasserstein_radius(x, x, eps, pos, pos, ...)` in blocks of query rows
    (one host read per block) and the components from hook-and-shortcut over them, on the rows' device.  Rows of up to
    8448 bins, as for `wasserstein_cdist`.  Returns `DBSCANResult(labels (R,) int64, core (R,) bool, n_clusters)`; the
    result carries no gradient."""
    if x.ndim != 2:
        raise ValueError(f"sot_b200: `x` must be (R, n), got {tuple(x.shape)}")
    R, n = x.shape
    if tuple(pos.shape) != (n,):
        raise ValueError(f"sot_b200: `pos` of shape {tuple(pos.shape)} for rows of {n} bins")
    if isinstance(eps, bool) or not isinstance(eps, numbers.Real) or eps != eps:
        raise ValueError(f"sot_b200: eps must be a real number and not NaN, got {eps!r}")
    if isinstance(min_samples, bool) or not isinstance(min_samples, numbers.Integral) or min_samples < 1:
        raise ValueError(f"sot_b200: min_samples must be an integer of at least 1, got {min_samples!r}")
    with torch.no_grad():
        src, dst = [], []
        step = max(1, _DBSCAN_BLOCK // max(R, 1))
        for q0 in range(0, R, step):
            hits = pairwise.wasserstein_radius(x[q0:q0 + step], x, eps, pos, pos, p=p, square_dist=square_dist).indices
            src.append(hits[:, 0] + q0)
            dst.append(hits[:, 1])
        dev = x.device if not src else src[0].device
        src = torch.cat(src) if src else torch.empty(0, dtype=torch.int64, device=dev)
        dst = torch.cat(dst) if dst else torch.empty(0, dtype=torch.int64, device=dev)
        core = torch.bincount(src, minlength=R) >= min_samples
        both = core[src] & core[dst]
        root, _ = _components(R, src[both], dst[both])
        roots = torch.unique(root[core])  # (sorted: the lowest core row of each cluster)
        labels = torch.full((R,), -1, dtype=torch.int64, device=dev)
        labels[core] = torch.searchsorted(roots, root[core])
        border = core[src] & ~core[dst]
        reach = torch.full((R,), R, dtype=torch.int64, device=dev)
        reach = reach.scatter_reduce(0, dst[border], labels[src[border]], reduce="amin")
        labels = torch.where(core | (reach == R), labels, reach)
        return DBSCANResult(labels, core, int(roots.numel()))
