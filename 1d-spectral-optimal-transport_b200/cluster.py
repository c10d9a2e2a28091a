"""Wasserstein k-means over spectra: Lloyd's algorithm in the W2 geometry of the SOT loss.

`wasserstein_kmeans(x, n_clusters, pos)` clusters the rows of `x` by their spectral shape.  The assignment step is
`pairwise.wasserstein_cdist` (W2^2 from every row to every centroid, nothing materialised) and the update step is
`barycenter.wasserstein_barycenter_groups` (the W2 barycenter of each cluster, whatever its size, in one call).  Two
harmonic spectra whose f0 differs average to one peak at the averaged frequency, so a centroid is a spectrum of the
cluster's shape, not a blur of its members.

Everything runs in the mass domain: each row is normalised once to a distribution (of x^2 with `square_dist`), so a
centroid, which is a distribution on `pos`, is compared with the rows as they are.  CUDA only, like the rest of the
package.
"""
from __future__ import annotations

from typing import NamedTuple

import torch

from . import _capi, barycenter, losses, pairwise

__all__ = ["KMeansResult", "wasserstein_kmeans"]

_BLOCK = 1 << 24  # entries of one (rows x centroids) block of the assignment step


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
