"""Pairwise SOT distances: the W_p^p matrix between two batches of spectra, the `torch.cdist` of the loss.

`wasserstein_cdist(x, y, x_pos, y_pos)` compares every row of `x` with every row of `y` (nearest-neighbour lookup over
a set of spectra, permutation-invariant losses over sets of sources, sweeps of one target against many candidates)
without materialising the P x R pairs: the kernels behind `sot_pairwise_device` build each row's CDF once and walk
only the merge of each pair.  Entry [b, i, j] is what `losses.sot_frames` gives for the single pair
(x[b, i], y[b, j]) with the same options; the result is differentiable with respect to x and y.

`wasserstein_knn(x, y, k, x_pos, y_pos)` returns each row's k nearest rows of `y` under the same distance, exactly
the first k columns of a stable sort of `wasserstein_cdist`, without forming the matrix and, in the default mode,
without walking the pairs that a lower bound rules out.  `wasserstein_radius(x, y, r, x_pos, y_pos)` returns every
pair within distance r, exactly `(wasserstein_cdist(...) <= r).nonzero()` and its values, pruned by the same bound.

CUDA only, like the rest of the package: there is no CPU or eager fallback.
"""
from __future__ import annotations

import numbers
from typing import NamedTuple

import torch

from . import _capi, losses

__all__ = ["wasserstein_cdist", "wasserstein_knn", "KnnResult", "wasserstein_radius", "RadiusResult"]


class _Cdist(torch.autograd.Function):
    """u (B, P, n), v (B, R, m) -> (B, P, R).  Nothing but the inputs is kept between the passes: the backward
    rebuilds the CDFs (one pass over the rows) and walks every pair again with its upstream value."""

    @staticmethod
    def forward(ctx, u, v, pos_u, pos_v, p, flags):
        ctx.p, ctx.flags = p, flags
        ctx.save_for_backward(u, v, pos_u, pos_v)
        return _capi.pairwise(u, v, pos_u, pos_v, p, flags)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad):
        u, v, pos_u, pos_v = ctx.saved_tensors
        need_u, need_v = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        gu, gv = _capi.pairwise_backward(u, v, pos_u, pos_v, ctx.p, ctx.flags, grad.contiguous().float(), need_u,
                                         need_v)
        return gu, gv, None, None, None, None


def _side(t: torch.Tensor, name: str, batched: bool) -> torch.Tensor:
    if t.ndim != (3 if batched else 2):
        raise ValueError(f"sot_b200: `{name}` must be {'(B, rows, bins)' if batched else '(rows, bins)'} "
                         f"like the other side, got {tuple(t.shape)}")
    return losses._magnitude(t)  # complex rows: |z| in torch (no fused complex prologue here)


def _prologue(x, y, x_pos, y_pos, p, square_dist, dont_normalize, limit_quantile_range, require_sort):
    """The checks and conversions of both entry points: (u (B, P, n), v (B, R, m), pu, pv, flags, batched)."""
    assert p >= 1, f"The OT loss is only valid for p>=1, {p} was given"  # losses.py:271
    batched = x.ndim == 3
    x, y = _side(x, "x", batched), _side(y, "y", batched)
    if batched and x.shape[0] != y.shape[0]:
        raise ValueError(f"sot_b200: batch sizes differ: {x.shape[0]} and {y.shape[0]}")
    for pos, name in ((x_pos, "x_pos"), (y_pos, "y_pos")):
        if pos.ndim != 1:
            raise NotImplementedError(f"sot_b200: `{name}` has shape {tuple(pos.shape)}: pairwise distances take one "
                                      "1-D grid per side (per-row supports are not supported)")
        if pos.requires_grad and torch.is_grad_enabled():
            raise NotImplementedError(f"sot_b200: `{name}` requires a gradient: pairwise distances have no gradient "
                                      "with respect to the support positions (detach them)")
    n, m = x.shape[-1], y.shape[-1]
    if max(n, m) > _capi.MAX_PAIRWISE_BINS:
        raise ValueError(f"sot_b200: pairwise rows of {n} / {m} bins: the limit is {_capi.MAX_PAIRWISE_BINS} bins")
    lead_u, lead_v = x.shape[:-1], y.shape[:-1]
    u, v = losses._rows(x.reshape(-1, n), "x"), losses._rows(y.reshape(-1, m), "y")
    pu, pv = losses._support(x_pos, u, "x_pos"), losses._support(y_pos, v, "y_pos")
    if require_sort:
        pu, u = losses._order(pu, u, x_pos)
        pv, v = losses._order(pv, v, y_pos)
    B = lead_u[0] if batched else 1
    u = u.reshape(B, lead_u[-1], n)
    v = v.reshape(B, lead_v[-1], m)
    return u, v, pu, pv, losses._flags(square_dist, dont_normalize, False, limit_quantile_range), batched


def wasserstein_cdist(x, y, x_pos, y_pos, p=1, square_dist=False, dont_normalize=False, limit_quantile_range=False,
                      require_sort=True) -> torch.Tensor:
    """W_p^p of every pair of rows: `x` (P, n) or (B, P, n) targets, `y` (R, m) or (B, R, m) predictions ->
    (P, R) or (B, P, R) float32, following `torch.cdist`'s batching.  `x_pos` (n,) and `y_pos` (m,) are one grid per
    side (n may differ from m); unsorted grids are sorted once with the columns permuted when `require_sort`.
    Options as in `losses.Wasserstein1D`: `square_dist` (weights = magnitude^2), `dont_normalize` (cut mode: y divided
    by x's mass), `limit_quantile_range` (strict `qs > 1` mask).  float16 / bfloat16 / float64 inputs are converted
    to float32 as `losses.sot_frames` converts them; complex rows are reduced to |z| first."""
    u, v, pu, pv, flags, batched = _prologue(x, y, x_pos, y_pos, p, square_dist, dont_normalize, limit_quantile_range,
                                             require_sort)
    dist = _Cdist.apply(u, v, pu, pv, float(p), flags)
    return dist if batched else dist[0]


class KnnResult(NamedTuple):
    values: torch.Tensor   # float32 (P, k) or (B, P, k)
    indices: torch.Tensor  # int64, rows of `y`


def _no_gradient(x, y, fn: str):
    for t, name in ((x, "x"), (y, "y")):
        if t.requires_grad and torch.is_grad_enabled():
            raise NotImplementedError(f"sot_b200: `{name}` requires a gradient: {fn} has none (detach it, "
                                      "or re-evaluate the selected pairs with wasserstein_cdist or losses.sot_frames "
                                      "to get gradients)")


def wasserstein_knn(x, y, k, x_pos, y_pos, p=1, square_dist=False, dont_normalize=False, limit_quantile_range=False,
                    require_sort=True) -> KnnResult:
    """The k nearest rows of `y` to each row of `x` under `wasserstein_cdist` with the same options: exactly
    `torch.sort(wasserstein_cdist(x, y, x_pos, y_pos, ...), dim=-1, stable=True)` cut to its first k columns -- values
    bit for bit, ascending, NaN after every number, the lower index first on equal values -- without forming the
    (P, R) matrix.  Without `dont_normalize` and `limit_quantile_range`, pairs whose lower bound exceeds the k-th value
    found so far are not walked; the result does not depend on which were.  1 <= k <= min(R, 128).  No gradient: pass
    rows that do not require one (or run under `torch.no_grad()`), and re-evaluate the selected pairs with
    `wasserstein_cdist` or `losses.sot_frames` where gradients are wanted."""
    _no_gradient(x, y, "wasserstein_knn")
    u, v, pu, pv, flags, batched = _prologue(x, y, x_pos, y_pos, p, square_dist, dont_normalize, limit_quantile_range,
                                             require_sort)
    if isinstance(k, bool) or int(k) != k:
        raise ValueError(f"sot_b200: k must be an integer, got {k!r}")
    k, R = int(k), v.shape[1]
    if k < 1 or k > R:
        raise ValueError(f"sot_b200: k = {k} must be at least 1 and at most the {R} rows of `y`")
    if k > _capi.KNN_MAX_K:
        raise ValueError(f"sot_b200: k = {k} is above the cap of {_capi.KNN_MAX_K} neighbours")
    if u.shape[0] * u.shape[1] == 0:
        values = torch.empty(u.shape[0], u.shape[1], k, dtype=torch.float32, device=u.device)
        indices = torch.empty(u.shape[0], u.shape[1], k, dtype=torch.int64, device=u.device)
    else:
        values, indices, _ = _capi.pairwise_knn(u, v, pu, pv, float(p), flags, k)
    return KnnResult(values, indices) if batched else KnnResult(values[0], indices[0])


class RadiusResult(NamedTuple):
    values: torch.Tensor   # float32 (E,)
    indices: torch.Tensor  # int64 (E, 2): (row of x, row of y), or (E, 3): (batch entry, row of x, row of y)


_FIRST_CAPACITY = 1 << 20  # pairs the first call has room for, at least (16 per row of x beyond 65 536 rows)


def wasserstein_radius(x, y, r, x_pos, y_pos, p=1, square_dist=False, dont_normalize=False,
                       limit_quantile_range=False, require_sort=True) -> RadiusResult:
    """Every pair within distance `r` under `wasserstein_cdist` with the same options and shapes: with
    `D = wasserstein_cdist(x, y, x_pos, y_pos, ...)` and `mask = D <= torch.tensor(r, dtype=torch.float32)`, `indices`
    is `mask.nonzero()` ((E, 2), or (E, 3) for batched rows) and `values` is `D[mask]`, bit for bit, without forming
    D.  A NaN distance is never within the radius.  Without `dont_normalize` and `limit_quantile_range`, pairs whose
    lower bound exceeds r are not walked; the result does not depend on which were.

    The call reads the number of pairs back to the host once (the result's size depends on it) and runs the search
    again, with room for exactly that many, when the first guess of min(B P R, max(2^20, 16 B P)) pairs was too
    small; to capture a CUDA graph, call `sot_pairwise_radius_device` with a fixed capacity.  No gradient, as for
    `wasserstein_knn`: re-evaluate the selected pairs with `wasserstein_cdist` or `losses.sot_frames` to train
    through them."""
    _no_gradient(x, y, "wasserstein_radius")
    if isinstance(r, bool) or not isinstance(r, numbers.Real) or r != r:
        raise ValueError(f"sot_b200: the radius must be a real number and not NaN, got {r!r}")
    u, v, pu, pv, flags, batched = _prologue(x, y, x_pos, y_pos, p, square_dist, dont_normalize, limit_quantile_range,
                                             require_sort)
    B, P, R = u.shape[0], u.shape[1], v.shape[1]
    pairs = B * P * R
    if pairs == 0:
        rows = cols = torch.empty(0, dtype=torch.int64, device=u.device)
        values = torch.empty(0, dtype=torch.float32, device=u.device)
    else:
        capacity = min(pairs, max(_FIRST_CAPACITY, 16 * B * P))
        rows, cols, values, count, _ = _capi.pairwise_radius(u, v, pu, pv, float(p), flags, float(r), capacity)
        E = int(count.item())
        if E > capacity:
            rows, cols, values, count, _ = _capi.pairwise_radius(u, v, pu, pv, float(p), flags, float(r), E)
        rows, cols, values = rows[:E], cols[:E], values[:E]
    parts = (rows // max(P, 1), rows % max(P, 1), cols) if batched else (rows, cols)
    return RadiusResult(values, torch.stack(parts, 1))
