"""Pairwise SOT distances: the W_p^p matrix between two batches of spectra, the `torch.cdist` of the loss.

`wasserstein_cdist(x, y, x_pos, y_pos)` compares every row of `x` with every row of `y` (nearest-neighbour lookup over
a set of spectra, permutation-invariant losses over sets of sources, sweeps of one target against many candidates)
without materialising the P x R pairs: the kernels behind `sot_pairwise_device` build each row's CDF once and walk
only the merge of each pair.  Entry [b, i, j] is what `losses.sot_frames` gives for the single pair
(x[b, i], y[b, j]) with the same options; the result is differentiable with respect to x and y.

CUDA only, like the rest of the package: there is no CPU or eager fallback.
"""
from __future__ import annotations

import torch

from . import _capi, losses

__all__ = ["wasserstein_cdist"]


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


def wasserstein_cdist(x, y, x_pos, y_pos, p=1, square_dist=False, dont_normalize=False, limit_quantile_range=False,
                      require_sort=True) -> torch.Tensor:
    """W_p^p of every pair of rows: `x` (P, n) or (B, P, n) targets, `y` (R, m) or (B, R, m) predictions ->
    (P, R) or (B, P, R) float32, following `torch.cdist`'s batching.  `x_pos` (n,) and `y_pos` (m,) are one grid per
    side (n may differ from m); unsorted grids are sorted once with the columns permuted when `require_sort`.
    Options as in `losses.Wasserstein1D`: `square_dist` (weights = magnitude^2), `dont_normalize` (cut mode: y divided
    by x's mass), `limit_quantile_range` (strict `qs > 1` mask).  float16 / bfloat16 / float64 inputs are converted
    to float32 as `losses.sot_frames` converts them; complex rows are reduced to |z| first."""
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
    flags = losses._flags(square_dist, dont_normalize, False, limit_quantile_range)
    dist = _Cdist.apply(u, v, pu, pv, float(p), flags)
    return dist if batched else dist[0]
