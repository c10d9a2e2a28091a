"""Wasserstein barycenters and displacement interpolation of spectra in the SOT geometry (W2, 1-D).

`wasserstein_barycenter(x, weights, pos)` is the mean of a set of spectra in the geometry of the loss: the spectrum
whose quantile function is the weighted mean of the inputs' quantile functions.  Two harmonic spectra whose f0 differs
average to one peak at the averaged frequency, not to the two peaks of the Euclidean mean -- the centroid step of
k-means over spectra (whose assignment step is `pairwise.wasserstein_cdist`), templates and class prototypes.
`wasserstein_interpolate(x, y, t, pos)` is the point at t on the W2 geodesic from x to y: peaks move instead of
cross-fading (morphing, OT-mixup).  Both are differentiable with respect to the spectra.

Each input row is normalised by its own mass, so every output row is a distribution: mass per output grid point,
summing to 1.  Multiply by sum_j weights_j * M_j (M_j the input masses, of |x|^2 with `square_dist`) to get the
loudness back.  CUDA only, like the rest of the package: there is no CPU or eager fallback.
"""
from __future__ import annotations

import torch

from . import _capi, losses

__all__ = ["wasserstein_barycenter", "wasserstein_interpolate"]


class _Barycenter(torch.autograd.Function):
    """x (N, K, n) -> (N, M).  Nothing but the inputs is kept between the passes: the backward rebuilds the merged
    CDFs and walks them again with the upstream values."""

    @staticmethod
    def forward(ctx, x, weights, pos, out_pos, flags):
        ctx.flags = flags
        ctx.save_for_backward(x, weights, pos, out_pos)
        return _capi.barycenter(x, weights, pos, out_pos, flags)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad):
        x, weights, pos, out_pos = ctx.saved_tensors
        return _capi.barycenter_backward(x, weights, pos, out_pos, ctx.flags, grad.contiguous().float()), \
            None, None, None, None


def _no_grad_for(t, name):
    if isinstance(t, torch.Tensor) and t.requires_grad and torch.is_grad_enabled():
        raise NotImplementedError(f"sot_b200: `{name}` requires a gradient: barycenters are differentiable with "
                                  "respect to the spectra only (detach it)")


def wasserstein_barycenter(x, weights, pos, out_pos=None, square_dist=False, require_sort=True) -> torch.Tensor:
    """W2 barycenter of K spectra: `x` (K, n) -> (M,), or (N, K, n) -> (N, M) float32, one barycenter per leading
    index.  `weights` (K,) shared or (N, K) per barycenter: non-negative and summing to 1 (used as given; a negative
    weight gives a NaN row).  `pos` (n,) is the support of the input rows (unsorted grids are sorted once with the
    columns permuted when `require_sort`); `out_pos` (M,), ascending, is the grid the result is deposited on (default:
    `pos`), by linear split between the two grid points around each atom.  `square_dist`: the rows' weights are
    magnitude^2.  float16 / bfloat16 / float64 rows are converted to float32 and complex rows reduced to |z|.  A
    non-finite row makes its barycenter (and its gradient rows) NaN."""
    for t, name in ((weights, "weights"), (pos, "pos"), (out_pos, "out_pos")):
        _no_grad_for(t, name)
    if x.ndim not in (2, 3):
        raise ValueError(f"sot_b200: `x` must be (K, n) or (N, K, n), got {tuple(x.shape)}")
    single = x.ndim == 2
    x = losses._magnitude(x[None] if single else x)
    N, K, n = x.shape
    rows = losses._rows(x.reshape(N * K, n), "x")
    if pos.ndim != 1:
        raise NotImplementedError(f"sot_b200: `pos` has shape {tuple(pos.shape)}: barycenters take one 1-D grid "
                                  "(per-row supports are not supported)")
    p = losses._support(pos, rows, "pos")
    if require_sort:
        p, rows = losses._order(p, rows, pos)
    if out_pos is None:
        op = p
    else:
        if out_pos.ndim != 1 or out_pos.shape[0] < 1:
            raise ValueError(f"sot_b200: `out_pos` must be a non-empty 1-D grid, got {tuple(out_pos.shape)}")
        op = losses._support(out_pos, out_pos[None], "out_pos")
        if not losses._is_ascending(op, out_pos):
            raise ValueError("sot_b200: `out_pos` must be ascending")
    w = torch.as_tensor(weights).detach().to(device=rows.device, dtype=torch.float32).contiguous()
    out = _Barycenter.apply(rows.reshape(N, K, n), w, p, op, losses._flags(square_dist, False, False))
    return out[0] if single else out


def wasserstein_interpolate(x, y, t, pos, out_pos=None, square_dist=False, require_sort=True) -> torch.Tensor:
    """Displacement interpolation: the point at `t` on the W2 geodesic from `x` to `y`, i.e. the barycenter of [x, y]
    with weights (1 - t, t).  `x`, `y` (n,) or (N, n); `t` a float or a tensor that broadcasts against the leading
    shape (a morph of T steps between one pair: `t` of shape (T,) gives (T, M)).  Other arguments as in
    `wasserstein_barycenter`."""
    x, y = losses._magnitude(x), losses._magnitude(y)
    t = torch.as_tensor(t, dtype=torch.float32, device=x.device)
    lead = torch.broadcast_shapes(x.shape[:-1], y.shape[:-1], t.shape)
    n = x.shape[-1]
    pair = torch.stack((x.expand(lead + (n,)), y.expand(lead + (n,))), -2).reshape(-1, 2, n)
    t = t.expand(lead).reshape(-1)
    out = wasserstein_barycenter(pair, torch.stack((1 - t, t), -1), pos, out_pos, square_dist, require_sort)
    return out.reshape(lead + out.shape[-1:])
