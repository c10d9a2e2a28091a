"""Torch oracle of the W2 barycenter of spectra (`sot_b200.barycenter`) -- TEST INFRASTRUCTURE ONLY.

A restatement, op for op, of the semantics the kernels implement, built on the SOT oracle's building blocks
(`spectra_to_weights`, `lower_bound_lookup`) and `torch.sort(stable=True)`.  Runs in float32 or float64, on any
device; its gradient with respect to `x` is autograd's.  The product never imports it.

Per barycenter, rows x_1 .. x_K of n bins on one ascending grid `pos`, weights lambda:
  1. w_j = x_j^2 (square) or x_j;  c_j = cumsum(safe_divide(w_j, sum w_j))
  2. qs = stable sort of cat(c_1, ..., c_K) (row first, then bin, on equal values), K * n levels
  3. z_k = sum_j lambda_j pos[clamp(searchsorted_left(c_j, qs_k), 0, n - 1)]  (one z per tie group)
  4. delta_k = qs_k - qs_{k-1}, qs_{-1} = 0
  5. delta_k deposited at z_k onto `out_pos` by linear split: b the largest index with out_pos[b] <= z_k, bin b gets
     delta_k (out_pos[b+1] - z_k) / (out_pos[b+1] - out_pos[b]) and bin b+1 the rest; z below the grid goes to bin 0,
     z at or above its last point to bin M - 1.
"""
from __future__ import annotations

import torch

from oracle.sot_oracle import lower_bound_lookup, spectra_to_weights


def barycenter(x, weights, pos, out_pos=None, square=False):
    """x (N, K, n), weights (K,) or (N, K), pos (n,), out_pos (M,) -> (N, M) in x's dtype."""
    N, K, n = x.shape
    dt = x.dtype
    pos = pos.to(dt)
    out_pos = pos if out_pos is None else out_pos.to(dt)
    lam = weights.to(dt).expand(N, K)
    flat = x.reshape(N * K, n)
    w, _ = spectra_to_weights(flat, flat, square, False)
    c = torch.cumsum(w, 1).reshape(N, K, n)
    qs = torch.sort(c.reshape(N, K * n), dim=1, stable=True)[0]
    levels = qs.detach()
    z = torch.zeros_like(levels)
    grid = pos.expand(N, n)
    for j in range(K):
        zj, _ = lower_bound_lookup(levels, c[:, j].detach(), grid)
        z = z + lam[:, j:j + 1] * zj
    delta = qs - torch.nn.functional.pad(qs, (1, 0))[:, :-1]
    M = out_pos.shape[0]
    if M == 1:
        return delta.sum(1, keepdim=True)
    b = (torch.searchsorted(out_pos, z, right=True) - 1).clamp(0, M - 2)
    lo, hi = out_pos[b], out_pos[b + 1]
    f = (hi - z) / (hi - lo)
    f = torch.where(z < out_pos[0], torch.ones_like(f), torch.where(z >= out_pos[-1], torch.zeros_like(f), f))
    out = torch.zeros(N, M, dtype=dt, device=x.device)
    return out.scatter_add(1, b, delta * f).scatter_add(1, b + 1, delta * (1 - f))


def interpolate(x, y, t, pos, out_pos=None, square=False):
    """x, y (N, n), t (N,) -> (N, M): the barycenter of [x, y] with weights (1 - t, t)."""
    t = torch.as_tensor(t, dtype=x.dtype, device=x.device).expand(x.shape[0])
    return barycenter(torch.stack((x, y), 1), torch.stack((1 - t, t), 1), pos, out_pos, square)
