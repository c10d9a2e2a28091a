"""Torch oracle of the grouped barycenter (`sot_b200.barycenter.wasserstein_barycenter_groups`) -- TEST INFRASTRUCTURE
ONLY: a loop over the groups calling the dense oracle, `oracle.barycenter_oracle.barycenter`.  The product never
imports it."""
import torch

from oracle.barycenter_oracle import barycenter


def barycenter_groups(x, labels, n_groups, pos, weights=None, out_pos=None, square=False):
    """x (R, n), labels (R,) in [0, n_groups) -> (n_groups, M): row g is `barycenter` of the rows labelled g in
    increasing row order, with their `weights` (R,) or, None, torch.full((K_g,), 1.0 / K_g); NaN for a group with no
    rows."""
    M = (pos if out_pos is None else out_pos).shape[0]
    rows = []
    for g in range(n_groups):
        idx = (labels == g).nonzero()[:, 0]
        K = idx.shape[0]
        if K == 0:
            rows.append(torch.full((M,), float("nan"), dtype=x.dtype, device=x.device))
            continue
        w = torch.full((K,), 1.0 / K, device=x.device) if weights is None else weights[idx]
        rows.append(barycenter(x[idx][None], w, pos, out_pos, square)[0])
    return torch.stack(rows) if rows else x.new_zeros(0, M)
