"""Pairwise SOT distances without a GPU: the host layer of `sot_b200.pairwise` with recording stand-ins for the two
`_capi` wrappers, the refusals (all before any launch), the ABI's argument checks, and an fp64 model of the backward
decomposition the kernels use (dL/dCDF accumulated per row, chain rule once per row)."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import sot_oracle as O
from tests import fake_kernels


def _materialised(x, y):
    P, R = x.shape[0], y.shape[0]
    return (x[:, None].expand(P, R, x.shape[1]).reshape(-1, x.shape[1]),
            y[None].expand(P, R, y.shape[1]).reshape(-1, y.shape[1]))


def _oracle_dist(u, v, pu, pv, p, flags):
    """(B, P, n), (B, R, m) -> (B, P, R) with the oracle's arithmetic on the materialised pairs."""
    out = []
    for b in range(u.shape[0]):
        U, V = _materialised(u[b], v[b])
        out.append(fake_kernels._rows(U, V, pu, pv, p, flags).reshape(u.shape[1], v.shape[1]))
    return torch.stack(out)


@pytest.fixture
def rec(monkeypatch):
    from sot_b200 import _capi, losses
    calls = []

    def pairwise(u, v, pu, pv, p, flags):
        calls.append(dict(op="fwd", u=u, v=v, pu=pu, pv=pv, p=p, flags=flags))
        return _oracle_dist(u, v, pu, pv, p, flags).detach()

    def pairwise_backward(u, v, pu, pv, p, flags, upstream, want_gu=True, want_gv=True):
        calls.append(dict(op="bwd", want=(want_gu, want_gv)))
        with torch.enable_grad():
            ur, vr = u.detach().clone().requires_grad_(True), v.detach().clone().requires_grad_(True)
            gu, gv = torch.autograd.grad((_oracle_dist(ur, vr, pu, pv, p, flags) * upstream).sum(), (ur, vr))
        return (gu if want_gu else None), (gv if want_gv else None)

    monkeypatch.setattr(_capi, "pairwise", pairwise)
    monkeypatch.setattr(_capi, "pairwise_backward", pairwise_backward)
    fake_kernels.allow_cpu_rows(monkeypatch, losses)
    return calls


def _data(P=3, R=4, n=9, m=7, B=None, seed=0):
    gen = torch.Generator().manual_seed(seed)
    lead_x, lead_y = ((B,) if B else ()) + (P,), ((B,) if B else ()) + (R,)
    x = torch.rand(lead_x + (n,), generator=gen, dtype=torch.float64) + 0.05
    y = torch.rand(lead_y + (m,), generator=gen, dtype=torch.float64) + 0.05
    return x, y, torch.linspace(0, 1, n), torch.linspace(0, 1, m) ** 2


def test_shapes_dtypes_flags_and_batching(rec):
    from sot_b200 import pairwise
    x, y, px, py = _data()
    D = pairwise.wasserstein_cdist(x, y, px, py, p=2, square_dist=True, dont_normalize=True,
                                   limit_quantile_range=True)
    assert D.shape == (3, 4) and D.dtype == torch.float32
    c = rec[-1]
    assert c["u"].shape == (1, 3, 9) and c["v"].shape == (1, 4, 7)
    assert c["u"].dtype == torch.float32 and c["v"].dtype == torch.float32  # float64 converted like `_rows` does
    assert c["flags"] == 1 | 2 | 4 and c["p"] == 2.0
    xb, yb, _, _ = _data(B=2)
    assert pairwise.wasserstein_cdist(xb, yb, px, py).shape == (2, 3, 4)
    assert rec[-1]["u"].shape == (2, 3, 9) and rec[-1]["flags"] == 0
    for dt in (torch.float16, torch.bfloat16):
        pairwise.wasserstein_cdist(x.to(dt), y.to(dt), px, py)
        assert rec[-1]["u"].dtype == torch.float32
    z = torch.polar(x.float(), torch.rand(x.shape, dtype=torch.float32))  # complex rows: |z| first
    Dz = pairwise.wasserstein_cdist(z, y, px, py)
    assert torch.allclose(rec[-1]["u"][0], z.abs()) and Dz.shape == (3, 4)
    with pytest.raises(ValueError):
        pairwise.wasserstein_cdist(xb, y, px, py)  # (B, P, n) against (R, m)


def test_unsorted_grids_are_sorted_once_with_their_columns(rec):
    from sot_b200 import pairwise
    x, y, px, py = _data()
    perm_x, perm_y = torch.randperm(9, generator=torch.Generator().manual_seed(1)), torch.tensor([3, 0, 6, 1, 5, 2, 4])
    xs, ys = x[:, perm_x].clone().requires_grad_(True), y[:, perm_y].clone().requires_grad_(True)
    D = pairwise.wasserstein_cdist(xs, ys, px[perm_x], py[perm_y], p=2)
    c = rec[-1]
    assert torch.equal(c["pu"], px) and torch.equal(c["pv"], py)
    assert torch.equal(c["u"][0], x.float()) and torch.equal(c["v"][0], y.float())
    assert torch.allclose(D, pairwise.wasserstein_cdist(x, y, px, py, p=2))
    Gm = torch.rand(3, 4, generator=torch.Generator().manual_seed(2))
    (Gm * D).sum().backward()
    assert rec[-1] == dict(op="bwd", want=(True, True))
    # gradients follow the columns back through the sort: the oracle on the materialised, unsorted pairs
    X, Y = _materialised(xs.detach(), ys.detach())
    _, gx, gy = O.sot_loss_and_grads(X.float(), Y.float(), px[perm_x], py[perm_y], upstream=Gm.reshape(-1), p=2,
                                     stable=True)
    assert torch.allclose(xs.grad.float(), gx.reshape(3, 4, 9).sum(1), rtol=1e-5, atol=1e-6)
    assert torch.allclose(ys.grad.float(), gy.reshape(3, 4, 7).sum(0), rtol=1e-5, atol=1e-6)


def test_refusals_happen_before_any_launch(rec):
    from sot_b200 import _capi, pairwise
    x, y, px, py = _data()
    before = _capi.launch_count()
    with pytest.raises(NotImplementedError, match="1-D grid"):
        pairwise.wasserstein_cdist(x, y, px.expand(3, 9), py)
    with pytest.raises(NotImplementedError, match="gradient"):
        pairwise.wasserstein_cdist(x, y, px, py.clone().requires_grad_(True))
    with pytest.raises(ValueError, match="8448"):
        pairwise.wasserstein_cdist(torch.rand(2, 8449), y, torch.linspace(0, 1, 8449), py)
    with pytest.raises(AssertionError, match="p>=1"):
        pairwise.wasserstein_cdist(x, y, px, py, p=0.5)
    assert rec == [] and _capi.launch_count() == before


def test_abi_validation_before_any_launch():
    from sot_b200 import _capi
    lib = _capi.load()
    before = _capi.launch_count()
    fake = ctypes.c_void_p(16)

    def prob(B=1, P=2, R=3, n=9, m=9, flags=0, p=2.0):
        return _capi.SotPairwiseProblem(B, P, R, n, m, 16, 16, 16, 16, p, flags)

    def fwd(pr, dist=fake):
        return lib.sot_pairwise_device(ctypes.byref(pr), dist, None)

    assert fwd(prob(flags=_capi.SOT_RAW_WEIGHTS)) == -1
    assert fwd(prob(flags=_capi.SOT_COMPLEX_INPUT)) == -1
    assert b"SOT_SQUARE" in lib.sot_last_error()
    assert fwd(prob(flags=64)) == -1
    assert fwd(prob(n=8449)) == -2 and b"8448" in lib.sot_last_error()
    assert fwd(prob(m=8449)) == -2
    assert fwd(prob(p=0.5)) == -3
    assert fwd(prob(n=0)) == -1 and fwd(prob(P=-1)) == -1
    assert fwd(prob(B=1, P=1 << 20, R=1 << 12)) == -2  # more than 2^31 - 1 pairs
    assert fwd(prob(), dist=None) == -1
    for empty in (prob(B=0), prob(P=0), prob(R=0)):
        assert fwd(empty, dist=None) == 0
        assert lib.sot_pairwise_backward_device(ctypes.byref(empty), None, fake, fake, None) == 0
    assert lib.sot_pairwise_backward_device(ctypes.byref(prob()), None, fake, fake, None) == -1  # upstream NULL
    assert lib.sot_pairwise_backward_device(ctypes.byref(prob(p=0.9)), fake, fake, fake, None) == -3
    assert lib.sot_pairwise_backward_device(ctypes.byref(prob()), fake, None, None, None) == 0  # nothing wanted
    assert _capi.launch_count() == before


# ---- fp64 model of the backward decomposition -------------------------------------------------------------------
def _pair_cdf_grads(a, b, pu, pv, p, square, cut, limit):
    """One pair in fp64: CDFs as the pair kernel sees them, dL/dCDF of both rows, and the masses (clamped)."""
    eps = np.float64(np.float32(O.SAFE_EPS))
    wa, wb = (a * a, b * b) if square else (a, b)
    Ma, Mb = wa.sum(), wb.sum()
    Ma_c, Mb_c = max(Ma, eps) if Ma > eps else eps, max(Mb, eps) if Mb > eps else eps
    cu, cv = np.cumsum(wa / Ma_c), np.cumsum(wb / (Ma_c if cut else Mb_c))  # (the oracle's rounding: the mask is
    # discontinuous in the last ulp of the CDF)
    _, gcu, gcv, _, _ = O.closed_form_from_cdfs(cu, cv, pu, pv, p, limit)
    return cu, cv, gcu, gcv, Ma, Ma_c, Mb, Mb_c


@pytest.mark.parametrize("cut", [False, True])
@pytest.mark.parametrize("square", [False, True])
@pytest.mark.parametrize("p,limit", [(1, False), (2, True), (3, False)])
def test_backward_decomposition_matches_the_sum_over_pairs(cut, square, p, limit):
    rng = np.random.default_rng(3)
    P, R, n, m = 4, 5, 7, 6
    x, y = rng.random((P, n)) + 0.01, rng.random((R, m)) + 0.01
    x[1] *= 1e-9  # a target at the safe_divide floor: no mass term
    pu, pv = np.sort(rng.random(n)), np.sort(rng.random(m))
    Gm = rng.standard_normal((P, R))
    eps = np.float64(np.float32(O.SAFE_EPS))
    # reference: the sum over pairs of the oracle's per-pair gradients
    want_x, want_y = np.zeros_like(x), np.zeros_like(y)
    for i in range(P):
        for j in range(R):
            _, gx, gy = O.closed_form_backward(x[i:i + 1], y[j:j + 1], pu, pv, p, square, cut, limit)
            want_x[i] += Gm[i, j] * gx[0]
            want_y[j] += Gm[i, j] * gy[0]
    # the kernels' decomposition: accumulate dL/dCDF per row, then the chain rule once per row
    A_u, S_u = np.zeros((P, n)), np.zeros(P)
    A_v = np.zeros((R, m))
    cu_rows, Mx, My = {}, {}, {}
    for i in range(P):
        for j in range(R):
            cu, cv, gcu, gcv, Ma, Ma_c, Mb, Mb_c = _pair_cdf_grads(x[i], y[j], pu, pv, p, square, cut, limit)
            A_u[i] += Gm[i, j] * gcu
            if cut:
                S_u[i] += Gm[i, j] * np.dot(gcv, cv)
                A_v[j] += Gm[i, j] / Ma_c * gcv
            else:
                A_v[j] += Gm[i, j] * gcv
            cu_rows[i], Mx[i], My[j] = cu, (Ma, Ma_c), (Mb, Mb_c)
    got_x, got_y = np.zeros_like(x), np.zeros_like(y)
    for i in range(P):
        Ma, Ma_c = Mx[i]
        corr = (np.dot(A_u[i], cu_rows[i]) + (S_u[i] if cut else 0.0)) if Ma > eps else 0.0
        ga = (np.cumsum(A_u[i][::-1])[::-1] - corr) / Ma_c
        got_x[i] = 2 * x[i] * ga if square else ga
    for j in range(R):
        Mb, Mb_c = My[j]
        wb = y[j] ** 2 if square else y[j]
        suffix = np.cumsum(A_v[j][::-1])[::-1]
        if cut:
            gb = suffix
        else:
            corr = np.dot(A_v[j], np.cumsum(wb / Mb_c)) if Mb > eps else 0.0
            gb = (suffix - corr) / Mb_c
        got_y[j] = 2 * y[j] * gb if square else gb
    scale = max(np.abs(want_x).max(), np.abs(want_y).max())
    assert np.abs(got_x - want_x).max() <= 1e-12 * scale
    assert np.abs(got_y - want_y).max() <= 1e-12 * scale
