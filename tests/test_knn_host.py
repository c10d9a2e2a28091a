"""Exact k-NN of spectra without a GPU: the host layer of `sot_b200.pairwise.wasserstein_knn` with a recording
stand-in for `_capi.pairwise_knn`, the refusals (all before any launch), the ABI's argument checks, and an fp64 model
of the quantile lower bound the kernels prune with, checked against the float64 oracle."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import sot_oracle as O
from tests import fake_kernels


def _oracle_dist(u, v, pu, pv, p, flags):
    out = []
    for b in range(u.shape[0]):
        P, R = u.shape[1], v.shape[1]
        U = u[b][:, None].expand(P, R, u.shape[2]).reshape(-1, u.shape[2])
        V = v[b][None].expand(P, R, v.shape[2]).reshape(-1, v.shape[2])
        out.append(fake_kernels._rows(U, V, pu, pv, p, flags).reshape(P, R))
    return torch.stack(out)


@pytest.fixture
def rec(monkeypatch):
    from sot_b200 import _capi, losses
    calls = []

    def pairwise_knn(u, v, pu, pv, p, flags, k, want_walked=False):
        calls.append(dict(u=u, v=v, pu=pu, pv=pv, p=p, flags=flags, k=k))
        vals, idx = torch.sort(_oracle_dist(u, v, pu, pv, p, flags).float(), dim=-1, stable=True)
        return vals[..., :k], idx[..., :k], None

    monkeypatch.setattr(_capi, "pairwise_knn", pairwise_knn)
    fake_kernels.allow_cpu_rows(monkeypatch, losses)
    return calls


def _data(P=3, R=6, n=9, m=7, B=None, seed=0):
    gen = torch.Generator().manual_seed(seed)
    lead_x, lead_y = ((B,) if B else ()) + (P,), ((B,) if B else ()) + (R,)
    x = torch.rand(lead_x + (n,), generator=gen, dtype=torch.float64) + 0.05
    y = torch.rand(lead_y + (m,), generator=gen, dtype=torch.float64) + 0.05
    return x, y, torch.linspace(0, 1, n), torch.linspace(0, 1, m) ** 2


def test_shapes_dtypes_flags_and_batching(rec):
    from sot_b200 import pairwise
    x, y, px, py = _data()
    r = pairwise.wasserstein_knn(x, y, 4, px, py, p=2, square_dist=True, dont_normalize=True,
                                 limit_quantile_range=True)
    assert r.values.shape == (3, 4) and r.indices.shape == (3, 4)
    assert r.values.dtype == torch.float32 and r.indices.dtype == torch.int64
    assert isinstance(r, pairwise.KnnResult) and r[0] is r.values
    c = rec[-1]
    assert c["u"].shape == (1, 3, 9) and c["v"].shape == (1, 6, 7) and c["u"].dtype == torch.float32
    assert c["flags"] == 1 | 2 | 4 and c["p"] == 2.0 and c["k"] == 4
    xb, yb, _, _ = _data(B=2)
    rb = pairwise.wasserstein_knn(xb, yb, 2, px, py)
    assert rb.values.shape == (2, 3, 2) and rec[-1]["u"].shape == (2, 3, 9) and rec[-1]["flags"] == 0
    for dt in (torch.float16, torch.bfloat16):
        pairwise.wasserstein_knn(x.to(dt), y.to(dt), 1, px, py)
        assert rec[-1]["u"].dtype == torch.float32
    z = torch.polar(x.float(), torch.rand(x.shape, dtype=torch.float32))  # complex rows: |z| first
    pairwise.wasserstein_knn(z, y, 1, px, py)
    assert torch.allclose(rec[-1]["u"][0], z.abs())
    with pytest.raises(ValueError):
        pairwise.wasserstein_knn(xb, y, 1, px, py)  # (B, P, n) against (R, m)


def test_the_result_is_the_sorted_cdist_and_unsorted_grids_are_sorted_first(rec):
    from sot_b200 import pairwise
    x, y, px, py = _data(P=4, R=8)
    perm_x, perm_y = torch.randperm(9, generator=torch.Generator().manual_seed(1)), torch.tensor([3, 0, 6, 1, 5, 2, 4])
    r = pairwise.wasserstein_knn(x[:, perm_x], y[:, perm_y], 5, px[perm_x], py[perm_y], p=2)
    c = rec[-1]
    assert torch.equal(c["pu"], px) and torch.equal(c["pv"], py)
    assert torch.equal(c["u"][0], x.float()) and torch.equal(c["v"][0], y.float())
    D = _oracle_dist(x.float()[None], y.float()[None], px, py, 2.0, 0)[0].float()  # what wasserstein_cdist gives
    want_v, want_i = torch.sort(D, dim=-1, stable=True)
    assert torch.equal(r.values, want_v[:, :5]) and torch.equal(r.indices, want_i[:, :5])


def test_refusals_happen_before_any_launch(rec):
    from sot_b200 import _capi, pairwise
    x, y, px, py = _data()
    before = _capi.launch_count()
    with pytest.raises(NotImplementedError, match="1-D grid"):
        pairwise.wasserstein_knn(x, y, 1, px.expand(3, 9), py)
    with pytest.raises(NotImplementedError, match="gradient"):
        pairwise.wasserstein_knn(x, y, 1, px, py.clone().requires_grad_(True))
    with pytest.raises(ValueError, match="8448"):
        pairwise.wasserstein_knn(torch.rand(2, 8449), y, 1, torch.linspace(0, 1, 8449), py)
    with pytest.raises(AssertionError, match="p>=1"):
        pairwise.wasserstein_knn(x, y, 1, px, py, p=0.5)
    for k in (0, -1, 7):  # R = 6
        with pytest.raises(ValueError, match="at least 1"):
            pairwise.wasserstein_knn(x, y, k, px, py)
    with pytest.raises(ValueError, match="integer"):
        pairwise.wasserstein_knn(x, y, 1.5, px, py)
    big = torch.rand(200, 7, dtype=torch.float64)
    with pytest.raises(ValueError, match="cap of 128"):
        pairwise.wasserstein_knn(x, big, 129, px, py)
    for t in ("x", "y"):
        xs, ys = x.clone().requires_grad_(t == "x"), y.clone().requires_grad_(t == "y")
        with pytest.raises(NotImplementedError, match="detach it, or re-evaluate the selected pairs"):
            pairwise.wasserstein_knn(xs, ys, 1, px, py)
    assert rec == [] and _capi.launch_count() == before
    with torch.no_grad():  # no gradient is dropped here: grad mode is off
        pairwise.wasserstein_knn(x.clone().requires_grad_(True), y, 1, px, py)
    assert len(rec) == 1
    pairwise.wasserstein_knn(x, big, 128, px, py)  # the cap itself is accepted
    assert rec[-1]["k"] == 128


def test_empty_inputs_launch_nothing(rec):
    from sot_b200 import pairwise
    x, y, px, py = _data()
    r = pairwise.wasserstein_knn(x[:0], y, 2, px, py)
    assert r.values.shape == (0, 2) and r.indices.shape == (0, 2) and r.indices.dtype == torch.int64
    xb, yb, _, _ = _data(B=2)
    assert pairwise.wasserstein_knn(xb[:0], yb[:0], 2, px, py).values.shape == (0, 3, 2)
    assert rec == []


def test_abi_validation_before_any_launch():
    from sot_b200 import _capi
    lib = _capi.load()
    before = _capi.launch_count()
    fake = ctypes.c_void_p(16)

    def prob(B=1, P=2, R=300, n=9, m=9, flags=0, p=2.0):
        return _capi.SotPairwiseProblem(B, P, R, n, m, 16, 16, 16, 16, p, flags)

    def knn(pr, k=3, values=fake, indices=fake):
        return lib.sot_pairwise_knn_device(ctypes.byref(pr) if pr is not None else None, k, values, indices, None,
                                           None)

    assert knn(None) == -1
    assert knn(prob(), k=0) == -1 and knn(prob(), k=-5) == -1
    assert knn(prob(), k=129) == -1 and b"128" in lib.sot_last_error()
    assert knn(prob(R=5), k=6) == -1
    assert knn(prob(flags=64)) == -1
    assert knn(prob(flags=_capi.SOT_RAW_WEIGHTS)) == -1 and knn(prob(flags=_capi.SOT_COMPLEX_INPUT)) == -1
    assert knn(prob(p=0.5)) == -3
    assert knn(prob(n=8449)) == -2
    assert knn(prob(), values=None) == -1 and knn(prob(), indices=None) == -1
    assert lib.sot_pairwise_knn_device(ctypes.byref(_capi.SotPairwiseProblem(1, 2, 300, 9, 9, None, 16, 16, 16, 2.0,
                                                                              0)), 3, fake, fake, None, None) == -1
    assert knn(prob(B=1 << 20, P=1 << 12)) == -2  # more than 2^31 - 1 rows
    for empty in (prob(B=0), prob(P=0)):
        assert knn(empty, values=None, indices=None) == 0
    assert _capi.launch_count() == before


# ---- fp64 model of the bound: interval means of the step quantile function ------------------------------------------
L, T0 = 32, 1.0 - 2.0 ** -20


def _means(c, pos):
    """The kernel's arithmetic: mean of Q(t) = pos[min(lb(t), n - 1)] over [l h, (l + 1) h], h = t0 / L."""
    h = T0 / L
    out = np.zeros(L)
    lo_c = np.concatenate([[0.0], c[:-1]])
    for l in range(L):
        a, b = l * h, (l + 1) * h
        seg = np.clip(np.minimum(c, b) - np.maximum(lo_c, a), 0.0, None)
        out[l] = np.dot(pos, seg) / h
    return out


def _lower_bound(eu, ev, p):
    """LB = h L^(1 - e) S^e with S = sum d (e = p) for p < 2, sum d^2 (e = p / 2) for p >= 2."""
    d, h = np.abs(eu - ev), T0 / L
    e = p / 2 if p >= 2 else p
    s = np.sum(d * d) if p >= 2 else np.sum(d)
    return h * L ** (1 - e) * s ** e


def _cdf(w):
    return np.cumsum(w / w.sum())


@pytest.mark.parametrize("p", [1, 1.5, 2, 3])
def test_the_bound_never_exceeds_the_oracle_distance(p):
    rng = np.random.default_rng(7)
    n, m = 37, 90
    pu, pv = np.sort(rng.random(n)), np.sort(rng.random(m)) ** 2  # different grids per side
    cases = []
    for _ in range(40):
        cases.append((rng.random(n) ** 4, rng.random(m) ** 4, pu, pv))
    x = np.zeros(n)
    x[[3, 4, 20]] = [1.0, 1.0, 2.0]  # heavy ties: few non-zero bins
    y = np.zeros(m)
    y[[10, 11, 60]] = [2.0, 2.0, 4.0]
    cases.append((x, y, pu, pv))
    cases.append((x, np.interp(np.arange(m), np.linspace(0, m - 1, n), x) + 1e-12, pu, pv))
    a = rng.random(n)
    cases.append((a, a * (1 + 1e-9) + 1e-12, pu, pu))  # a near-zero distance
    for wx, wy, gx, gy in cases:
        lb = _lower_bound(_means(_cdf(wx), gx), _means(_cdf(wy), gy), p)
        d = O.sot_per_frame(torch.tensor(wx)[None], torch.tensor(wy)[None], torch.tensor(gx), torch.tensor(gy),
                            p=p, stable=True).item()
        assert lb <= d * (1 + 1e-12) + 1e-15, (lb, d)
    # equal interval means: the same row on the same grid gives a zero bound (and is never skipped)
    w = rng.random(n)
    assert _lower_bound(_means(_cdf(w), pu), _means(_cdf(w), pu), p) == 0.0


def test_the_bound_is_tight_for_step_distributions():
    # two Diracs: Q is constant, so every interval mean is the position and LB is h L |x - y|^p of the full integral
    n = 16
    pos = np.linspace(0, 1, n)
    for p in (1, 2):
        x, y = np.zeros(n), np.zeros(n)
        x[2], y[9] = 1.0, 1.0
        lb = _lower_bound(_means(_cdf(x), pos), _means(_cdf(y), pos), p)
        d = O.sot_per_frame(torch.tensor(x)[None], torch.tensor(y)[None], torch.tensor(pos), torch.tensor(pos), p=p,
                            stable=True).item()
        assert lb <= d and lb >= d * T0 * (1 - 1e-12)
