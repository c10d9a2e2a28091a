"""Exact radius search over spectra without a GPU: the host layer of `sot_b200.pairwise.wasserstein_radius` with a
recording stand-in for `_capi.pairwise_radius` (shapes, conversions, the second call when the first capacity is too
small), the refusals (all before any launch), and the ABI's argument checks through the real library."""
import ctypes
import math

import pytest
import torch

from tests import fake_kernels


def _oracle_dist(u, v, pu, pv, p, flags):
    out = []
    for b in range(u.shape[0]):
        P, R = u.shape[1], v.shape[1]
        U = u[b][:, None].expand(P, R, u.shape[2]).reshape(-1, u.shape[2])
        V = v[b][None].expand(P, R, v.shape[2]).reshape(-1, v.shape[2])
        out.append(fake_kernels._rows(U, V, pu, pv, p, flags).reshape(P, R))
    return torch.stack(out).float()


@pytest.fixture
def rec(monkeypatch):
    from sot_b200 import _capi, losses
    calls = []

    def pairwise_radius(u, v, pu, pv, p, flags, radius, capacity, want_walked=False):
        calls.append(dict(u=u, v=v, pu=pu, pv=pv, p=p, flags=flags, radius=radius, capacity=capacity))
        D = _oracle_dist(u, v, pu, pv, p, flags)
        D = D.reshape(-1, D.shape[-1])
        mask = D <= torch.tensor(radius, dtype=torch.float32)
        hits = mask.nonzero()
        E = hits.shape[0]
        rows = torch.full((capacity,), -7, dtype=torch.int64)  # (unspecified past the count, or all of it when short)
        cols = torch.full((capacity,), -7, dtype=torch.int64)
        values = torch.full((capacity,), float("nan"))
        if E <= capacity:
            rows[:E], cols[:E], values[:E] = hits[:, 0], hits[:, 1], D[mask]
        return rows, cols, values, torch.tensor([E]), None

    monkeypatch.setattr(_capi, "pairwise_radius", pairwise_radius)
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
    r = pairwise.wasserstein_radius(x, y, 0.05, px, py, p=2, square_dist=True, dont_normalize=True,
                                    limit_quantile_range=True)
    assert isinstance(r, pairwise.RadiusResult) and r[0] is r.values
    assert r.values.dtype == torch.float32 and r.indices.dtype == torch.int64
    assert r.values.ndim == 1 and r.indices.shape == (r.values.shape[0], 2)
    c = rec[-1]
    assert c["u"].shape == (1, 3, 9) and c["v"].shape == (1, 6, 7) and c["u"].dtype == torch.float32
    assert c["flags"] == 1 | 2 | 4 and c["p"] == 2.0 and c["radius"] == 0.05
    assert c["capacity"] == 18  # min(B P R, max(2^20, 16 B P))
    xb, yb, _, _ = _data(B=2)
    rb = pairwise.wasserstein_radius(xb, yb, math.inf, px, py)
    assert rb.indices.shape == (2 * 3 * 6, 3) and rec[-1]["u"].shape == (2, 3, 9) and rec[-1]["flags"] == 0
    assert torch.equal(rb.indices, torch.ones(2, 3, 6).nonzero())
    for dt in (torch.float16, torch.bfloat16, torch.float64):
        pairwise.wasserstein_radius(x.to(dt), y.to(dt), 1.0, px, py)
        assert rec[-1]["u"].dtype == torch.float32 and rec[-1]["v"].dtype == torch.float32
    z = torch.polar(x.float(), torch.rand(x.shape, dtype=torch.float32))  # complex rows: |z| first
    pairwise.wasserstein_radius(z, y, 1.0, px, py)
    assert torch.allclose(rec[-1]["u"][0], z.abs())
    with pytest.raises(ValueError):
        pairwise.wasserstein_radius(xb, y, 1.0, px, py)  # (B, P, n) against (R, m)


@pytest.mark.parametrize("batched", [False, True])
def test_the_result_is_the_masked_cdist_and_unsorted_grids_are_sorted_first(rec, batched):
    from sot_b200 import pairwise
    x, y, px, py = _data(P=4, R=8, B=2 if batched else None)
    perm_x, perm_y = torch.randperm(9, generator=torch.Generator().manual_seed(1)), torch.tensor([3, 0, 6, 1, 5, 2, 4])
    D = _oracle_dist(x.float().reshape(-1, 4, 9), y.float().reshape(-1, 8, 7), px, py, 2.0, 1)
    D = D if batched else D[0]  # what wasserstein_cdist gives
    r = float(D.flatten().median())
    got = pairwise.wasserstein_radius(x[..., perm_x], y[..., perm_y], r, px[perm_x], py[perm_y], p=2,
                                      square_dist=True)
    c = rec[-1]
    assert torch.equal(c["pu"], px) and torch.equal(c["pv"], py)
    mask = D <= torch.tensor(r, dtype=torch.float32)
    assert 0 < mask.sum() < mask.numel()
    assert torch.equal(got.indices, mask.nonzero()) and torch.equal(got.values, D[mask])


def test_a_second_call_when_the_first_capacity_is_too_small(rec, monkeypatch):
    from sot_b200 import pairwise
    monkeypatch.setattr(pairwise, "_FIRST_CAPACITY", 4)
    x, y, px, py = _data(P=5, R=40)
    D = _oracle_dist(x.float()[None], y.float()[None], px, py, 1.0, 0)[0]
    # 16 P = 80 places first; a radius with more hits than that takes a second call with room for exactly all
    r = float(D.flatten().sort().values[150])
    got = pairwise.wasserstein_radius(x, y, r, px, py)
    mask = D <= r
    assert [c["capacity"] for c in rec] == [80, int(mask.sum())]
    assert torch.equal(got.indices, mask.nonzero()) and torch.equal(got.values, D[mask])
    rec.clear()
    r = float(D.flatten().sort().values[30])  # fits: one call
    got = pairwise.wasserstein_radius(x, y, r, px, py)
    assert [c["capacity"] for c in rec] == [80] and torch.equal(got.indices, (D <= r).nonzero())
    rec.clear()
    got = pairwise.wasserstein_radius(x, y, -1.0, px, py)  # nothing within: one call, empty result
    assert len(rec) == 1 and got.indices.shape == (0, 2) and got.values.shape == (0,)


def test_refusals_happen_before_any_launch(rec):
    from sot_b200 import _capi, pairwise
    x, y, px, py = _data()
    before = _capi.launch_count()
    for r in (float("nan"), torch.tensor(float("nan")).item(), 1 + 2j, "1", None, True, torch.tensor(1.0)):
        with pytest.raises(ValueError, match="radius"):
            pairwise.wasserstein_radius(x, y, r, px, py)
    with pytest.raises(NotImplementedError, match="1-D grid"):
        pairwise.wasserstein_radius(x, y, 1.0, px.expand(3, 9), py)
    with pytest.raises(NotImplementedError, match="gradient"):
        pairwise.wasserstein_radius(x, y, 1.0, px, py.clone().requires_grad_(True))
    with pytest.raises(ValueError, match="8448"):
        pairwise.wasserstein_radius(torch.rand(2, 8449), y, 1.0, torch.linspace(0, 1, 8449), py)
    with pytest.raises(AssertionError, match="p>=1"):
        pairwise.wasserstein_radius(x, y, 1.0, px, py, p=0.5)
    for t in ("x", "y"):
        xs, ys = x.clone().requires_grad_(t == "x"), y.clone().requires_grad_(t == "y")
        with pytest.raises(NotImplementedError, match="wasserstein_radius has none .*re-evaluate the selected pairs "
                                                      "with wasserstein_cdist or losses.sot_frames"):
            pairwise.wasserstein_radius(xs, ys, 1.0, px, py)
    assert rec == [] and _capi.launch_count() == before
    with torch.no_grad():  # no gradient is dropped here: grad mode is off
        pairwise.wasserstein_radius(x.clone().requires_grad_(True), y, 1.0, px, py)
    assert len(rec) == 1
    for r in (3, -math.inf, math.inf, torch.tensor(0.5).item()):  # any real number that is not NaN
        pairwise.wasserstein_radius(x, y, r, px, py)
    assert len(rec) == 5


def test_empty_inputs_launch_nothing(rec):
    from sot_b200 import pairwise
    x, y, px, py = _data()
    for a, b in ((x[:0], y), (x, y[:0])):
        r = pairwise.wasserstein_radius(a, b, 1.0, px, py)
        assert r.values.shape == (0,) and r.indices.shape == (0, 2) and r.indices.dtype == torch.int64
    xb, yb, _, _ = _data(B=2)
    for a, b in ((xb[:0], yb[:0]), (xb[:, :0], yb), (xb, yb[:, :0])):
        r = pairwise.wasserstein_radius(a, b, 1.0, px, py)
        assert r.values.shape == (0,) and r.indices.shape == (0, 3)
    assert rec == []


def test_abi_validation_before_any_launch():
    from sot_b200 import _capi
    lib = _capi.load()
    before = _capi.launch_count()
    fake = ctypes.c_void_p(16)

    def prob(B=1, P=2, R=300, n=9, m=9, flags=0, p=2.0, u=16):
        return _capi.SotPairwiseProblem(B, P, R, n, m, u, 16, 16, 16, p, flags)

    def radius(pr, r=1.0, capacity=10, rows=fake, cols=fake, values=fake, count=fake):
        return lib.sot_pairwise_radius_device(ctypes.byref(pr) if pr is not None else None, r, capacity, rows, cols,
                                              values, count, None, None)

    assert radius(None) == -1
    assert radius(prob(), r=float("nan")) == -1 and b"NaN" in lib.sot_last_error()
    assert radius(prob(), capacity=-1) == -1 and b"capacity" in lib.sot_last_error()
    assert radius(prob(n=8449)) == -2 and radius(prob(m=8449)) == -2
    assert radius(prob(flags=64)) == -1
    assert radius(prob(flags=_capi.SOT_RAW_WEIGHTS)) == -1 and radius(prob(flags=_capi.SOT_COMPLEX_INPUT)) == -1
    assert radius(prob(p=0.5)) == -3
    assert radius(prob(u=None)) == -1
    assert radius(prob(), count=None) == -1
    for missing in (dict(rows=None), dict(cols=None), dict(values=None)):
        assert radius(prob(), **missing) == -1
    assert radius(prob(B=1 << 20, P=1 << 12)) == -2  # more than 2^31 - 1 rows
    assert radius(prob(B=0), count=None) == -1  # the count is written even for an empty problem
    # empty problems pass every check (and then only zero the count, which needs a device: see test_gpu_radius.py),
    # with NULL rows and positions
    for empty in (prob(B=0, u=None), prob(P=0, u=None), prob(R=0, u=None)):
        assert radius(empty, rows=None, cols=None, values=None) >= 0
    assert _capi.launch_count() == before
