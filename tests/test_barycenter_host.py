"""Wasserstein barycenters without a GPU: the host layer of `sot_b200.barycenter` with recording stand-ins for the two
`_capi` wrappers, the refusals (all before any launch), the ABI's argument checks, and an fp64 model of the backward
decomposition the kernels use (slot gradient -> dL/dCDF -> suffix sums and the normalisation's chain rule)."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import barycenter_oracle as BO
from oracle import sot_oracle as O
from tests import fake_kernels


@pytest.fixture
def rec(monkeypatch):
    from sot_b200 import _capi, losses
    calls = []

    def barycenter(x, w, pos, pos_out, flags):
        calls.append(dict(op="fwd", x=x, w=w, pos=pos, pos_out=pos_out, flags=flags))
        return BO.barycenter(x, w, pos, pos_out, bool(flags & _capi.SOT_SQUARE)).detach()

    def barycenter_backward(x, w, pos, pos_out, flags, upstream):
        calls.append(dict(op="bwd", upstream=upstream))
        with torch.enable_grad():
            xr = x.detach().clone().requires_grad_(True)
            out = BO.barycenter(xr, w, pos, pos_out, bool(flags & _capi.SOT_SQUARE))
            return torch.autograd.grad((out * upstream).sum(), xr)[0]

    monkeypatch.setattr(_capi, "barycenter", barycenter)
    monkeypatch.setattr(_capi, "barycenter_backward", barycenter_backward)
    fake_kernels.allow_cpu_rows(monkeypatch, losses)
    return calls


def _data(N=3, K=4, n=9, seed=0):
    gen = torch.Generator().manual_seed(seed)
    x = torch.rand(N, K, n, generator=gen, dtype=torch.float64) + 0.05
    w = torch.rand(K, generator=gen, dtype=torch.float64)
    return x, w / w.sum(), torch.linspace(0, 1, n)


def test_shapes_dtypes_flags_and_weights(rec):
    from sot_b200 import barycenter as BC
    x, w, pos = _data()
    out = BC.wasserstein_barycenter(x, w, pos, square_dist=True)
    assert out.shape == (3, 9) and out.dtype == torch.float32
    c = rec[-1]
    assert c["x"].shape == (3, 4, 9) and c["x"].dtype == torch.float32 and c["x"].is_contiguous()
    assert c["w"].shape == (4,) and c["w"].dtype == torch.float32 and c["flags"] == 1
    assert c["pos_out"] is c["pos"] or torch.equal(c["pos_out"], c["pos"])  # out_pos defaults to pos
    assert torch.allclose(out.sum(1), torch.ones(3))
    one = BC.wasserstein_barycenter(x[1], w, pos)  # (K, n) -> (M,)
    assert one.shape == (9,) and rec[-1]["x"].shape == (1, 4, 9) and rec[-1]["flags"] == 0
    per = torch.rand(3, 4, dtype=torch.float64)
    BC.wasserstein_barycenter(x, per, pos)
    assert rec[-1]["w"].shape == (3, 4) and torch.equal(rec[-1]["w"], per.float())
    coarse = torch.linspace(0, 1, 5)
    assert BC.wasserstein_barycenter(x, w, pos, out_pos=coarse).shape == (3, 5)
    assert torch.equal(rec[-1]["pos_out"], coarse)
    for dt in (torch.float16, torch.bfloat16):
        BC.wasserstein_barycenter(x.to(dt), w, pos)
        assert rec[-1]["x"].dtype == torch.float32
    z = torch.polar(x.float(), torch.rand(x.shape))
    BC.wasserstein_barycenter(z, w, pos)
    assert torch.allclose(rec[-1]["x"], z.abs())
    assert BC.wasserstein_barycenter(x[:0], w, pos).shape == (0, 9)


def test_unsorted_grid_is_sorted_once_with_its_columns(rec):
    from sot_b200 import barycenter as BC
    x, w, pos = _data()
    perm = torch.randperm(9, generator=torch.Generator().manual_seed(1))
    xs = x[..., perm].clone().requires_grad_(True)
    out = BC.wasserstein_barycenter(xs, w, pos[perm])
    assert torch.equal(rec[-1]["pos"], pos) and torch.equal(rec[-1]["x"], x.float())
    assert torch.equal(out, BC.wasserstein_barycenter(x, w, pos))
    G = torch.rand(3, 9, generator=torch.Generator().manual_seed(2))
    (G * out).sum().backward()
    assert rec[-1]["op"] == "bwd" and rec[-1]["upstream"].is_contiguous()
    xr = x.float().clone().requires_grad_(True)
    (G * BO.barycenter(xr, w.float(), pos)).sum().backward()
    assert torch.allclose(xs.grad[..., torch.argsort(perm)].float(), xr.grad, atol=1e-6)


def test_interpolate_broadcasts_t_and_stacks_the_pair(rec):
    from sot_b200 import barycenter as BC
    x, _, pos = _data()
    a, b = x[0, 0], x[0, 1]
    t = torch.tensor([0.0, 0.25, 1.0])
    out = BC.wasserstein_interpolate(a, b, t, pos)
    assert out.shape == (3, 9)
    c = rec[-1]
    assert c["x"].shape == (3, 2, 9) and torch.equal(c["x"][:, 0], a.float().expand(3, 9))
    assert torch.equal(c["w"], torch.stack((1 - t, t), 1))
    assert BC.wasserstein_interpolate(a, b, 0.5, pos).shape == (9,)
    assert BC.wasserstein_interpolate(x[:, 0], x[:, 1], 0.5, pos).shape == (3, 9)
    assert BC.wasserstein_interpolate(x[:, 0], b, torch.rand(3), pos, out_pos=torch.linspace(0, 1, 4)).shape == (3, 4)
    assert torch.allclose(out[0], BO.barycenter(a.float()[None, None], torch.ones(1), pos)[0])


def test_refusals_happen_before_any_launch(rec):
    from sot_b200 import _capi, barycenter as BC
    x, w, pos = _data()
    before = _capi.launch_count()
    with pytest.raises(NotImplementedError, match="weights"):
        BC.wasserstein_barycenter(x, w.clone().requires_grad_(True), pos)
    with pytest.raises(NotImplementedError, match="`pos`"):
        BC.wasserstein_barycenter(x, w, pos.clone().requires_grad_(True))
    with pytest.raises(NotImplementedError, match="out_pos"):
        BC.wasserstein_barycenter(x, w, pos, out_pos=pos.clone().requires_grad_(True))
    with pytest.raises(NotImplementedError, match="1-D grid"):
        BC.wasserstein_barycenter(x, w, pos.expand(12, 9).clone())
    with pytest.raises(NotImplementedError, match="weights"):
        BC.wasserstein_interpolate(x[0, 0], x[0, 1], torch.tensor(0.5, requires_grad=True), pos)
    with pytest.raises(ValueError, match="ascending"):
        BC.wasserstein_barycenter(x, w, pos, out_pos=pos.flip(0))
    with pytest.raises(ValueError):
        BC.wasserstein_barycenter(x[0, 0], w, pos)
    assert rec == [] and _capi.launch_count() == before


def test_abi_validation_before_any_launch():
    from sot_b200 import _capi
    lib = _capi.load()
    before = _capi.launch_count()
    fake = ctypes.c_void_p(16)

    def prob(N=2, K=3, n=9, M=9, flags=0, stride=0, ptr=16):
        return _capi.SotBarycenterProblem(N, K, n, M, ptr, ptr, stride, ptr, ptr, flags)

    def fwd(pr, out=fake):
        return lib.sot_barycenter_device(ctypes.byref(pr), out, None)

    def bwd(pr, up=fake, grad=fake):
        return lib.sot_barycenter_backward_device(ctypes.byref(pr), up, grad, None)

    assert lib.sot_barycenter_device(None, fake, None) == -1
    for flags in (_capi.SOT_CUT_SCALE, _capi.SOT_LIMIT, _capi.SOT_RAW_WEIGHTS, _capi.SOT_COMPLEX_INPUT, 64):
        assert fwd(prob(flags=flags)) == -1 and bwd(prob(flags=flags)) == -1
    assert b"SOT_SQUARE" in lib.sot_last_error()
    for bad in (prob(K=0), prob(n=0), prob(M=0), prob(N=-1), prob(stride=2), prob(ptr=0)):
        assert fwd(bad) == -1 and bwd(bad) == -1
    assert fwd(prob(), out=None) == -1
    assert bwd(prob(), up=None) == -1 and bwd(prob(), grad=None) == -1
    assert fwd(prob(K=4097, n=4097)) == -2 and b"2^24" in lib.sot_last_error()
    assert bwd(prob(K=1 << 14, n=1025)) == -2
    for empty in (prob(N=0), prob(N=0, K=0, ptr=0)):  # no barycenters: nothing is launched
        assert fwd(empty, out=None) == 0 and bwd(empty, up=None, grad=None) == 0
    assert _capi.launch_count() == before


# ---- fp64 model of the backward decomposition -------------------------------------------------------------------
def _model_grad(x, lam, pos, out_pos, G, square):
    """One barycenter in fp64 the way the kernels decompose the backward."""
    K, n = x.shape
    eps = np.float64(np.float32(O.SAFE_EPS))
    w = x * x if square else x
    mass = w.sum(1)
    mc = np.where(mass > eps, mass, eps)
    c = np.cumsum(w / mc[:, None], 1)
    flat = c.reshape(-1)
    order = np.argsort(flat, kind="stable")  # the merged slots: row first, then bin, on ties
    qs = flat[order]
    z = np.zeros_like(qs)
    for j in range(K):
        z += lam[j] * pos[np.minimum(np.searchsorted(c[j], qs, side="left"), n - 1)]
    M = out_pos.shape[0]
    b = np.clip(np.searchsorted(out_pos, z, side="right") - 1, 0, M - 2)
    f = np.where(z < out_pos[0], 1.0, np.where(z >= out_pos[-1], 0.0,
                                                (out_pos[b + 1] - z) / (out_pos[b + 1] - out_pos[b])))
    gamma = G[b] * f + G[b + 1] * (1 - f)
    dqs = gamma - np.append(gamma[1:], 0.0)  # dL/dqs_k = gamma_k - gamma_{k+1}
    dc = np.empty_like(flat)
    dc[order] = dqs  # one writer per CDF entry
    dc = dc.reshape(K, n)
    grad = np.empty_like(x)
    for j in range(K):
        suffix = np.cumsum(dc[j][::-1])[::-1]
        corr = np.dot(dc[j], c[j]) if mass[j] > eps else 0.0
        g = (suffix - corr) / mc[j]
        grad[j] = 2 * x[j] * g if square else g
    return grad, dqs, z


@pytest.mark.parametrize("square", [False, True])
@pytest.mark.parametrize("case", ["ties", "diracs", "random"])
def test_backward_decomposition_matches_the_oracle_autograd(square, case):
    rng = np.random.default_rng(7)
    K, n = 4, 9
    x = rng.random((K, n)) + 0.01
    if case == "ties":
        x[:, [0, 3, 4, 8]] = 0.0  # CDF plateaus: tie groups inside each row
        x[2] = x[0]  # identical rows: tie groups across rows
        x[3, 5:] *= 1e-9
    elif case == "diracs":
        x[:] = 0.0
        x[0, 2] = x[1, 6] = x[2, 6] = x[3, 0] = 1.0
    pos = np.linspace(0.0, 1.0, n)
    out_pos = np.concatenate(([-0.1], np.sort(rng.random(6)), [0.95]))  # non-uniform, atoms beyond both ends
    lam = rng.random(K)
    lam /= lam.sum()
    G = rng.standard_normal(out_pos.shape[0])
    got, dqs, z = _model_grad(x, lam, pos, out_pos, G, square)
    xt = torch.tensor(x[None], requires_grad=True)
    out = BO.barycenter(xt, torch.tensor(lam), torch.tensor(pos), torch.tensor(out_pos), square)
    (torch.tensor(G) * out[0]).sum().backward()
    want = xt.grad[0].numpy()
    assert np.abs(got - want).max() <= 1e-12 * max(np.abs(want).max(), 1.0)
    if case != "random":  # a tie group shares z, so only its last slot carries a gradient
        same = np.append(z[1:] == z[:-1], False)
        assert (dqs[same] == 0).all() and same.any()
