"""Pins oracle/sot_oracle.py to the reference: bit-for-bit against the committed golden fixtures
(generated from the unmodified reference by tests/golden/make_golden.py)."""
import numpy as np
import pytest
import torch

from oracle import sot_oracle as O
from tests import golden_io as G


@pytest.mark.parametrize("name", G.MODULE_CASES)
def test_module_cases_bit_exact(name):
    g = G.load(name)
    kw = G.oracle_kwargs(g["meta"]["ctor"])
    x, y, px, py = g["x"], g["y"], g["pos_x"], g["pos_y"]
    assert torch.equal(O.sot_loss(x, y, px, py, **kw), g["value"])
    assert torch.equal(O.sot_per_frame(x, y, px, py, **kw), g["rows"])
    _, gx, gy = O.sot_loss_and_grads(x, y, px, py, **kw)
    assert torch.equal(gx, g["grad_x"]) and torch.equal(gy, g["grad_y"])
    q = O.sot_quantiles(x, y, px, py, square=kw["square"], cut_scale=kw["cut_scale"])
    for got, key in zip(q[:5], ("uq", "vq", "qs", "cu", "cv")):
        assert torch.equal(got, g[key]), key


@pytest.mark.parametrize("p", [1, 2])
def test_fixed_grid_metric_path(p):
    g = G.load(f"fixedx65_p{p}")
    grid = torch.linspace(0, 1, 65)
    assert torch.equal(O.sot_loss(g["x"], g["y"], grid, grid, p=p), g["value"])
    assert torch.equal(O.sot_per_frame(g["x"], g["y"], grid, grid, p=p), g["rows"])
    assert torch.equal(O.sot_loss(g["x"], g["y"], grid, grid, p=p, dims=1), g["per_item"])


def test_hinge():
    g = G.load("fixedx65_hinge")
    grid = torch.linspace(0, 1, 65)
    x = g["x"].clone().requires_grad_(True)
    y = g["y"].clone().requires_grad_(True)
    v = O.sot_loss(x, y, grid, grid, p=2, square=True, hinge_gate=True, hinge_at=0.02)
    v.backward()
    assert torch.equal(v.detach(), g["value"])
    assert torch.equal(x.grad, g["grad_x"]) and torch.equal(y.grad, g["grad_y"])


@pytest.mark.parametrize("p,limit", [(1, False), (2, True)])
def test_module_level_w1d(p, limit):
    g = G.load(f"w1d_n37_m90_p{p}")
    uw = g["u_weights"].clone().requires_grad_(True)
    vw = g["v_weights"].clone().requires_grad_(True)
    rows = O.w1d_rows(g["u_values"], g["v_values"], uw, vw, p=p, limit=limit)
    rows.sum().backward()
    assert torch.equal(rows.detach(), g["rows"])
    assert torch.equal(uw.grad, g["grad_uw"]) and torch.equal(vw.grad, g["grad_vw"])
    out = O.transport_plan(g["u_values"], g["v_values"], g["u_weights"], g["v_weights"])
    for got, key in zip(out[:5], ("uq", "vq", "qs", "cu", "cv")):
        assert torch.equal(got, g[key]), key
    u = G.load("w1d_uniform_p2")
    assert torch.equal(O.w1d_rows(u["u_values"], u["v_values"], p=2), u["rows"])


def test_quantile_function_and_kats():
    g = G.load("quantile_function")
    assert torch.equal(O.lower_bound_lookup(g["qs"], g["cws"], g["xs"])[0], g["out"])
    k = G.load("kat_diracs")
    grid = torch.linspace(0, 1, 9)
    assert O.sot_loss(k["x"], k["y"], grid, grid, p=1).item() == pytest.approx(0.5, abs=1e-7) == k["w1"].item()
    assert O.sot_loss(k["x"], k["y"], grid, grid, p=2).item() == pytest.approx(0.25, abs=1e-7) == k["w2"].item()
    assert O.sot_loss(k["x"], k["x"], grid, grid, p=2).item() == 0.0 == k["zero"].item()
    z = torch.zeros(1, 9)
    assert torch.equal(O.sot_loss(z, k["y"], grid, grid, p=2, cut_scale=True, limit=True), k["dead_cut"])
    assert torch.equal(O.sot_loss(z, k["y"], grid, grid, p=2), k["dead_nocut"])


def test_p_below_one_asserts():
    grid = torch.linspace(0, 1, 9)
    with pytest.raises(AssertionError):
        O.sot_loss(torch.rand(2, 9), torch.rand(2, 9), grid, grid, p=0.5)


def test_closed_form_matches_stable_autograd_fp64():
    g = G.load("sot512_nocut")
    x, y = g["x"].reshape(-1, 257)[:6].double(), g["y"].reshape(-1, 257)[:6].double()
    pos = g["pos_x"].double()
    for cut in (False, True):
        rows, gx, gy = O.sot_loss_and_grads(x, y, pos, pos, upstream=torch.ones(6, dtype=torch.float64), p=2,
                                            square=True, cut_scale=cut, limit=cut, stable=True)
        cl, cgx, cgy = O.closed_form_backward(x.numpy(), y.numpy(), pos.numpy(), pos.numpy(), 2, True, cut, cut)
        assert np.allclose(cl, rows.numpy(), rtol=1e-13, atol=0)
        assert np.abs(cgx - gx.numpy()).max() <= 1e-13 * np.abs(cgx).max()
        assert np.abs(cgy - gy.numpy()).max() <= 1e-13 * np.abs(cgy).max()


@pytest.mark.parametrize("cut", [True, False])
@pytest.mark.parametrize("n_fft", [512, 2048])
def test_live_reference_bit_exact(cut, n_fft):
    """The paper's configurations (p = 2, squared distance, the project's linear grid, with and without the cutoff)
    against what the unmodified reference's `Wasserstein1D` returned for them: value and both gradients, bit for bit.
    The reference's outputs are the ones make_golden.py recorded, so the comparison needs no copy of the reference."""
    from sot_b200 import synthetic as S
    g = G.load(f"sot{n_fft}_{'cut' if cut else 'nocut'}")
    ctor = g["meta"]["ctor"]
    assert (ctor["p"], ctor["square_dist"], ctor["dont_normalize"], ctor["limit_quantile_range"]) == (2, True, cut, cut)
    x, y, pos = g["x"], g["y"], g["pos_x"]
    assert torch.equal(pos, S.linear_positions(n_fft)) and torch.equal(g["pos_y"], pos)
    kw = dict(p=2, square=True, cut_scale=cut, limit=cut)
    assert torch.equal(O.sot_loss(x, y, pos, pos.clone(), **kw), g["value"])
    _, gx, gy = O.sot_loss_and_grads(x, y, pos, pos.clone(), **kw)
    assert torch.equal(gx, g["grad_x"]) and torch.equal(gy, g["grad_y"])
