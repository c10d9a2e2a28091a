"""What the host prologue of the SOT loss hands to the CUDA entry points.

Recording stand-ins take the place of the `_capi` launch wrappers, so the public surface (`Wasserstein1D`, the sharded
module, `wasserstein_1d`) runs on CPU tensors.  Each test checks what reached `_capi`: rows, supports, flags, shapes,
dtypes and contiguity.  The expected tensors are computed directly from the inputs: `reshape`, `float`, `abs`,
`torch.sort` of the positions and the matching permutation of the rows."""
import pytest
import torch

from sot_b200 import _capi, losses as L, sharding

SQUARE, CUT, LIMIT, RAW, UNIFORM = (_capi.SOT_SQUARE, _capi.SOT_CUT_SCALE, _capi.SOT_LIMIT, _capi.SOT_RAW_WEIGHTS,
                                    _capi.SOT_UNIFORM_GRID)


@pytest.fixture
def calls(monkeypatch):
    """Replaces the launch wrappers `losses` calls with recorders; returns the list of (name, arguments)."""
    from tests import fake_kernels
    log = []

    def forward(u, v, pos_u, pos_v, p, flags):
        log.append(("forward", dict(u=u, v=v, pu=pos_u, pv=pos_v, p=p, flags=flags)))
        return torch.ones(u.shape[0])

    def forward_backward(u, v, pos_u, pos_v, p, flags, upstream=None, want_loss=True, want_gu=True, want_gv=True):
        log.append(("forward_backward", dict(u=u, v=v, pu=pos_u, pv=pos_v, p=p, flags=flags, upstream=upstream,
                                             want=(want_loss, want_gu, want_gv))))
        return (torch.ones(u.shape[0]) if want_loss else None, torch.ones_like(u) if want_gu else None,
                torch.ones_like(v) if want_gv else None)

    def mean_step(u, v, pos_u, pos_v, p, flags, grad_scale, mean_scale, want_gu=True, want_gv=True, **kw):
        log.append(("mean_step", dict(u=u, v=v, pu=pos_u, pv=pos_v, p=p, flags=flags, grad_scale=grad_scale,
                                      mean_scale=mean_scale, want=(want_gu, want_gv), kw=kw)))
        return (torch.ones(()), None, torch.ones_like(u) if want_gu else None,
                torch.ones_like(v) if want_gv else None)

    def scale_inplace(a, b, scale):
        log.append(("scale_inplace", dict(a=a, b=b, scale=scale)))

    def scale_rows(unit, scale):
        log.append(("scale_rows", dict(unit=unit, scale=scale)))
        return unit * scale[:, None]

    def quantiles(u, v, pos_u, pos_v, flags, from_cdf=False, want_indices=False):
        log.append(("quantiles", dict(u=u, v=v, pu=pos_u, pv=pos_v, flags=flags, want_indices=want_indices)))
        N, n, m = u.shape[0], u.shape[1], v.shape[1]
        out = (torch.zeros(N, n + m), torch.zeros(N, n + m), torch.zeros(N, n + m), torch.zeros(N, n),
               torch.zeros(N, m), torch.zeros(N, n + m, dtype=torch.int32), torch.zeros(N, n + m, dtype=torch.int32))
        return out if want_indices else out[:5]

    for name, fn in dict(forward=forward, forward_backward=forward_backward, mean_step=mean_step,
                         scale_inplace=scale_inplace, scale_rows=scale_rows, quantiles=quantiles).items():
        monkeypatch.setattr(_capi, name, fn)
    fake_kernels.allow_cpu_rows(monkeypatch, L)
    return log


def _same(got, want):
    assert got.dtype == want.dtype, (got.dtype, want.dtype)
    assert tuple(got.shape) == tuple(want.shape), (tuple(got.shape), tuple(want.shape))
    assert got.is_contiguous()
    assert torch.equal(got, want)


def _launch(rec, u, v, pu, pv, flags, p=None):
    _same(rec["u"], u), _same(rec["v"], v), _same(rec["pu"], pu), _same(rec["pv"], pv)
    assert rec["flags"] == flags, (rec["flags"], flags)
    assert not rec["pu"].requires_grad and not rec["pv"].requires_grad
    if p is not None:
        assert rec["p"] == float(p) and type(rec["p"]) is float


def _names(log):
    return [name for name, _ in log]


def _sorted(pos, rows):
    """Positions sorted along the bins, and the rows permuted to match (a stable sort, like the reference's)."""
    if pos.ndim == 1:
        s, perm = torch.sort(pos, stable=True)
        return s, rows[:, perm]
    s, perm = torch.sort(pos, dim=1, stable=True)
    return s, torch.gather(rows, 1, perm)


def _rand(*shape, seed, dtype=torch.float32):
    return torch.rand(*shape, generator=torch.Generator().manual_seed(seed)).to(dtype)


def _crand(*shape, seed):
    return torch.complex(_rand(*shape, seed=seed), _rand(*shape, seed=seed + 1))


# ---- the plain mean ------------------------------------------------------------------------------------------------
def test_mean_3d_fixed_x_is_uniform_and_unsorted(calls):
    x, y = _rand(2, 3, 33, seed=1).requires_grad_(True), _rand(2, 3, 33, seed=2).requires_grad_(True)
    mod = L.Wasserstein1D(p=2, fixed_x=33, square_dist=True)
    value = mod(x, y)
    value.backward()
    assert _names(calls) == ["mean_step", "scale_inplace"]
    rec = calls[0][1]
    grid = torch.linspace(0, 1, 33)
    _launch(rec, x.detach().reshape(6, 33), y.detach().reshape(6, 33), grid, grid, SQUARE | UNIFORM, p=2)
    assert rec["grad_scale"] == 1 / 6 and rec["mean_scale"] == 1 / 6 and rec["want"] == (True, True)
    assert rec["kw"] == {}
    scaled = calls[1][1]
    assert scaled["scale"].dtype == torch.float32 and scaled["scale"].shape == (1,)
    assert value.dtype == torch.float32 and value.shape == ()


def test_mean_2d_float64_unsorted_shared_support(calls):
    x, y = _rand(6, 33, seed=3, dtype=torch.float64), _rand(6, 33, seed=4, dtype=torch.float64)
    pos_x, pos_y = _rand(33, seed=5), _rand(33, seed=6)
    mod = L.Wasserstein1D(p=1, dont_normalize=True, limit_quantile_range=True)
    value = mod(x.requires_grad_(True), y.requires_grad_(True), x_pos=pos_x, y_pos=pos_y)
    assert _names(calls) == ["mean_step"]
    pu, u = _sorted(pos_x, x.detach().float())
    pv, v = _sorted(pos_y, y.detach().float())
    _launch(calls[0][1], u, v, pu, pv, CUT | LIMIT, p=1)
    assert value.dtype == torch.float64


def test_mean_half_with_expanded_supports(calls):
    x, y = _rand(2, 3, 33, seed=7, dtype=torch.float16), _rand(2, 3, 33, seed=8, dtype=torch.float16)
    grid = torch.linspace(0, 1, 33)
    mod = L.Wasserstein1D(p=2, square_dist=True, backward_mode="recompute")
    value = mod(x.requires_grad_(True), y.requires_grad_(True), x_pos=grid.expand(6, 33), y_pos=grid[None])
    value.backward()
    assert _names(calls) == ["mean_step", "mean_step"]
    fwd, bwd = calls[0][1], calls[1][1]
    _launch(fwd, x.detach().float().reshape(6, 33), y.detach().float().reshape(6, 33), grid, grid, SQUARE | UNIFORM)
    assert fwd["want"] == (False, False)
    _launch(bwd, fwd["u"], fwd["v"], grid, grid, SQUARE | UNIFORM)
    assert bwd["want"] == (True, True) and bwd["mean_scale"] == 0.0 and bwd["kw"]["want_mean"] is False
    assert value.dtype == torch.float32


def test_mean_per_frame_supports(calls):
    x, y = _rand(2, 3, 33, seed=9), _rand(2, 3, 33, seed=10)
    pos_x, pos_y = _rand(2, 3, 33, seed=11), _rand(6, 33, seed=12)
    L.Wasserstein1D(p=3)(x, y, x_pos=pos_x, y_pos=pos_y)
    pu, u = _sorted(pos_x.reshape(6, 33), x.reshape(6, 33))
    pv, v = _sorted(pos_y, y.reshape(6, 33))
    _launch(calls[0][1], u, v, pu, pv, 0, p=3)


def test_require_sort_false_keeps_the_order(calls):
    x, y = _rand(6, 33, seed=13), _rand(6, 33, seed=14)
    pos_x, pos_y = _rand(6, 33, seed=15), _rand(33, seed=16)
    L.Wasserstein1D(p=1, require_sort=False)(x, y, x_pos=pos_x, y_pos=pos_y)
    _launch(calls[0][1], x, y, pos_x, pos_y, 0)


# ---- complex rows ----------------------------------------------------------------------------------------------------
def test_complex_rows_stay_complex_for_the_loss_launch(calls):
    x, y = _crand(2, 3, 33, seed=17).requires_grad_(True), _crand(2, 3, 33, seed=19).requires_grad_(True)
    grid = torch.linspace(0, 1, 33)
    mod = L.Wasserstein1D(p=1, hinge=True)
    loss = mod(x, y, x_pos=grid, y_pos=grid, hinge=0.25)
    loss.backward()
    assert _names(calls) == ["forward_backward", "scale_rows", "scale_rows"]
    rec = calls[0][1]
    _launch(rec, x.detach().reshape(6, 33), y.detach().reshape(6, 33), grid, grid, UNIFORM)
    assert rec["upstream"] is None and rec["want"] == (True, True, True)
    for _, scaled in calls[1:]:
        unit = scaled["unit"]
        if not unit.is_complex():  # the interleaved (re, im) view of the complex unit gradient
            unit = torch.view_as_complex(unit.reshape(6, 33, 2))
        _same(unit, torch.ones(6, 33, dtype=torch.complex64))
        _same(scaled["scale"], torch.full((6,), 1 / 6))
    assert torch.equal(x.grad, torch.full((2, 3, 33), 1 / 6, dtype=torch.complex64))
    assert loss.item() == pytest.approx(0.75)


def test_mixed_complex_and_real_rows_take_the_magnitude(calls):
    x, y = _crand(6, 33, seed=21), _rand(6, 33, seed=23)
    grid = torch.linspace(0, 1, 33)
    L.Wasserstein1D(p=2)(x, y, x_pos=grid, y_pos=grid)
    L.Wasserstein1D(p=2)(y, x, x_pos=grid, y_pos=grid)
    _launch(calls[0][1], x.abs(), y, grid, grid, UNIFORM)
    _launch(calls[1][1], y, x.abs(), grid, grid, UNIFORM)


def test_long_complex_rows_take_the_magnitude(calls):
    F = _capi.MAX_COMPLEX_BINS + 1
    x, y = _crand(2, F, seed=25), _crand(2, F, seed=27)
    pos = _rand(F, seed=29)
    L.Wasserstein1D(p=2, square_dist=True)(x, y, x_pos=pos, y_pos=pos)
    pu, u = _sorted(pos, x.abs())
    _, v = _sorted(pos, y.abs())
    _launch(calls[0][1], u, v, pu, pu, SQUARE)


def test_complex_raw_weights_are_refused(calls):
    w = _crand(2, 9, seed=31)
    with pytest.raises(TypeError, match="weights must be real"):
        L.wasserstein_1d(_rand(2, 9, seed=33), _rand(2, 9, seed=34), w, w)
    assert calls == []


# ---- per-frame values: hinge and dims ------------------------------------------------------------------------------
def test_hinge_and_dims_run_per_frame(calls):
    x, y = _rand(2, 3, 33, seed=35, dtype=torch.float64), _rand(2, 3, 33, seed=36, dtype=torch.float64)
    pos = _rand(33, seed=37)
    mod = L.Wasserstein1D(p=2, square_dist=True, hinge=True)
    loss = mod(x, y, x_pos=pos, y_pos=pos, hinge=0.5)
    assert loss.dtype == torch.float64 and loss.item() == pytest.approx(0.5)
    per_frame = L.Wasserstein1D(p=2)(x.float().requires_grad_(True), y.float(), x_pos=pos, y_pos=pos, dims=1)
    assert per_frame.shape == (2,)
    assert _names(calls) == ["forward", "forward_backward"]
    pu, u = _sorted(pos, x.float().reshape(6, 33))
    _, v = _sorted(pos, y.float().reshape(6, 33))
    _launch(calls[0][1], u, v, pu, pu, SQUARE, p=2)
    _launch(calls[1][1], u, v, pu, pu, 0, p=2)
    assert calls[1][1]["want"] == (True, True, False)


def test_empty_batch_runs_per_frame(calls):
    grid = torch.linspace(0, 1, 33)
    value = L.Wasserstein1D(p=2)(torch.rand(0, 3, 33), torch.rand(0, 3, 33), x_pos=grid, y_pos=grid)
    assert _names(calls) == ["forward"] and torch.isnan(value)
    _launch(calls[0][1], torch.rand(0, 33), torch.rand(0, 33), grid, grid, UNIFORM)


def test_sharded_module_without_ranks(calls):
    """A single process has no peers: the mean path is the plain module's, and the per-frame path reduces with
    `sharding.global_mean`, whose value is float32 even for float64 inputs."""
    x, y = _rand(2, 3, 33, seed=38, dtype=torch.float64), _rand(2, 3, 33, seed=39, dtype=torch.float64)
    grid = torch.linspace(0, 1, 33)
    mod = sharding.ShardedWasserstein1D(p=2, fixed_x=33, square_dist=True)
    assert mod(x, y).dtype == torch.float64
    hinged = sharding.ShardedWasserstein1D(p=2, fixed_x=33, square_dist=True, hinge=True)
    loss = hinged(x, y, hinge=0.5)
    assert loss.dtype == torch.float32 and loss.shape == () and loss.item() == pytest.approx(0.5)
    local = hinged(x, y, hinge=0.5, dims=1)
    assert local.dtype == torch.float64 and local.shape == (2,)
    empty = mod(torch.rand(0, 3, 33), torch.rand(0, 3, 33))
    assert empty.dtype == torch.float32 and torch.isnan(empty)
    assert _names(calls) == ["mean_step", "forward", "forward", "forward"]
    u, v = x.float().reshape(6, 33), y.float().reshape(6, 33)
    for _, rec in calls[:3]:
        _launch(rec, u, v, grid, grid, SQUARE | UNIFORM, p=2)


# ---- quantile taps and wasserstein_1d ------------------------------------------------------------------------------
def test_return_quantiles_takes_magnitudes_and_no_limit_or_grid_flag(calls):
    x, y = _crand(2, 3, 33, seed=41), _crand(2, 3, 33, seed=43)
    grid = torch.linspace(0, 1, 33)
    mod = L.Wasserstein1D(p=2, square_dist=True, dont_normalize=True, limit_quantile_range=True)
    out = mod(x, y, x_pos=grid, y_pos=grid, return_quantiles=True)
    assert [tuple(t.shape) for t in out] == [(2, 3, 66)] * 3 + [(2, 3, 33)] * 2
    assert _names(calls) == ["quantiles"]
    rec = calls[0][1]
    _launch(rec, x.abs().reshape(6, 33), y.abs().reshape(6, 33), grid, grid, SQUARE | CUT)
    assert rec["want_indices"] is False


def test_return_quantiles_sorts_per_frame_supports(calls):
    x, y = _rand(6, 33, seed=45, dtype=torch.float64), _rand(6, 33, seed=46)
    pos_x, pos_y = _rand(6, 33, seed=47), _rand(33, seed=48)
    L.Wasserstein1D(p=1)(x, y, x_pos=pos_x, y_pos=pos_y, return_quantiles=True)
    pu, u = _sorted(pos_x, x.float())
    pv, v = _sorted(pos_y, y)
    _launch(calls[0][1], u, v, pu, pv, 0)


@pytest.mark.parametrize("require_sort", [True, False])
def test_wasserstein_1d(calls, require_sort):
    u_values, v_values = _rand(4, 9, seed=49), _rand(4, 7, seed=50, dtype=torch.float64)
    u_weights, v_weights = _rand(4, 9, seed=51), _rand(4, 7, seed=52, dtype=torch.float64)
    rows = L.wasserstein_1d(u_values, v_values, u_weights, v_weights, p=2, require_sort=require_sort,
                            limit_quantile_range=True)
    L.wasserstein_1d(u_values, v_values, u_weights, v_weights, require_sort=require_sort, return_quantiles=True)
    L.wasserstein_1d(u_values, v_values, p=3, require_sort=require_sort)
    assert rows.shape == (4,)
    assert _names(calls) == ["forward", "quantiles", "forward"]
    pu, wu, pv, wv = u_values, u_weights, v_values.float(), v_weights.float()
    if require_sort:
        (pu, wu), (pv, wv) = _sorted(pu, wu), _sorted(pv, wv)
    _launch(calls[0][1], wu, wv, pu, pv, RAW | LIMIT, p=2)
    _launch(calls[1][1], wu, wv, pu, pv, RAW)
    _launch(calls[2][1], torch.full((4, 9), 1 / 9), torch.full((4, 7), 1 / 7), pu, pv, RAW, p=3)


# ---- positions that require a gradient ------------------------------------------------------------------------------
@pytest.mark.parametrize("shared", [True, False])
def test_position_gradients_see_the_loss_launchs_rows(calls, shared):
    """The plan launch behind the position gradients must see the sorted supports and permuted rows of the loss
    launch, and carries neither the cutoff nor the uniform-grid flag."""
    x, y = _rand(2, 3, 33, seed=53), _rand(2, 3, 33, seed=54)
    shape = (33,) if shared else (2, 3, 33)
    pos_x, pos_y = _rand(*shape, seed=55).requires_grad_(True), _rand(*shape, seed=56).requires_grad_(True)
    mod = L.Wasserstein1D(p=2, square_dist=True, dont_normalize=True, limit_quantile_range=True)
    mod(x.requires_grad_(True), y.requires_grad_(True), x_pos=pos_x, y_pos=pos_y).backward()
    assert _names(calls) == ["mean_step", "quantiles", "scale_inplace"]
    flat = (33,) if shared else (6, 33)
    pu, u = _sorted(pos_x.detach().reshape(flat), x.detach().reshape(6, 33))
    pv, v = _sorted(pos_y.detach().reshape(flat), y.detach().reshape(6, 33))
    _launch(calls[0][1], u, v, pu, pv, SQUARE | CUT | LIMIT, p=2)
    plan = calls[1][1]
    _launch(plan, u, v, pu, pv, SQUARE | CUT)
    assert plan["want_indices"] is True
    assert pos_x.grad is not None and pos_y.grad is not None and pos_x.grad.shape == shape


def test_position_gradients_of_ascending_complex_rows(calls):
    x, y = _crand(4, 33, seed=57), _crand(4, 33, seed=59)
    grid = torch.linspace(0, 1, 33).requires_grad_(True)
    rows = L.sot_frames(x, y, grid, grid, p=1, backward_mode="fused")
    rows.sum().backward()
    assert _names(calls) == ["forward", "quantiles"]
    g = grid.detach()
    _launch(calls[0][1], x, y, g, g, UNIFORM, p=1)
    _launch(calls[1][1], x.abs(), y.abs(), g, g, 0)
    assert grid.grad is not None


def test_position_gradients_of_wasserstein_1d_values(calls):
    u_values, v_values = _rand(4, 9, seed=61).requires_grad_(True), _rand(4, 9, seed=62).requires_grad_(True)
    L.wasserstein_1d(u_values, v_values, p=2).sum().backward()
    assert _names(calls) == ["forward", "quantiles"]
    pu, wu = _sorted(u_values.detach(), torch.full((4, 9), 1 / 9))
    pv, wv = _sorted(v_values.detach(), torch.full((4, 9), 1 / 9))
    _launch(calls[0][1], wu, wv, pu, pv, RAW, p=2)
    _launch(calls[1][1], wu, wv, pu, pv, RAW)
    assert u_values.grad is not None and v_values.grad is not None


# ---- refusals --------------------------------------------------------------------------------------------------------
def test_prologue_refusals(calls):
    grid = torch.linspace(0, 1, 9)
    mod = L.Wasserstein1D(p=2)
    with pytest.raises(ValueError, match="frames"):
        mod(torch.rand(4, 9), torch.rand(3, 9), x_pos=grid, y_pos=grid)
    with pytest.raises(ValueError, match="positions for"):
        mod(torch.rand(4, 9), torch.rand(4, 9), x_pos=torch.linspace(0, 1, 8), y_pos=grid)
    with pytest.raises(ValueError, match="has shape"):
        mod(torch.rand(4, 9), torch.rand(4, 9), x_pos=torch.rand(3, 9), y_pos=grid)
    with pytest.raises(TypeError, match="must be float32"):
        mod(torch.ones(4, 9, dtype=torch.int32), torch.rand(4, 9), x_pos=grid, y_pos=grid)
    with pytest.raises(ValueError, match="batch, time, features"):
        mod(torch.rand(9), torch.rand(9), x_pos=grid, y_pos=grid)
    assert calls == []


def test_loss_grad_host_refuses_mismatched_shapes():
    """The host-buffer entry point applies the shape rules of the device entry points before it reaches the library:
    a (1, n) position tensor or fewer frames in `y` than in `x` would make it read past a buffer."""
    x, y, pos = torch.rand(4, 9), torch.rand(4, 9), torch.linspace(0, 1, 9)
    with pytest.raises(ValueError, match="x_pos"):
        _capi.loss_grad_host(x, y, pos[None], pos, 2.0, 0)
    with pytest.raises(ValueError, match=r"\(N, n\) and \(N, m\)"):
        _capi.loss_grad_host(x, y[:3], pos, pos, 2.0, 0)
    with pytest.raises(ValueError, match="y_pos"):
        _capi.loss_grad_host(x, y, pos, torch.rand(3, 9), 2.0, 0)
    with pytest.raises(ValueError, match="CPU tensor"):
        _capi.loss_grad_host(x.double(), y, pos, pos, 2.0, 0)
