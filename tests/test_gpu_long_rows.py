"""Rows longer than one CTA's shared memory holds: the split-frame path (csrc/sot_long.cu).

Gates (float32), the ones of tests/test_gpu_parity.py:
  * split path forced onto rows that fit (`set_tuning(-1, 0, 0)`) against the shared-memory kernels on the golden
    fixtures: per-frame loss rel 1e-5 without the cutoff (and as close to the float64 value as the reference's float32
    value is); with it, the batch mean as close to the float64 value as the reference's float32 value is; gradients
    through the fp64-relative gate (b) at ratio 3;
  * long rows against the oracle (the reference's formula, pinned bit for bit): the batch loss within rel 1e-5 of the
    reference's float32 value (cutoff mode: as close to its float64 value as the float32 one is), gradients through
    gate (b) at ratio 3 -- the gates of `test_rows_that_fill_a_kernel_configuration_exactly`.
"""
import numpy as np
import pytest
import torch

from oracle import sot_oracle as O
from tests import golden_io as G
from tests.test_gpu_parity import _assert_grad_gate

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


@pytest.fixture(scope="module")
def capi():
    from sot_b200 import _capi
    _capi.load()
    return _capi


@pytest.fixture(scope="module")
def L():
    from sot_b200 import losses
    return losses


class _forced_split:
    def __init__(self, capi):
        self.capi = capi

    def __enter__(self):
        self.capi.set_tuning(-1, 0, 0)

    def __exit__(self, *exc):
        self.capi.set_tuning(0, 0, 0)
        return False


def _run_module(L, x, y, px, py, ctor, mode="onepass"):
    mod = L.Wasserstein1D(**ctor, backward_mode=mode)
    xd, yd = x.to(DEV).requires_grad_(True), y.to(DEV).requires_grad_(True)
    value = mod(xd, yd, x_pos=px.to(DEV), y_pos=py.to(DEV))
    value.backward()
    with torch.no_grad():
        rows = mod(x.reshape(-1, 1, x.shape[-1]).to(DEV), y.reshape(-1, 1, y.shape[-1]).to(DEV), x_pos=px.to(DEV),
                   y_pos=py.to(DEV), dims=1)
    return value.detach(), rows.reshape(-1), xd.grad, yd.grad


# ------------------------------------------------------------------------------------------
# 1. the split path on rows the shared-memory kernels hold
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["sot2048_cut", "sot2048_nocut", "sot2048_logf_unsorted", "sot512_cut",
                                  "sot512_nocut", "sot512_p1_nosquare", "sot512_p3", "sot512_logf_cut"])
def test_split_path_forced_on_fixtures(capi, L, name):
    g = G.load(name)
    ctor = dict(g["meta"]["ctor"])
    kw = G.oracle_kwargs(ctor)
    F = g["x"].shape[-1]
    ref = _run_module(L, g["x"], g["y"], g["pos_x"], g["pos_y"], ctor)
    before = capi.launch_count()
    with _forced_split(capi):
        mine = _run_module(L, g["x"], g["y"], g["pos_x"], g["pos_y"], ctor)
    assert capi.launch_count() > before
    xs, ys = g["x"].reshape(-1, F), g["y"].reshape(-1, F)
    rows64, t64x, t64y = O.sot_loss_and_grads(xs.double(), ys.double(), g["pos_x"].double(), g["pos_y"].double(),
                                              stable=True, **kw)
    if not kw["limit"]:
        # the two paths sum different groups of bins locally (16 here, 17 or 33 there): CDFs a few ulp apart, per-frame
        # losses up to 4.8e-6 apart on sot512_nocut (measured); each as close to the float64 value as the reference is
        rel = (mine[1] - ref[1]).abs() / ref[1].abs().clamp_min(1e-30)
        assert rel.max().item() <= 1e-5, rel.max().item()
        _assert_rows_close(mine[1].cpu(), O.sot_per_frame(xs, ys, g["pos_x"], g["pos_y"], **kw), rows64)
    else:
        # the strict `qs > 1` mask decides over whole slots on the last ulp of the CDFs: as close to the float64 value
        # as the reference's float32 value is (sot2048_cut: 2.3e-8 here, 7.1e-5 for the reference, measured)
        v64 = rows64.mean().item()
        slack = max(1e-5, 1.5 * abs(g["value"].item() - v64) / abs(v64))
        assert abs(mine[0].item() - v64) <= slack * abs(v64), (mine[0].item(), g["value"].item(), v64)
    N = g["x"].reshape(-1, F).shape[0]
    for mine_g, ref32, t64, nm in ((mine[2], g["grad_x"], t64x, "x"), (mine[3], g["grad_y"], t64y, "y")):
        _assert_grad_gate(mine_g.cpu().reshape(-1, F) * N, ref32.reshape(-1, F) * N, t64.reshape(-1, F) * N,
                          f"{name} forced split grad_{nm}", 3.0)


def test_split_path_forced_on_module_level_w1d(capi, L):
    for p, limit in ((1, False), (2, True)):
        g = G.load(f"w1d_n37_m90_p{p}")
        with _forced_split(capi):
            uw = g["u_weights"].to(DEV).requires_grad_(True)
            vw = g["v_weights"].to(DEV).requires_grad_(True)
            rows = L.wasserstein_1d(g["u_values"].to(DEV), g["v_values"].to(DEV), uw, vw, p=p,
                                    limit_quantile_range=limit)
            rows.sum().backward()
        assert torch.allclose(rows.detach().cpu(), g["rows"], rtol=1e-5, atol=1e-8)


# ------------------------------------------------------------------------------------------
# 2. long rows against the oracle
# ------------------------------------------------------------------------------------------
def _spectra(n_frames, n, m, seed, zero_runs=False):
    gen = torch.Generator().manual_seed(seed)
    x = torch.rand(n_frames, n, generator=gen) ** 4 + 1e-4
    y = torch.rand(n_frames, m, generator=gen) ** 4 + 1e-4
    if zero_runs:  # runs of thousands of zero bins across the 4096-bin tiles and the merge chunks
        for r in range(n_frames):
            for lo in (1000 + 37 * r, 4000, 8190, 12000):
                x[r, lo:min(n, lo + 3000)] = 0.0
                y[r, lo + 500:min(m, lo + 2500)] = 0.0
    return x, y


def _assert_rows_close(mine, r32, r64):
    tol = torch.maximum(torch.full_like(r64, 1e-5), 1.5 * (r32.double() - r64).abs() / r64.abs())
    err = (mine.double() - r64).abs()
    assert (err <= tol * r64.abs() + 1e-12).all(), (err / r64.abs()).max().item()


def _grid(kind, n):
    if kind == "uniform":
        return torch.linspace(0, 1, n)
    f = torch.linspace(1.0, 24000.0, n)  # log-f: ascending, non-uniform
    return (torch.log2(f) / np.log2(24000.0)).float()


CASES = [
    # n, m, frames, p, square, cut, limit, support, grid, zero_runs
    (8449, 8449, 6, 2, True, False, False, "shared", "uniform", False),
    (8449, 8449, 5, 2, True, True, True, "shared", "uniform", False),
    (16385, 16385, 4, 2, True, True, True, "shared", "uniform", True),
    (16385, 16385, 3, 1, False, False, False, "per-frame", "logf", False),
    (16385, 9000, 3, 2, True, False, False, "shared", "logf", False),
    (32769, 32769, 2, 3.5, True, False, True, "shared", "logf", True),
    (32769, 32769, 2, 2, False, True, False, "unsorted", "uniform", False),
    (65536, 65536, 2, 1, True, False, False, "per-frame", "uniform", True),
    (65536, 65536, 1, 2, True, False, True, "shared", "uniform", False),
    (1048576, 1048576, 1, 2, True, False, False, "shared", "uniform", False),
]


@pytest.mark.parametrize("case", CASES, ids=lambda c: f"{c[0]}x{c[1]}-f{c[2]}-p{c[3]}-{c[7]}-{c[8]}")
def test_long_rows_against_the_oracle(capi, L, case):
    n, m, N, p, square, cut, limit, support, grid, zero_runs = case
    x, y = _spectra(N, n, m, seed=n + m + N, zero_runs=zero_runs)
    px, py = _grid(grid, n), _grid(grid, m)
    if support == "per-frame":
        px = px.unsqueeze(0).repeat(N, 1)
        py = (py.unsqueeze(0) + 1e-3 * torch.arange(N).unsqueeze(1)).contiguous()
    elif support == "unsorted":
        perm = torch.randperm(n, generator=torch.Generator().manual_seed(1))
        px, py = px[perm].contiguous(), py[perm].contiguous()
    kw = dict(p=p, square=square, cut_scale=cut, limit=limit)
    rows32, g32x, g32y = O.sot_loss_and_grads(x, y, px, py, stable=True, **kw)
    rows64, g64x, g64y = O.sot_loss_and_grads(x.double(), y.double(), px.double(), py.double(), stable=True, **kw)
    ctor = dict(p=p, square_dist=square, dont_normalize=cut, limit_quantile_range=limit)
    value, rows, gx, gy = _run_module(L, x, y, px, py, ctor)
    # the batch loss and every frame: within 1e-5 of the float64 value, or as close to it as the reference's own
    # float32 value is (long rows: its fp32 CDFs drift further than that; cutoff mode: the strict `qs > 1` mask)
    ref32, ref64 = rows32.double().mean().item(), rows64.mean().item()
    slack = max(1e-5, 1.5 * abs(ref32 - ref64) / abs(ref64))
    assert abs(value.item() - ref64) <= slack * abs(ref64), (value.item(), ref32, ref64)
    _assert_rows_close(rows.cpu(), rows32, rows64)
    _assert_grad_gate(gx.cpu(), g32x, g64x, f"{case} d/dtarget", 3.0)
    _assert_grad_gate(gy.cpu(), g32y, g64y, f"{case} d/dprediction", 3.0)


@pytest.mark.parametrize("atoms,p,limit", [(20000, 1, False), (50000, 2, True)])
def test_long_module_level_w1d_raw_weights(L, atoms, p, limit):
    gen = torch.Generator().manual_seed(atoms)
    uv = torch.randn(3, atoms, generator=gen)
    vv = torch.randn(3, atoms + 123, generator=gen) * 1.5 + 0.2
    uw = torch.rand(3, atoms, generator=gen)
    vw = torch.rand(3, atoms + 123, generator=gen)
    uw, vw = uw / uw.sum(1, keepdim=True), vw / vw.sum(1, keepdim=True)

    def ref(dtype):
        a, b = uw.to(dtype).clone().requires_grad_(True), vw.to(dtype).clone().requires_grad_(True)
        rows = O.w1d_rows(uv.to(dtype), vv.to(dtype), a, b, p=p, limit=limit, stable=True)
        ga, gb = torch.autograd.grad(rows.sum(), (a, b))
        return rows.detach(), ga, gb

    r32, a32, b32 = ref(torch.float32)
    r64, a64, b64 = ref(torch.float64)
    a, b = uw.to(DEV).requires_grad_(True), vw.to(DEV).requires_grad_(True)
    rows = L.wasserstein_1d(uv.to(DEV), vv.to(DEV), a, b, p=p, limit_quantile_range=limit)
    rows.sum().backward()
    _assert_rows_close(rows.detach().cpu(), r32, r64)
    _assert_grad_gate(a.grad.cpu(), a32, a64, "raw weights d/du", 3.0)
    _assert_grad_gate(b.grad.cpu(), b32, b64, "raw weights d/dv", 3.0)


def test_degenerate_frames_and_batches(capi, L):
    n = 16385
    x, y = _spectra(7, n, n, seed=5)
    x[2] = 0.0  # an all-zero target row: clamped mass, like the reference's safe_divide
    y[4, 100] = float("nan")  # poisons frame 4 only
    pos = torch.linspace(0, 1, n)
    loss, gu, gv = capi.forward_backward(x.to(DEV), y.to(DEV), pos.to(DEV), pos.to(DEV), 2.0, capi.SOT_SQUARE)
    ok = [0, 1, 2, 3, 5, 6]
    assert torch.isnan(loss[4]) and torch.isfinite(loss[ok]).all()
    assert torch.isnan(gu[4]).all() and torch.isnan(gv[4]).all()
    assert torch.isfinite(gu[ok]).all() and torch.isfinite(gv[ok]).all()
    _assert_rows_close(loss[ok].cpu(), O.sot_per_frame(x[ok], y[ok], pos, pos, p=2, square=True),
                       O.sot_per_frame(x[ok].double(), y[ok].double(), pos.double(), pos.double(), p=2, square=True))
    # frame counts that are not a multiple of the resident slice (more frames than CTAs)
    xs, ys = _spectra(700, 8449, 8449, seed=6)
    p8 = torch.linspace(0, 1, 8449)
    many = capi.forward(xs.to(DEV), ys.to(DEV), p8.to(DEV), p8.to(DEV), 2.0, capi.SOT_SQUARE)
    _assert_rows_close(many.cpu(), O.sot_per_frame(xs, ys, p8, p8, p=2, square=True),
                       O.sot_per_frame(xs.double(), ys.double(), p8.double(), p8.double(), p=2, square=True))
    # an empty batch
    empty = capi.forward(xs[:0].to(DEV), ys[:0].to(DEV), p8.to(DEV), p8.to(DEV), 2.0, capi.SOT_SQUARE)
    assert empty.shape == (0,)
    assert L.sot_frames(xs[:0].to(DEV), ys[:0].to(DEV), p8.to(DEV), p8.to(DEV), p=2, square=True).shape == (0,)


# ------------------------------------------------------------------------------------------
# 3. properties at 16 385 bins x 512 frames
# ------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def batch():
    from sot_b200 import synthetic as S
    x, y = S.sot_batch(32, 32768, seed=3)  # 512 frames x 16385 bins
    return x.reshape(-1, 16385).to(DEV), y.reshape(-1, 16385).to(DEV), S.linear_positions(32768).to(DEV)


def test_properties_of_long_rows(capi, batch):
    x, y, pos = batch
    sq = capi.SOT_SQUARE
    loss, gu, gv = capi.forward_backward(x, x.clone(), pos, pos, 2.0, sq)
    assert (loss == 0).all(), "identical spectra"
    a = capi.forward(x, y, pos, pos, 2.0, sq)
    b = capi.forward(y, x, pos, pos, 2.0, sq)
    assert torch.equal(a, b), "symmetry without the cutoff"
    # scaling by powers of two is exact, except where it moves a mass across the safe_divide floor (near-silent
    # frames of the synthetic batch): compare the frames whose masses stay above it
    live = ((x * 0.125).square().sum(1) > 1e-6) & ((y * 0.125).square().sum(1) > 1e-6)
    assert live.sum() >= 256
    scaled = capi.forward(x * 4.0, y * 0.125, pos, pos, 2.0, sq)
    assert torch.equal(scaled[live], a[live]), "power-of-two scaling"
    fused = capi.forward_backward(x, y, pos, pos, 2.0, sq)
    assert torch.equal(fused[0], a), "forward-only and fused loss"
    again = capi.forward_backward(x, y, pos, pos, 2.0, sq)
    for s, t in zip(fused, again):
        assert torch.equal(s, t), "two runs"
    # scale invariance of the normalised loss: <x, dL/dx> = 0 up to rounding
    dot = (x * fused[1]).sum(1).abs()[live]
    assert (dot <= 1e-4 * (x.abs() * fused[1].abs()).sum(1)[live] + 1e-12).all()


def test_backward_modes_agree_on_long_rows(L, batch):
    x, y, pos = batch
    outs = {}
    for mode in ("onepass", "recompute", "fused"):
        xd, yd = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
        v = L.Wasserstein1D(p=2, square_dist=True, backward_mode=mode)(xd, yd, x_pos=pos, y_pos=pos)
        v.backward()
        outs[mode] = (v.detach(), xd.grad, yd.grad)
    for mode in ("recompute", "fused"):
        for s, t in zip(outs["onepass"], outs[mode]):
            assert torch.equal(s, t), mode


# ------------------------------------------------------------------------------------------
# 4. the training step
# ------------------------------------------------------------------------------------------
def test_training_step_without_host_sync_in_a_graph_and_from_host_buffers(capi, L, batch):
    x, y, pos = batch
    x, y = x[:64].contiguous(), y[:64].contiguous()
    mod = L.Wasserstein1D(p=2, square_dist=True, dont_normalize=True, limit_quantile_range=True)
    xd = x.clone().requires_grad_(True)
    mod(xd, y, x_pos=pos, y_pos=pos).backward()  # (first call: the positions tensor is checked once, then cached)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        xd2 = x.clone().requires_grad_(True)
        value = mod(xd2, y, x_pos=pos, y_pos=pos)
        value.backward()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert torch.equal(xd2.grad, xd.grad)
    # a CUDA graph of the step, replayed
    static_x = x.clone().requires_grad_(True)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            static_x.grad = None
            mod(static_x, y, x_pos=pos, y_pos=pos).backward()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    static_x.grad = None
    with torch.cuda.graph(graph):
        static_loss = mod(static_x, y, x_pos=pos, y_pos=pos)
        static_loss.backward()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(static_loss, value.detach()) and torch.equal(static_x.grad, xd.grad)
    # the host-buffer entry point equals the device path bit for bit
    xh, yh, ph = x.cpu().pin_memory(), y.cpu().pin_memory(), pos.cpu()
    up = torch.rand(64)
    hl, hu, hv = capi.loss_grad_host(xh, yh, ph, ph, 2.0, capi.SOT_SQUARE, upstream=up.pin_memory())
    dl, du, dv = capi.forward_backward(x, y, pos, pos, 2.0, capi.SOT_SQUARE, upstream=up.to(DEV))
    assert torch.equal(hl, dl.cpu()) and torch.equal(hu, du.cpu()) and torch.equal(hv, dv.cpu())


# ------------------------------------------------------------------------------------------
# 5. complex rows past the complex limit, 6. refusals
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_fft", [16384, 32768])
def test_complex_rows_past_the_complex_limit(L, n_fft):
    from sot_b200 import features as FE
    gen = torch.Generator().manual_seed(n_fft)
    audio = torch.randn(2, n_fft * 2, generator=gen).to(DEV)
    target = torch.randn(2, n_fft * 2, generator=gen).to(DEV)
    zx = FE.complex_frames(audio, size=n_fft)
    zy = FE.complex_frames(target, size=n_fft)
    F = zx.shape[-1]
    pos = torch.linspace(0, 1, F, device=DEV)
    mod = L.Wasserstein1D(p=2, square_dist=True)
    a = zx.clone().requires_grad_(True)
    v_c = mod(a, zy, x_pos=pos, y_pos=pos)
    v_c.backward()
    v_m = mod(zx.abs(), zy.abs(), x_pos=pos, y_pos=pos)
    assert torch.equal(v_c, v_m)
    assert torch.isfinite(torch.view_as_real(a.grad)).all()
    tr = FE.Wasserstein1DWithTransform(p=2, square_dist=True, transform_kwargs=dict(
        type="stft", log=False, n_fft=n_fft, hop_length=n_fft // 4, sr=48000))
    sig = audio.clone().requires_grad_(True)
    out = tr(sig, target)
    out.backward()
    ref = tr.wasserstein(tr.transform(audio), tr.transform(target), x_pos=tr._positions(DEV), y_pos=tr._positions(DEV))
    assert torch.equal(out.detach(), ref)
    assert torch.isfinite(sig.grad).all()


def test_refusals_on_long_rows(capi, L):
    n = 9000
    x, y = _spectra(2, n, n, seed=9)
    pos = torch.linspace(0, 1, n, device=DEV)
    x, y = x.to(DEV), y.to(DEV)
    with pytest.raises(ValueError):
        L.Wasserstein1D(p=2)(x, y, x_pos=pos, y_pos=pos, return_quantiles=True)
    with pytest.raises(ValueError):
        L.Wasserstein1D(p=2)(x, y, x_pos=pos.clone().requires_grad_(True), y_pos=pos)
    with pytest.raises(ValueError):
        capi.loss_from_cdf(x, y, pos, pos, 2.0, 0)
    assert capi.max_bins() == 2 ** 24 - 1
    big = torch.zeros(1, 2 ** 24, device=DEV)
    bpos = torch.zeros(2 ** 24, device=DEV)
    with pytest.raises(ValueError):
        capi.forward(big, big, bpos, bpos, 2.0, 0)
