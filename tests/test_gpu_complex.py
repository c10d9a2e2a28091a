"""GPU parity of the fused STFT-magnitude prologue (flag SOT_COMPLEX_INPUT, SURVEY.md section 8 row f1):
complex64 STFT rows in, complex gradient rows out, against the reference fixtures of
`tests/golden/make_golden_stft.py` (reference route: `stft(x).abs()` -> `Wasserstein1D`, features.py:217-237,
losses.py:316-343) and against this repository's own magnitude path.

Tolerances (float32): loss rel 1e-5 without the cutoff, 2e-3 in cutoff mode (the reference's strict `qs > 1`
mask is discontinuous in the last ulp of the target CDF, see test_gpu_parity.py); gradients as rel-L2 over the
whole tensor: 1e-3 without the cutoff, 5e-3 with it.  (The gradient subtracts two nearly equal terms --
the conditioning argument of test_gpu_parity.py -- so two correct fp32 evaluations differ by ~1e-4; the tight
per-frame conditioning bound is checked there on the same kernels, here the fused |z| chain rule is the subject.)
"""
import pytest
import torch

from tests import golden_io as G

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
CASES = ["stft512_cut", "stft512_nocut", "stft512_p1_abs", "stft2048_cut", "stft2048_nocut"]


@pytest.fixture(scope="module")
def capi():
    from sot_b200 import _capi
    _capi.load()
    return _capi


@pytest.fixture(scope="module")
def L():
    from sot_b200 import losses
    return losses


@pytest.fixture(scope="module")
def FEAT():
    from sot_b200 import features
    return features


def _rel_l2(a, b):
    return (torch.linalg.vector_norm(a - b) / torch.linalg.vector_norm(b).clamp_min(1e-30)).item()


def _positions(n_bins):
    return torch.linspace(0, 1, n_bins, device=DEV)


def _tols(ctor):
    cut = bool(ctor.get("limit_quantile_range", False))
    if ctor.get("p", 1) == 1:
        # W_1 is piecewise linear in the weights: its gradient is piecewise CONSTANT and jumps whenever two CDF
        # values swap order, which a 1-ulp difference in |z| (CPU hypot / CUDA hypot / sqrt(re^2+im^2)) triggers
        # in some frames.  Measured: frames agree to 1e-7 or differ by ~1e-2; the loss itself agrees to 1e-7.
        return (1e-5, 2e-2)
    return (2e-3, 5e-3) if cut else (1e-5, 1e-3)


@pytest.mark.parametrize("name", CASES)
@pytest.mark.parametrize("mode", ["mean", "recompute", "fused"])
def test_complex_frames_vs_reference_fixture(L, name, mode):
    g = G.load(name)
    ctor = dict(g["meta"]["ctor"])
    tol_loss, tol_grad = _tols(ctor)
    zx = g["zx"].to(DEV).requires_grad_(True)
    zy = g["zy"].to(DEV).requires_grad_(True)
    n_fft = g["meta"]["transform"]["n_fft"]
    pos = torch.fft.rfftfreq(n_fft, d=1 / 16000)
    pos = (pos / pos.max()).to(DEV)
    if mode == "mean":
        mod = L.Wasserstein1D(**ctor)
        value = mod(zx, zy, x_pos=pos, y_pos=pos)
    else:
        mod = L.Wasserstein1D(**ctor, backward_mode=mode)
        value = mod(zx, zy, x_pos=pos, y_pos=pos, dims=(0, 1))  # per-frame route + torch.mean
    value.backward()
    assert zx.grad.dtype == torch.complex64 and zx.grad.shape == zx.shape
    ref = g["value"].item()
    assert abs(value.item() - ref) <= tol_loss * abs(ref)
    assert _rel_l2(torch.view_as_real(zx.grad.cpu()), torch.view_as_real(g["grad_zx"])) <= tol_grad
    assert _rel_l2(torch.view_as_real(zy.grad.cpu()), torch.view_as_real(g["grad_zy"])) <= tol_grad
    if ctor.get("p", 1) == 1:  # the frames whose merge order did not flip pin the formula tightly
        mine = torch.view_as_real(zx.grad.cpu()).flatten(0, 1).flatten(1)
        want = torch.view_as_real(g["grad_zx"]).flatten(0, 1).flatten(1)
        per_frame = torch.linalg.vector_norm(mine - want, dim=1) / torch.linalg.vector_norm(want, dim=1)
        assert (per_frame <= 1e-5).sum().item() >= 8, per_frame


@pytest.mark.parametrize("name", CASES)
def test_complex_path_agrees_with_magnitude_path(L, name):
    """Same kernels, |z| formed by torch on one side and inside the kernel on the other."""
    g = G.load(name)
    ctor = dict(g["meta"]["ctor"])
    tol_loss, tol_grad = _tols(ctor)
    pos = _positions(g["zx"].shape[-1])
    mod = L.Wasserstein1D(**ctor)
    zx = g["zx"].to(DEV).requires_grad_(True)
    zy = g["zy"].to(DEV).requires_grad_(True)
    fused = mod(zx, zy, x_pos=pos, y_pos=pos)
    fused.backward()
    wx = g["zx"].to(DEV).requires_grad_(True)
    wy = g["zy"].to(DEV).requires_grad_(True)
    plain = mod(wx.abs(), wy.abs(), x_pos=pos, y_pos=pos)
    plain.backward()
    assert abs(fused.item() - plain.item()) <= tol_loss * abs(plain.item())
    assert _rel_l2(torch.view_as_real(zx.grad), torch.view_as_real(wx.grad)) <= tol_grad
    assert _rel_l2(torch.view_as_real(zy.grad), torch.view_as_real(wy.grad)) <= tol_grad


@pytest.mark.parametrize("name", ["stft512_nocut", "stft2048_cut", "stft512_p1_abs"])
def test_wrapper_audio_in_audio_gradients_out(FEAT, name):
    g = G.load(name)
    ctor = dict(g["meta"]["ctor"])
    tol_loss, tol_grad = _tols(ctor)
    mod = FEAT.Wasserstein1DWithTransform(transform_kwargs=dict(g["meta"]["transform"]), **ctor).to(DEV)
    xa = g["audio_x"].to(DEV).requires_grad_(True)
    ya = g["audio_y"].to(DEV).requires_grad_(True)
    value = mod(xa, ya)
    value.backward()
    ref = g["value"].item()
    assert abs(value.item() - ref) <= tol_loss * abs(ref)
    assert _rel_l2(xa.grad.cpu(), g["grad_audio_x"]) <= tol_grad
    assert _rel_l2(ya.grad.cpu(), g["grad_audio_y"]) <= tol_grad


def test_stft_frames_are_handed_over_without_a_copy(FEAT):
    audio = torch.randn(4, 4096, device=DEV)
    spec = FEAT.stft(audio, frame_size=512, overlap=0.5)
    frames = FEAT.complex_frames(audio, size=512, overlap=0.5)
    assert frames.shape == (4, 16, 257) and frames.is_contiguous()
    assert spec.transpose(1, 2).is_contiguous(), "torch.stft no longer returns a transposed frame-major view"


@pytest.mark.parametrize("n_bins", [257, 1025])
@pytest.mark.parametrize("n_frames", [1, 2, 3, 5, 8])
@pytest.mark.parametrize("offset", [0, 1])
@pytest.mark.parametrize("uniform", [False, True])
def test_ragged_and_unaligned_complex_batches(capi, n_bins, n_frames, offset, uniform):
    """An odd number of complex bins makes consecutive rows alternate between 16-byte phases 0 and 8; a slice
    starting at row 1 has the opposite phase from its (freshly allocated) gradient rows, which is the path
    where the row moves inside its landing buffer; ragged tails take the non-bulk loads."""
    gen = torch.Generator().manual_seed(n_bins)
    full_x = torch.view_as_complex(torch.randn(12, n_bins, 2, generator=gen)).to(DEV)
    full_y = torch.view_as_complex(torch.randn(12, n_bins, 2, generator=gen)).to(DEV)
    pos = _positions(n_bins) if uniform else torch.sort(torch.rand(n_bins, generator=gen))[0].to(DEV)
    if uniform:
        pos = torch.arange(n_bins, device=DEV, dtype=torch.float32) / 1024.0  # exact power-of-two step
    flags = capi.SOT_SQUARE | (capi.SOT_UNIFORM_GRID if uniform else 0)
    ref_loss, ref_gu, ref_gv = capi.forward_backward(full_x, full_y, pos, pos, 2.0, flags)
    sx, sy = full_x[offset:offset + n_frames], full_y[offset:offset + n_frames]
    loss, gu, gv = capi.forward_backward(sx, sy, pos, pos, 2.0, flags)
    assert torch.equal(loss, ref_loss[offset:offset + n_frames])
    assert torch.equal(torch.view_as_real(gu), torch.view_as_real(ref_gu[offset:offset + n_frames]))
    assert torch.equal(torch.view_as_real(gv), torch.view_as_real(ref_gv[offset:offset + n_frames]))
    assert torch.equal(capi.forward(sx, sy, pos, pos, 2.0, flags), loss)
    # against the magnitude rows through the same kernels
    mag_loss, mgu, mgv = capi.forward_backward(sx.abs(), sy.abs(), pos, pos, 2.0, flags)
    assert torch.allclose(loss, mag_loss, rtol=1e-5, atol=0)
    # |z|^2 is re^2 + im^2 on one side and fl(|z|)^2 on the other: CDFs an ulp apart.  That creates or breaks an
    # exact tie between a u and a v entry in the odd frame, where the gradient (not the loss) jumps: all frames
    # within 5e-3, all but one within 1e-4.
    want = torch.view_as_real(mgu * (sx / sx.abs())).flatten(1)
    err = torch.linalg.vector_norm(torch.view_as_real(gu).flatten(1) - want, dim=1) / torch.linalg.vector_norm(want, dim=1)
    assert err.max().item() <= 5e-3 and (err <= 1e-4).sum().item() >= n_frames - 1, err


def test_every_kernel_configuration_takes_complex_rows(capi):
    gen = torch.Generator().manual_seed(5)
    for n_bins, tunings in ((257, [(32, 9, 1), (64, 9, 2), (64, 17, 1), (128, 17, 2), (256, 17, 2)]),
                            (1025, [(64, 17, 1), (128, 9, 1), (128, 17, 2), (256, 17, 2)])):
        x = torch.view_as_complex(torch.randn(9, n_bins, 2, generator=gen)).to(DEV)
        y = torch.view_as_complex(torch.randn(9, n_bins, 2, generator=gen)).to(DEV)
        pos = _positions(n_bins)
        base = capi.forward_backward(x, y, pos, pos, 2.0, capi.SOT_SQUARE | capi.SOT_CUT_SCALE | capi.SOT_LIMIT)
        try:
            for tpf, e, nch in tunings:
                capi.set_tuning(tpf, e, nch)
                got = capi.forward_backward(x, y, pos, pos, 2.0, capi.SOT_SQUARE | capi.SOT_CUT_SCALE | capi.SOT_LIMIT)
                # (configurations sum different groups of bins locally: CDFs a few ulp apart)
                assert torch.allclose(got[0], base[0], rtol=1e-5, atol=0), (tpf, e, nch)
                assert _rel_l2(torch.view_as_real(got[1]), torch.view_as_real(base[1])) <= 5e-3, (tpf, e, nch)
                assert _rel_l2(torch.view_as_real(got[2]), torch.view_as_real(base[2])) <= 5e-3, (tpf, e, nch)
        finally:
            capi.set_tuning(0, 0, 0)


def test_zero_bins_nan_frames_and_misuse(capi, L):
    n_bins = 257
    gen = torch.Generator().manual_seed(9)
    x = torch.view_as_complex(torch.randn(6, n_bins, 2, generator=gen)).to(DEV)
    y = torch.view_as_complex(torch.randn(6, n_bins, 2, generator=gen)).to(DEV)
    pos = _positions(n_bins)
    x[2, 10:40] = 0  # |z| = 0: torch.abs has gradient 0 there, not NaN
    y[4, 7] = complex(float("nan"), 0.0)
    for flags in (0, capi.SOT_SQUARE):
        loss, gu, gv = capi.forward_backward(x, y, pos, pos, 1.0 if flags == 0 else 2.0, flags)
        assert torch.isnan(loss[4]) and torch.isfinite(loss[[0, 1, 2, 3, 5]]).all()
        assert torch.isnan(torch.view_as_real(gv[4])).all() and torch.isnan(torch.view_as_real(gu[4])).all()
        keep = [0, 1, 2, 3, 5]
        assert torch.isfinite(torch.view_as_real(gu[keep])).all() and torch.isfinite(torch.view_as_real(gv[keep])).all()
        assert (torch.view_as_real(gu[2, 10:40]) == 0).all()
    # the quantile taps and the CDF harness are real-only at the ABI; the module takes |z| itself
    with pytest.raises(ValueError):
        capi.quantiles(x, y, pos, pos, capi.SOT_SQUARE)
    with pytest.raises(TypeError):
        capi.forward(x, y.abs(), pos, pos, 2.0, capi.SOT_SQUARE)
    taps = L.Wasserstein1D(p=2, square_dist=True)(x[:2, None], y[:2, None], x_pos=pos, y_pos=pos, return_quantiles=True)
    taps_mag = L.Wasserstein1D(p=2, square_dist=True)(x[:2, None].abs(), y[:2, None].abs(), x_pos=pos, y_pos=pos,
                                                      return_quantiles=True)
    assert all(torch.equal(a, b) for a, b in zip(taps, taps_mag))
    # one side already a magnitude: the other is reduced by torch, gradients still flow
    zx = x[:2].clone().requires_grad_(True)
    out = L.Wasserstein1D(p=2, square_dist=True)(zx, y[:2].abs(), x_pos=pos, y_pos=pos)
    out.backward()
    assert torch.isfinite(torch.view_as_real(zx.grad)).all()


def test_complex_rows_too_long_for_shared_memory_are_refused(capi):
    n_bins = 4400  # real rows of this length run (8448-bin configuration), complex ones do not fit
    x = torch.view_as_complex(torch.randn(2, n_bins, 2)).to(DEV)
    pos = _positions(n_bins)
    capi.forward(x.abs(), x.abs(), pos, pos, 2.0, capi.SOT_SQUARE)
    with pytest.raises(ValueError, match="do not fit"):
        capi.forward(x, x, pos, pos, 2.0, capi.SOT_SQUARE)
