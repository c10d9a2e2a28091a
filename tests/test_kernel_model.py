"""The kernel's algorithm (tests/kernel_model.py) against the oracle's closed form and autograd."""
import numpy as np
import pytest
import torch

from oracle import sot_oracle as O
from sot_b200 import synthetic as S
from tests import kernel_model as KM


def _frames(n_fft, n_frames, seed):
    x, y = S.sot_batch(max(1, -(-n_frames // 16)), n_fft, seed=seed)
    F = x.shape[-1]
    return x.reshape(-1, F)[:n_frames].numpy(), y.reshape(-1, F)[:n_frames].numpy()


@pytest.mark.parametrize("n_fft,T,L", [(512, 32, 17), (512, 7, 80), (2048, 128, 17)])
@pytest.mark.parametrize("cut", [True, False])
@pytest.mark.parametrize("p", [1, 2, 3])
def test_walk_matches_closed_form_bit_exact(n_fft, T, L, cut, p):
    x, y = _frames(n_fft, 6 if n_fft == 2048 else 16, seed=123)
    pos = S.linear_positions(n_fft).numpy()
    for r in range(x.shape[0]):
        *_, cu, cv = KM.normalise(x[r], y[r], True, cut)
        loss, g_cu, g_cv = KM.walk_frame(cu, cv, pos, pos, p, cut, T, L)
        ref_loss, r_cu, r_cv, _, _ = O.closed_form_from_cdfs(cu, cv, pos, pos, p, cut)
        assert np.array_equal(g_cu, r_cu), f"frame {r}: dL/dcu"
        assert np.array_equal(g_cv, r_cv), f"frame {r}: dL/dcv"
        assert abs(loss - float(ref_loss)) <= 2e-6 * abs(float(ref_loss)) + 1e-12


def test_walk_ties_and_long_plateaus():
    # heavy exact ties: many zero weights, identical spectra, and a plateau spanning many threads
    rng = np.random.default_rng(0)
    n = 200
    pos = np.linspace(0, 1, n).astype(np.float32)
    for trial in range(30):
        wu = rng.random(n).astype(np.float32) * (rng.random(n) < 0.15)
        wv = rng.random(n).astype(np.float32) * (rng.random(n) < 0.15)
        if trial % 3 == 0:
            wv = wu.copy()
        if trial % 5 == 0:
            wu[60:] = 0
        wu[0] += 1e-3
        wv[0] += 1e-3
        cu = np.cumsum((wu / wu.sum()).astype(np.float64)).astype(np.float32)
        cv = np.cumsum((wv / wu.sum()).astype(np.float64)).astype(np.float32)
        for T, L in ((32, 13), (128, 4), (400, 1)):
            for limit in (False, True):
                loss, g_cu, g_cv = KM.walk_frame(cu, cv, pos, pos, 2, limit, T, L)
                ref_loss, r_cu, r_cv, _, _ = O.closed_form_from_cdfs(cu, cv, pos, pos, 2, limit)
                assert np.array_equal(g_cu, r_cu) and np.array_equal(g_cv, r_cv)
                assert abs(loss - float(ref_loss)) <= 2e-6 * abs(float(ref_loss)) + 1e-12


def test_unequal_supports():
    rng = np.random.default_rng(1)
    n, m = 37, 90
    pu = np.sort(rng.random(n)).astype(np.float32)
    pv = np.sort(rng.random(m)).astype(np.float32)
    cu = np.cumsum(rng.random(n) / n).astype(np.float32)
    cv = np.cumsum(rng.random(m) / m * 1.3).astype(np.float32)
    for limit in (False, True):
        loss, g_cu, g_cv = KM.walk_frame(cu, cv, pu, pv, 2, limit, 32, 4)
        ref_loss, r_cu, r_cv, _, _ = O.closed_form_from_cdfs(cu, cv, pu, pv, 2, limit)
        assert np.array_equal(g_cu, r_cu) and np.array_equal(g_cv, r_cv)
        assert abs(loss - float(ref_loss)) <= 2e-6 * abs(float(ref_loss))


@pytest.mark.parametrize("cut", [True, False])
def test_end_to_end_model_vs_stable_autograd(cut):
    """From magnitudes.  The model's fp64-accumulated masses/CDFs often land on exactly the
    reference's fp32 CDFs; on those frames the loss agrees to rounding and the gradient is at
    least as close to the fp64 continuation of the same CDFs as the reference's own fp32
    autograd is (the gradient is ill-conditioned in fp32: SURVEY.md App. B)."""
    x, y = _frames(512, 32, seed=456)
    pos = S.linear_positions(512)
    tx, ty = torch.from_numpy(x), torch.from_numpy(y)
    rows, gx, gy = O.sot_loss_and_grads(tx, ty, pos, pos, upstream=torch.ones(x.shape[0]), p=2,
                                        square=True, cut_scale=cut, limit=cut, stable=True)
    _, _, _, cu_ref, cv_ref, _, _ = O.sot_quantiles(tx, ty, pos, pos, square=True, cut_scale=cut,
                                                    stable=True)
    same_cdf = 0
    for r in range(x.shape[0]):
        loss, mgx, mgy, cu, cv, _, _ = KM.frame_loss_and_grads(x[r], y[r], pos.numpy(), pos.numpy(),
                                                              2, True, cut, cut, 32, 17)
        if not (np.array_equal(cu, cu_ref[r].numpy()) and np.array_equal(cv, cv_ref[r].numpy())):
            continue
        same_cdf += 1
        Ma, Mb = KM.normalise(x[r], y[r], True, cut)[2:4]
        tl, tgx, tgy = O.fp64_chain_from_cdfs(x[r], y[r], cu, cv, pos.numpy(), pos.numpy(), Ma, Mb,
                                              2, True, cut, cut)
        assert abs(loss - rows[r].item()) <= 2e-6 * abs(rows[r].item())
        assert abs(loss - tl) <= 2e-6 * abs(tl)
        for mine, ref32, truth in ((mgx, gx[r].numpy(), tgx), (mgy, gy[r].numpy(), tgy)):
            e_mine = np.linalg.norm(mine - truth) / np.linalg.norm(truth)
            e_ref = np.linalg.norm(ref32 - truth) / np.linalg.norm(truth)
            assert e_mine <= max(2e-6, 1.5 * e_ref), (r, e_mine, e_ref)
    assert same_cdf >= x.shape[0] // 4, f"only {same_cdf} frames reproduced the reference CDFs"


@pytest.mark.parametrize("threads,per_thread,n", [(64, 17, 1025), (32, 9, 257), (128, 17, 2049), (32, 33, 1025)])
def test_cdf_stage_model_is_monotone_and_tracks_fp64(threads, per_thread, n):
    """The design argument of the packed-fp32 CDF stage, checked on the CPU model for adversarial rows: the row is
    non-decreasing across thread boundaries (the cap by the next thread's head), ends at fl32(total / mass), and
    stays within ~(longest local run)/2 ulp of the float64 CDF."""
    rng = np.random.default_rng(threads * 1000 + n)
    rows = [np.exp(6.0 * rng.standard_normal(n) - 8.0), rng.random(n), np.full(n, 0.37),
            np.where(rng.random(n) < 0.02, 1.0, 1e-7 * rng.random(n)),   # isolated peaks over a noise floor
            np.concatenate((np.full(n - 1, 1e-12), [1.0])), np.concatenate(([1.0], np.full(n - 1, 1e-9)))]
    for x in rows:
        x = x.astype(np.float32)
        c = KM.cdf_stage_model(x, threads, per_thread)
        assert np.all(np.diff(c) >= 0), "CDF must be non-decreasing"
        w = x.astype(np.float64) ** 2
        mass = max(float(np.float32(w.sum())), 1e-7)  # utils.py:135-142: a mass <= eps is replaced by eps
        c64 = np.cumsum(w) / mass
        ulp = np.spacing(c64.astype(np.float32))
        longest = max(np.diff(KM.cdf_segments(per_thread)))  # fp32 adds behind a local prefix
        assert np.max(np.abs(c.astype(np.float64) - c64) / ulp) <= longest / 2 + 2 + len(KM.cdf_segments(per_thread)) / 2
        assert abs(float(c[-1]) - c64[-1]) <= 1.2e-7 * c64[-1]


def test_cutoff_mask_on_the_fma_pipe_is_exactly_zero_or_one():
    """The walk replaces `q > 1 ? 0 : x` by x * keep(q), keep(q) = sat(fma(q, -2^60, thr+ * 2^60)) with thr+ the
    float after 1 (csrc/sot_kernels.cuh, `keep_c`).  Model of that FFMA.SAT (the product and the sum are exact in
    float64 for float32 operands this close to 1, one rounding to float32, clamp to [0, 1]): keep is exactly 1 for
    every float32 q <= 1 and exactly 0 for every q > 1, including the neighbours of 1, zero, denormals, huge values
    and +inf; without a limit the constant is +inf and keep is 1 for every finite q."""
    f32 = np.float32
    thr_plus = np.nextafter(f32(1.0), f32(2.0))
    keep_c = np.float64(thr_plus) * 2.0 ** 60

    def keep(q, c):
        with np.errstate(invalid="ignore", over="ignore"):
            v = f32(np.float64(q) * -(2.0 ** 60) + c)
        return f32(0.0) if np.isnan(v) else f32(min(max(v, f32(0.0)), f32(1.0)))

    below = [f32(0.0), f32(1e-45), f32(1e-30), f32(0.5), np.nextafter(f32(1.0), f32(0.0)), f32(1.0)]
    above = [thr_plus, np.nextafter(thr_plus, f32(2.0)), f32(1.5), f32(1e20), f32(3.4e38), f32(np.inf)]
    rng = np.random.default_rng(0)
    below += list(rng.random(2000).astype(np.float32))
    above += list((1.0 + rng.random(2000) * 1e-3).astype(np.float32) + f32(2e-7))
    assert all(keep(q, keep_c) == 1.0 for q in below)
    assert all(keep(q, keep_c) == 0.0 for q in above if q > 1.0)
    finite = [f32(0.0), f32(1.0), f32(7.0), f32(3.4e38)]
    assert all(keep(q, np.float64(np.inf)) == 1.0 for q in finite) and keep(f32(np.inf), np.float64(np.inf)) == 0.0


@pytest.mark.parametrize("name", ["sot2048_cut", "sot2048_nocut", "sot2048_logf_unsorted"])
def test_cdf_stage_model_on_the_reference_fixtures_one_warp_per_frame(name):
    """The production configuration for 1025 bins is one warp per frame, 33 bins per thread.  33 sequential fp32
    adds leave the CDF up to 5 ulp from the float64 CDF on these fixtures; with the local prefix sums restarted in
    four segments the model -- which the GPU test `test_kernel_cdfs_within_ulps_of_fp64` shows the kernel
    follows -- stays within 3 (the reference's own float32 CDFs: within 3)."""
    from tests import golden_io as G
    g = G.load(name)
    kw = G.oracle_kwargs(g["meta"]["ctor"])
    F = g["x"].shape[-1]
    x, y = g["x"].reshape(-1, F), g["y"].reshape(-1, F)
    wx, wy = O.spectra_to_weights(x.double(), y.double(), kw["square"], kw["cut_scale"])
    c64u, c64v = torch.cumsum(wx, 1).float().numpy(), torch.cumsum(wy, 1).float().numpy()

    def ulps(a, b):
        return int(np.abs(a.view(np.int32).astype(np.int64) - b.view(np.int32).astype(np.int64)).max())

    for r in range(x.shape[0]):
        cu, inv, _ = KM.cdf_stage_model(x[r].numpy(), 32, 33, square=kw["square"], return_inv=True)
        cv = KM.cdf_stage_model(y[r].numpy(), 32, 33, square=kw["square"], inv64=inv if kw["cut_scale"] else None)
        assert np.all(np.diff(cu) >= 0) and np.all(np.diff(cv) >= 0)
        assert ulps(cu, c64u[r]) <= 3 and ulps(cv, c64v[r]) <= 3, (r, ulps(cu, c64u[r]), ulps(cv, c64v[r]))
