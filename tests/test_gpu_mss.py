"""GPU parity of the MSS loss kernels (row f3) and of `metrics.wasserstein_distance` (row f4) against the
reference fixtures (tests/golden/make_golden_mss.py) and the oracle.

Tolerances (float32): loss rel 1e-5; audio gradients rel-L2 1e-4 (the L1 term's gradient is a sign: elements whose
two magnitudes agree to the last ulps may flip between cuFFT and the CPU FFT, hence not bit-exact)."""
import pytest
import torch

from oracle import mss_oracle as M
from tests import golden_io as G

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _rel_l2(a, b):
    return (torch.linalg.vector_norm(a - b) / torch.linalg.vector_norm(b).clamp_min(1e-30)).item()


@pytest.fixture(scope="module")
def MSS():
    from sot_b200 import mss
    return mss


@pytest.mark.parametrize("name", ["mss_paper_l1", "mss_l1_mag_log", "mss_l2_mag_log"])
def test_mss_module_vs_reference_fixture(MSS, name):
    g = G.load(name)
    mod = MSS.MSSLoss(**g["meta"]["ctor"])
    x = g["audio_x"].to(DEV).requires_grad_(True)
    y = g["audio_y"].to(DEV).requires_grad_(True)
    value = mod(x, y)
    (2.0 * value).backward()
    assert value.shape == () and value.dtype == torch.float32
    assert abs(value.item() - g["value"].item()) <= 1e-5 * abs(g["value"].item())
    # Gradients: the L1 term's derivative is a SIGN and the log term's is 1/|z|, so bins at rounding-noise level
    # (window leakage ~1e-8, where cuFFT and the CPU FFT disagree in every digit) contribute O(1) each with a
    # random sign.  Against the CPU fixture only a coarse bound holds; the tight check runs the oracle's torch ops
    # on the same device, i.e. on the same cuFFT spectrograms.
    assert _rel_l2(x.grad.cpu(), 2.0 * g["grad_audio_x"]) <= 0.1
    assert _rel_l2(y.grad.cpu(), 2.0 * g["grad_audio_y"]) <= 0.1
    xo = g["audio_x"].to(DEV).requires_grad_(True)
    yo = g["audio_y"].to(DEV).requires_grad_(True)
    want = M.mss_loss(xo, yo, **g["meta"]["ctor"])
    (2.0 * want).backward()
    assert abs(value.item() - want.item()) <= 2e-6 * abs(want.item())
    assert _rel_l2(x.grad, xo.grad) <= 1e-5
    assert _rel_l2(y.grad, yo.grad) <= 1e-5


@pytest.mark.parametrize("kind", ["L1", "L2"])
@pytest.mark.parametrize("count", [1, 2, 7, 4096 * 33 + 5])
@pytest.mark.parametrize("offset", [0, 1])
def test_mss_term_vs_oracle_on_spectrograms(MSS, kind, count, offset):
    """Odd counts and 8-byte-only alignment (offset 1) take the scalar path; zeros and sub-eps bins included."""
    gen = torch.Generator().manual_seed(count)
    zt = torch.view_as_complex(torch.randn(count + offset, 2, generator=gen))
    zv = torch.view_as_complex(torch.randn(count + offset, 2, generator=gen))
    zv[::5] *= 1e-6  # below safe_log's eps
    zt[::7] = 0  # |z| = 0: no gradient through abs
    zt_d = zt.to(DEV)[offset:].requires_grad_(True)
    zv_d = zv.to(DEV)[offset:].requires_grad_(True)
    mine = MSS.mss_term(zt_d, zv_d, 0.8, 0.3, kind)
    mine.backward()
    zt_c = zt[offset:].clone().requires_grad_(True)
    zv_c = zv[offset:].clone().requires_grad_(True)
    want = M.term_from_magnitudes(zt_c.abs(), zv_c.abs(), 0.8, 0.3, kind)
    want.backward()
    assert abs(mine.item() - want.item()) <= 2e-6 * abs(want.item())
    assert _rel_l2(torch.view_as_real(zt_d.grad.cpu()), torch.view_as_real(zt_c.grad)) <= 2e-6
    assert _rel_l2(torch.view_as_real(zv_d.grad.cpu()), torch.view_as_real(zv_c.grad)) <= 2e-6


def test_mss_only_prediction_needs_grad_and_misuse(MSS):
    from sot_b200 import _capi
    gen = torch.Generator().manual_seed(3)
    zt = torch.view_as_complex(torch.randn(4, 65, 9, 2, generator=gen)).to(DEV)
    zv = torch.view_as_complex(torch.randn(4, 65, 9, 2, generator=gen)).to(DEV).requires_grad_(True)
    before = _capi.launch_count()
    MSS.mss_term(zt.transpose(1, 2), zv.transpose(1, 2), 1.0, 0.0, "L1").backward()  # dense, permuted layout
    assert _capi.launch_count() - before == 2
    assert zv.grad is not None and zv.grad.shape == zv.shape
    with pytest.raises(ValueError, match="Loss type"):
        MSS.mss_term(zt, zv, 1.0, 0.0, "cosine")
    with pytest.raises(TypeError):
        MSS.mss_term(zt.abs(), zv.abs(), 1.0, 0.0, "L1")
    with pytest.raises(_capi.SotError):
        MSS.mss_term(zt.cpu(), zv.detach().cpu(), 1.0, 0.0, "L1")
    assert MSS.MSSLoss(mag_weight=0.0, logmag_weight=0.0)(torch.zeros(1, 4096, device=DEV), torch.zeros(1, 4096, device=DEV)) == 0.0
    mixed = MSS.MixOfLosses([MSS.MSSLoss(fft_sizes=(256, 64), mag_weight=1.0)], [0.05])
    out = mixed(torch.randn(2, 4096, device=DEV), torch.randn(2, 4096, device=DEV))
    assert set(out) == {"MSSLoss"} and out["MSSLoss"].item() > 0


def test_mss_partial_means_like_the_reference(MSS):
    """`MSSLoss(...)(x, y, dims=...)` (losses.py:409-421 via `mean_difference(dims=)`): per-item values."""
    from oracle import mss_oracle as MO
    gen = torch.Generator().manual_seed(11)
    a, b = torch.randn(3, 4096, generator=gen) * 0.1, torch.randn(3, 4096, generator=gen) * 0.1
    mod = MSS.MSSLoss(fft_sizes=(512, 128), mag_weight=1.0, logmag_weight=0.5, loss_type="L2")
    bd = b.to(DEV).requires_grad_(True)
    got = mod(a.to(DEV), bd, dims=(1, 2))
    assert got.shape == (3,)
    want = 0.0
    for size in (512, 128):
        tm, vm = MO.magnitude_frames(a, size), MO.magnitude_frames(b, size)
        want = want + ((tm - vm) ** 2).mean(dim=(1, 2)) + 0.5 * ((MO.guarded_log(tm) - MO.guarded_log(vm)) ** 2).mean(dim=(1, 2))
    assert torch.allclose(got.detach().cpu(), want, rtol=2e-4, atol=1e-7)
    got.sum().backward()
    assert bd.grad is not None and torch.isfinite(bd.grad).all()
    # and the full mean of the per-item values is the fused scalar
    full = mod(a.to(DEV), b.to(DEV))
    assert abs(full.item() - got.mean().item()) <= 1e-4 * abs(full.item())


@pytest.mark.parametrize("p", [1, 2])
def test_metrics_wasserstein_distance(p):
    from sot_b200 import metrics
    g = G.load(f"metric_wd_p{p}")
    value = metrics.wasserstein_distance(g["audio_x"].to(DEV), g["audio_y"].to(DEV), p=p, n_fft=512)
    assert abs(value.item() - g["value"].item()) <= 1e-5 * abs(g["value"].item())


def _run_example(*extra):
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "examples", "train_step.py"), *extra],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    return json.loads(out.stdout.strip().splitlines()[-1])


def test_training_step_example_reduces_the_loss():
    """examples/train_step.py (SURVEY section 8 row f2): the paper's loss mix inside a plain training loop."""
    line = _run_example("--steps", "60", "--batch", "32", "--lr", "1e-3", "--model", "standin", "--loss-share")
    assert line["last_loss"] < line["first_loss"] and line["frames_per_s"] > 0
    assert 0.0 <= line["loss_share"]["share_of_step_in_the_two_losses"] <= 1.0


def test_peer_memory_all_reduce_matches_nccl():
    """tools/p2p_check.py on 2 GPUs: the NVLink mailbox all-reduce against NCCL, bit for bit, and the sharded loss
    with either collective.  Needs two GPUs on the box (skipped otherwise)."""
    import json
    import os
    import subprocess
    import sys
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29577", os.path.join(root, "tools", "p2p_check.py")],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["values_match_nccl"] is True
    # the fused sharded path bench.py runs: value vs one GPU over all shards, gradients vs single-GPU gradients, with
    # every exchange; graph replay; unequal shards caught
    assert line["sharded_loss_ok"] and line["graph_replay_ok"] and line["unequal_shards_ok"] and line["all_ok"], line
    assert line["late_rank_ok"], "a rank arriving seconds late must be waited for, not turned into a NaN"
