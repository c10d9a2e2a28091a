"""The C-ABI library builds, loads, and exports exactly what include/sot_b200.h declares.
No compute calls here (no GPU needed)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    text = open(os.path.join(ROOT, "include", "sot_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(sot_[a-z_0-9]+)\s*\(", text)))


def test_header_and_binding_agree():
    from sot_b200 import _capi
    assert sorted(_capi.SIGNATURES) == _declared()


def test_library_loads_and_exports_every_symbol():
    from sot_b200 import _capi
    lib = _capi.load()
    assert os.path.samefile(_capi.library_path(), os.path.join(ROOT, "1d-spectral-optimal-transport_b200", "_lib",
                                                               "libsot_b200.so"))
    for name in _declared():
        assert hasattr(lib, name), name
    assert lib.sot_abi_version() == _capi.ABI_VERSION
    assert _capi.launch_count() == 0 or _capi.launch_count() > 0
    # paper shapes fit, with and without gradients, shared and per-frame supports
    assert _capi.max_bins(True, True) >= 4097 and _capi.max_bins(True, False) >= 2049


def test_argument_validation_happens_before_any_launch():
    from sot_b200 import _capi
    lib = _capi.load()
    before = _capi.launch_count()
    prob = _capi.SotProblem(4, 9, 9, 0, 0, 0, 0, 0, 0, 2.0, 0)
    assert lib.sot_forward_device(ctypes.byref(prob), None, None) == -1  # NULL pointers
    assert b"NULL" in lib.sot_last_error()
    prob = _capi.SotProblem(4, 9, 9, 16, 16, 16, 16, 0, 0, 0.5, 0)
    assert lib.sot_forward_device(ctypes.byref(prob), ctypes.c_void_p(16), None) == -3  # p < 1
    assert b"only valid for p>=1" in lib.sot_last_error()
    prob = _capi.SotProblem(4, 9, 9, 16, 16, 16, 16, 0, 0, 2.0, 64)
    assert lib.sot_forward_device(ctypes.byref(prob), ctypes.c_void_p(16), None) == -1  # unknown flag
    prob = _capi.SotProblem(4, 60000, 60000, 16, 16, 16, 16, 0, 0, 2.0, 0)
    assert lib.sot_forward_device(ctypes.byref(prob), ctypes.c_void_p(16), None) == -2  # does not fit
    # the host-buffer entry is sized for real rows: complex (STFT) rows are refused before anything is allocated
    prob = _capi.SotProblem(4, 9, 9, 16, 16, 16, 16, 0, 0, 2.0, _capi.SOT_COMPLEX_INPUT)
    assert lib.sot_loss_grad_host(ctypes.byref(prob), None, ctypes.c_void_p(16), None, None, 0) == -1
    assert b"SOT_COMPLEX_INPUT" in lib.sot_last_error()
    # the one-launch step: plan and workspace are required, peers must be described completely
    plan = _capi.SotMeanPlan()
    prob = _capi.SotProblem(4, 9, 9, 16, 16, 16, 16, 0, 0, 2.0, 0)
    assert lib.sot_mean_step_device(ctypes.byref(prob), ctypes.byref(plan), None, None, None, None) == -1
    plan.workspace, plan.post_world = 16, 3
    assert lib.sot_mean_step_device(ctypes.byref(prob), ctypes.byref(plan), None, None, None, None) == -1
    assert lib.sot_scale_inplace_device(ctypes.c_void_p(16), 4, None, 0, None, None) == -1
    assert lib.sot_set_tuning(48, 7, 0) == -1
    assert lib.sot_set_tuning(0, 0, 0) == 0
    assert _capi.launch_count() == before


def _cuobjdump(option):
    import shutil
    import subprocess
    from torch.utils.cpp_extension import CUDA_HOME
    from sot_b200 import _capi
    # the CUDA toolkit's own copy when its bin/ is not on PATH
    tool = shutil.which("cuobjdump") or os.path.join(CUDA_HOME or "", "bin", "cuobjdump")
    if not os.path.isfile(tool):
        pytest.skip("cuobjdump not available")
    return subprocess.run([tool, option, _capi.library_path()], capture_output=True, text=True).stdout


def test_sass_contains_tma_bulk_copies():
    """The hot kernels move rows with cp.async.bulk (SASS UBLKCP), not with per-thread loads."""
    sass = _cuobjdump("-sass")
    assert "UBLKCP" in sass and "SYNCS" in sass


def test_library_has_every_kernel_of_each_configuration_and_no_other():
    """sot_frame_kernel instantiations per (threads per frame, bins per thread, row floats, chains, frames per CTA):
    27 for a full configuration (10 real-spectra, 8 complex-input, 4 CDF-input, 3 raw-weight and 2 plan kernels),
    10 for the sub-warp one (real spectra, loss and gradients)."""
    names = re.findall(r"Function (_ZN3sot16sot_frame_kernelI\S+):", _cuobjdump("-res-usage"))
    counts = {}
    for name in names:
        args = tuple(int(a) for a in re.findall(r"L[ib](\d+)E", name))
        assert len(args) == 10, name
        key = args[:4] + args[9:]
        counts[key] = counts.get(key, 0) + 1
    full = [(32, 9, 296, 1), (64, 9, 584, 2), (32, 33, 1064, 1), (64, 17, 1096, 1), (128, 9, 1160, 1),
            (128, 17, 2184, 2), (256, 17, 4360, 2), (256, 33, 8456, 1)]
    assert counts == {**{c + (1,): 27 for c in full}, (16, 17, 280, 1, 2): 10}


def _build_c_demo(tmp_path):
    import shutil
    import subprocess
    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    from sot_b200 import _capi
    _capi.load()
    lib_dir = os.path.dirname(_capi.library_path())
    exe = os.path.join(str(tmp_path), "sot_c_demo")
    cmd = ["gcc", "-std=c99", "-O2", "-Wall", "-Werror", os.path.join(ROOT, "examples", "c_abi_demo.c"),
           "-I" + os.path.join(ROOT, "include"), "-L" + lib_dir, "-lsot_b200", "-Wl,-rpath," + lib_dir, "-lm", "-o", exe]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    return exe


def test_plain_c_caller_compiles_and_links_against_the_header(tmp_path):
    """The boundary is usable from C: examples/c_abi_demo.c builds with -Wall -Werror against include/sot_b200.h."""
    assert os.path.exists(_build_c_demo(tmp_path))


@pytest.mark.gpu
def test_plain_c_caller_gives_the_python_layers_numbers(tmp_path):
    import json
    import subprocess
    import numpy as np
    import torch
    from sot_b200 import losses
    out = subprocess.run([_build_c_demo(tmp_path)], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    line = json.loads(out.stdout.strip().splitlines()[-1])
    n_frames, n_bins = 64, 1025
    pos = np.arange(n_bins, dtype=np.float32) / np.float32(n_bins - 1)
    f = np.arange(n_frames, dtype=np.float64)[:, None]
    cx = 0.30 + 0.004 * f
    x = np.exp(-0.25 * (pos.astype(np.float64)[None] - cx) ** 2 / 0.02 ** 2).astype(np.float32)
    y = (0.7 * np.exp(-0.25 * (pos.astype(np.float64)[None] - cx - 0.05) ** 2 / 0.02 ** 2)).astype(np.float32)
    xt = torch.from_numpy(x).cuda().requires_grad_(True)
    yt = torch.from_numpy(y).cuda().requires_grad_(True)
    rows = losses.sot_frames(xt, yt, torch.from_numpy(pos).cuda(), torch.from_numpy(pos).cuda(), p=2, square=True)
    rows.sum().backward()
    assert line["frames"] == n_frames and line["launches"] >= 1
    assert abs(line["mean_loss"] - rows.mean().item()) <= 2e-6 * rows.mean().item()  # (libm exp vs numpy exp inputs)
    assert abs(line["mean_loss"] - 0.0025) <= 1e-4  # two unit-mass Gaussians 0.05 apart: W_2^2 = 0.05^2
    want = (xt.grad.abs().sum() + yt.grad.abs().sum()).item()
    assert abs(line["grad_abs_sum"] - want) <= 1e-4 * want
