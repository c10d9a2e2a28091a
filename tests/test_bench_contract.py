"""bench.py's CPU-side legs keep the JSON contract (no GPU needed: `--impl reference`); on the GPU, `--dump-outputs`
writes what the timed path computed."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                          "--warmup", "1", "--cpu-frames", "64", "--frames", "128", "--workload", "sot512-cut"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "frames/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("SOT loss fwd+bwd frames/s")
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"] == "sot512-cut" and d["gpu_launches"] == 0
    for key in ("n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data"):
        assert key in d


def test_non_zero_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step(tmp_path):
    """`--steps K --dump-outputs DIR`: K timed steps (two launches each on one GPU), then the loss and a fixed sample
    of both gradients of the last one, float32, under 64 MB -- the very numbers the same step gives when run here on
    the same seeded inputs (16384 frames of the default workload: one input set, no rotation)."""
    import numpy as np
    import bench
    from sot_b200 import sharding, synthetic as S
    frames, steps, n_fft = 16384, 3, 2048
    F = n_fft // 2 + 1
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1",
                          "--frames", str(frames), "--no-e2e", "--no-cpu", "--no-ref-cuda",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["config"]["workload"] == "sot2048-nocut-sweep" and d["steps"] == steps and d["gpu_launches"] == 2 * steps
    got = {p.name[:-4]: np.load(p) for p in tmp_path.iterdir()}
    assert sorted(got) == ["grad_x", "grad_y", "loss"]
    assert all(a.dtype == np.float32 for a in got.values()) and sum(a.nbytes for a in got.values()) <= 64e6
    idx = bench.sample_frames(frames, F)
    assert idx is not None and got["grad_x"].shape == got["grad_y"].shape == (idx.numel(), F)
    assert d["dumped_outputs"]["frames_written"] == idx.numel()

    x, y = S.sot_batch(-(-frames // 16), n_fft, seed=42, device="cuda")
    xg = x.reshape(-1, F)[:frames].contiguous().requires_grad_(True)
    yg = y.reshape(-1, F)[:frames].contiguous().requires_grad_(True)
    pos = S.linear_positions(n_fft).cuda()
    loss_fn = sharding.ShardedWasserstein1D(p=2, square_dist=True, dont_normalize=False, limit_quantile_range=False)
    value = loss_fn(xg, yg, x_pos=pos, y_pos=pos.clone())
    value.backward()
    assert got["loss"].shape == (1,) and got["loss"][0] == pytest.approx(value.item(), rel=1e-6)
    assert d["loss"] == pytest.approx(value.item(), rel=1e-6)
    i = idx.cuda()
    assert np.array_equal(got["grad_x"], xg.grad[i].cpu().numpy())
    assert np.array_equal(got["grad_y"], yg.grad[i].cpu().numpy())
