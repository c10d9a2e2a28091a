"""Speed of the split-frame path (rows longer than shared memory holds): loss plus both gradients in one fused launch
(`sot_forward_backward_device`) against the reference's eager op chain (the oracle's torch ops on CUDA tensors).

    python tools/bench_long_rows.py [--frames 4096] [--bins 16385] [--steps 20] [--warmup 3] [--profile DIR]

Prints one JSON line: ms per step and frames/s of both, the split path's share of the 6461 GB/s HBM peak measured
for this project (DESIGN §5) on the 16F+4 bytes a fused step has to move, and the card's name and power limit read in
the same run.  Inputs are drawn on the device from a fixed seed; 4096 x 16385 bins are 537 MB per spectrum, more than
four times the 126 MB L2, so every step reads its rows from HBM.  `--profile DIR` adds a separate torch.profiler
run of the split path and writes its per-kernel table to DIR.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from oracle import sot_oracle as O  # noqa: E402
from sot_b200 import _capi  # noqa: E402

HBM_PEAK_GBS = 6461.0


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return name, out or "unknown"


def timed(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(steps):
        fn()
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=4096)
    ap.add_argument("--bins", type=int, default=16385)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--eager-steps", type=int, default=3)
    ap.add_argument("--profile", default=None, help="directory for the per-kernel table of a profiled run")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_long_rows.py needs a CUDA device")
    N, F = args.frames, args.bins
    gen = torch.Generator(device="cuda").manual_seed(0)
    x = torch.rand(N, F, device="cuda", generator=gen) ** 4 + 1e-4
    y = torch.rand(N, F, device="cuda", generator=gen) ** 4 + 1e-4
    pos = torch.linspace(0, 1, F, device="cuda")
    flags = _capi.SOT_SQUARE
    _capi.load()

    def split_step():
        _capi.forward_backward(x, y, pos, pos, 2.0, flags)

    ms = timed(split_step, args.steps, args.warmup)

    def eager_step():  # the reference's chain: per-frame loss, mean, autograd backward
        O.sot_loss_and_grads(x, y, pos, pos, p=2, square=True)

    ms_eager = timed(eager_step, args.eager_steps, 1)
    bytes_step = (16 * F + 4) * N
    name, power = card()
    result = {
        "workload": f"{N} frames x {F} bins, p=2, square_dist, no cutoff, loss + both gradients",
        "split_ms_per_step": round(ms, 4), "split_frames_per_s": round(N / ms * 1e3, 1),
        "split_hbm_share": round(bytes_step / (ms * 1e-3) / (HBM_PEAK_GBS * 1e9), 4),
        "eager_ms_per_step": round(ms_eager, 3), "eager_frames_per_s": round(N / ms_eager * 1e3, 1),
        "speedup_vs_eager": round(ms_eager / ms, 2),
        "gpu": name, "power_limit": power, "steps": args.steps, "warmup": args.warmup,
    }
    print(json.dumps(result))
    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        os.makedirs(args.profile, exist_ok=True)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                split_step()
            torch.cuda.synchronize()
        table = prof.key_averages().table(sort_by="cuda_time_total", row_limit=15)
        with open(os.path.join(args.profile, "long_rows_kernels.txt"), "w") as f:
            f.write(table + "\n")
        print(table)


if __name__ == "__main__":
    main()
