"""Pairwise SOT distances against the materialised paired path, timed with CUDA events after warm-up.

    python tools/bench_pairwise.py [--P 1024] [--big 4096] [--reps 5] [--out FILE]

Paper-like spectra (synthetic.sot_batch, n_fft 2048: 1025 bins, linear grid, p = 2, square_dist, no cutoff).  At
P = R = 1024 the materialised path's rows are 2 x 4.3 GB, far larger than the 126 MB L2; the pairwise inputs are the
4 MB of rows themselves, which is the point.  The two paths alternate in the same run.  Prints one JSON line per
measurement, with the card's name and power limit read in the same run; `--out` also appends them to a file.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return torch.cuda.get_device_name(0), q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def timed(fn, reps):
    import torch
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(reps):
        fn()
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end) / 1e3 / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--P", type=int, default=1024)
    ap.add_argument("--big", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from sot_b200 import losses, pairwise, synthetic as S

    name, power = card()
    dev = "cuda"
    g = S.linear_positions(2048).to(dev)
    kw = dict(p=2, square_dist=True)
    lines = []

    def emit(rec):
        rec.update(card=name, power_limit=power)
        lines.append(json.dumps(rec))
        print(lines[-1], flush=True)

    def inputs(P):
        x, y = S.sot_batch(-(-P // 16), 2048, seed=42, device=dev)
        return x.reshape(-1, 1025)[:P].contiguous(), y.reshape(-1, 1025)[:P].contiguous()

    P = args.P
    x, y = inputs(P)
    G = torch.rand(P, P, device=dev)

    def cdist_fwd():
        pairwise.wasserstein_cdist(x, y, g, g, **kw)

    def cdist_fwd_bwd():
        xs, ys = x.detach().requires_grad_(True), y.detach().requires_grad_(True)
        torch.autograd.grad((G * pairwise.wasserstein_cdist(xs, ys, g, g, **kw)).sum(), (xs, ys))

    def mat(xs, ys):
        X = xs[:, None].expand(P, P, 1025).reshape(-1, 1025)
        Y = ys[None].expand(P, P, 1025).reshape(-1, 1025)
        return losses.sot_frames(X, Y, g, g, p=2, square=True).reshape(P, P)

    def mat_fwd():
        mat(x, y)

    def mat_fwd_bwd():
        xs, ys = x.detach().requires_grad_(True), y.detach().requires_grad_(True)
        torch.autograd.grad((G * mat(xs, ys)).sum(), (xs, ys))

    # the same values: every entry of the two paths within the loss gate
    with torch.no_grad():
        a, b = pairwise.wasserstein_cdist(x, y, g, g, **kw), mat(x, y)
        emit(dict(check="max_rel_diff_vs_materialised", P=P, value=((a - b).abs() / b.abs()).max().item()))
    runs = dict(cdist_fwd=cdist_fwd, materialised_fwd=mat_fwd, cdist_fwd_bwd=cdist_fwd_bwd,
                materialised_fwd_bwd=mat_fwd_bwd)
    for fn in runs.values():  # warm-up of every shape the timed window uses
        fn()
    for rnd in range(args.rounds):
        for label, fn in runs.items():
            t = timed(fn, args.reps)
            emit(dict(bench=label, round=rnd, P=P, R=P, bins=1025, seconds=t, pairs_per_s=P * P / t))
        del fn

    P = args.big
    x, y = inputs(P)
    G = torch.rand(P, P, device=dev)
    cdist_fwd()
    cdist_fwd_bwd()
    for rnd in range(args.rounds):
        for label, fn in (("cdist_fwd", cdist_fwd), ("cdist_fwd_bwd", cdist_fwd_bwd)):
            t = timed(fn, max(1, args.reps // 2))
            emit(dict(bench=label, round=rnd, P=P, R=P, bins=1025, seconds=t, pairs_per_s=P * P / t))
    if args.out:
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
