"""Wasserstein barycenters against the float32 torch oracle on the same GPU, timed with CUDA events after warm-up.

    python tools/bench_barycenter.py [--reps 5] [--rounds 3] [--out FILE]

Two workloads on paper-like spectra (synthetic.sot_batch, n_fft 2048: 1025 bins, linear grid, square_dist), output
grid = input grid:
  interpolation  N = 65 536 barycenters of K = 2 rows (OT-mixup / morphing of a large batch)
  templates      N = 64 barycenters of K = 1024 rows (class prototypes, k-means centroids)
The interpolation inputs are 537 MB, larger than the 126 MB L2.  The kernel path and the eager oracle alternate in the
same run.  Reported per measurement: seconds, slots per second (N * K * n / s) and, for the interpolation workload,
the share of 7.7 TB/s of HBM bandwidth on its algorithmic bytes (read 4 N K n and write 4 N M forward; the backward adds
the upstream read 4 N M and the gradient write 4 N K n).  Prints one JSON line per measurement, with the card's name
and power limit read in the same run; `--out` also appends them to a file.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_BYTES_PER_S = 7.7e12  # HGX B200 data sheet, one GPU


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
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from oracle import barycenter_oracle as BO
    from sot_b200 import barycenter, synthetic as S

    name, power = card()
    dev = "cuda"
    n = 1025
    g = S.linear_positions(2048).to(dev)
    lines = []

    def emit(rec):
        rec.update(card=name, power_limit=power)
        lines.append(json.dumps(rec))
        print(lines[-1], flush=True)

    def rows(count):
        x, y = S.sot_batch(-(-count // 32), 2048, seed=42, device=dev)
        return torch.cat((x, y), 1).reshape(-1, n)[:count].contiguous()

    for work, N, K in (("interpolation", 65536, 2), ("templates", 64, 1024)):
        x = rows(N * K).reshape(N, K, n)
        w = torch.rand(N, K, device=dev) + 0.1
        w = w / w.sum(1, keepdim=True)
        G = torch.rand(N, n, device=dev)

        def kern_fwd():
            barycenter.wasserstein_barycenter(x, w, g, square_dist=True)

        def kern_fwd_bwd():
            xs = x.detach().requires_grad_(True)
            torch.autograd.grad((G * barycenter.wasserstein_barycenter(xs, w, g, square_dist=True)).sum(), xs)

        def eager_fwd():
            BO.barycenter(x, w, g, square=True)

        def eager_fwd_bwd():
            xs = x.detach().requires_grad_(True)
            torch.autograd.grad((G * BO.barycenter(xs, w, g, square=True)).sum(), xs)

        with torch.no_grad():  # the same values: the largest CDF difference against the float64 oracle, both paths
            sub = slice(0, 64)
            r64 = BO.barycenter(x[sub].double(), w[sub].double(), g.double(), square=True).cumsum(1)
            mine = barycenter.wasserstein_barycenter(x[sub], w[sub], g, square_dist=True).double().cumsum(1)
            r32 = BO.barycenter(x[sub], w[sub], g, square=True).double().cumsum(1)
            emit(dict(check="max_cdf_diff_vs_fp64_oracle", workload=work, kernel=(mine - r64).abs().max().item(),
                      eager_fp32=(r32 - r64).abs().max().item()))
        runs = dict(kernel_fwd=kern_fwd, eager_fwd=eager_fwd, kernel_fwd_bwd=kern_fwd_bwd, eager_fwd_bwd=eager_fwd_bwd)
        for fn in runs.values():  # warm-up of every shape the timed window uses
            fn()
        slots = N * K * n
        for rnd in range(args.rounds):
            for label, fn in runs.items():
                # (one eager templates call runs 1024 searchsorted passes over 64 M levels: seconds)
                t = timed(fn, args.reps if work == "interpolation" or label.startswith("kernel") else 1)
                rec = dict(bench=label, workload=work, round=rnd, N=N, K=K, bins=n, seconds=t, slots_per_s=slots / t)
                if work == "interpolation":
                    fwd_bytes = 4 * N * K * n + 4 * N * n
                    total = fwd_bytes + (4 * N * n + 4 * N * K * n if label.endswith("bwd") else 0)
                    rec["hbm_share"] = total / t / HBM_BYTES_PER_S
                emit(rec)
        del x, G
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
