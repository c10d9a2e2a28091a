"""Grouped barycenters and one Wasserstein k-means iteration, timed with CUDA events after warm-up.

    python tools/bench_kmeans.py [--reps 3] [--rounds 3] [--out profiles/r06_kmeans.jsonl]

Paper-like spectra (synthetic.sot_batch, n_fft 2048: 1025 bins, linear grid), as mass rows (square_dist on the
magnitudes, normalised once, as `cluster.wasserstein_kmeans` feeds them), R = 65 536 rows:
  update_c256   the k-means update step: C = 256 clusters with Zipf sizes (size of rank r proportional to 1 / r; the
                largest has 10 700 rows).  `grouped` is one `wasserstein_barycenter_groups` call; `padded` is the dense
                `wasserstein_barycenter` on the clusters padded to the largest one with zero-weight rows (the only way
                before); `eager_tail` / `grouped_tail` are the float32 torch oracle looped over the clusters of at most
                256 rows against the grouped call on the same rows (the oracle is quadratic in a cluster's rows: the
                large clusters take minutes there).
  update_c4     C = 4 Zipf clusters: the largest has 31 400 rows, 32 M entries, past the dense path's 2^24 per
                barycenter (the dense call refuses it), so `grouped` runs alone.
  lloyd_c256    one full Lloyd iteration at C = 256: the assignment (`wasserstein_cdist` in row blocks + argmin) and the
                update (`wasserstein_barycenter_groups`).
The paths alternate within each round.  Prints one JSON line per measurement, with the card's name and power limit
read in the same run; `--out` also appends them to a file.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_barycenter import card, timed  # noqa: E402


def zipf_labels(R, C, gen):
    import torch
    share = 1.0 / torch.arange(1, C + 1, dtype=torch.float64)
    sizes = torch.floor(share / share.sum() * R).long()
    sizes[0] += R - sizes.sum()
    lab = torch.repeat_interleave(torch.arange(C), sizes)
    return lab[torch.randperm(R, generator=gen)], sizes


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from tests.groups_oracle import barycenter_groups as oracle_groups
    from sot_b200 import barycenter, cluster, synthetic as S

    name, power = card()
    dev = "cuda"
    n, R = 1025, 65536
    pos = S.linear_positions(2048).to(dev)
    x, y = S.sot_batch(R // 32, 2048, seed=42, device=dev)
    w = (torch.cat((x, y), 1).reshape(-1, n)[:R] ** 2)
    rows = (w / w.sum(1, keepdim=True)).contiguous()
    del x, y, w
    gen = torch.Generator().manual_seed(0)
    lines = []

    def emit(rec):
        rec.update(card=name, power_limit=power, R=R, bins=n)
        lines.append(json.dumps(rec))
        print(lines[-1], flush=True)

    def padded(lab, sizes):
        """(C, Kmax, n) rows and (C, Kmax) weights: each cluster's rows in increasing row order, then zero rows."""
        C, K = sizes.shape[0], int(sizes.max())
        xp = torch.zeros(C, K, n, device=dev)
        wp = torch.zeros(C, K, device=dev)
        order = torch.argsort(lab, stable=True)
        slot = torch.arange(R, device=dev) - torch.repeat_interleave(torch.cumsum(sizes, 0) - sizes, sizes).to(dev)
        sl = lab[order]
        xp[sl, slot] = rows[order]
        wp[sl, slot] = (1.0 / sizes.double()).float().to(dev)[sl]
        return xp, wp

    up256 = None
    for work, C in (("update_c256", 256), ("update_c4", 4)):
        lab_cpu, sizes = zipf_labels(R, C, gen)
        lab = lab_cpu.to(dev)
        up = torch.rand(C, n, device=dev)
        runs = {}

        def grouped():
            barycenter.wasserstein_barycenter_groups(rows, lab, C, pos)

        def grouped_bwd():
            xs = rows.detach().requires_grad_(True)
            torch.autograd.grad((up * barycenter.wasserstein_barycenter_groups(xs, lab, C, pos)).sum(), xs)

        runs.update(grouped_fwd=grouped, grouped_fwd_bwd=grouped_bwd)
        if int(sizes.max()) * n <= 1 << 24:
            xp, wp = padded(lab, sizes)
            ref = barycenter.wasserstein_barycenter(xp, wp, pos)
            got = barycenter.wasserstein_barycenter_groups(rows, lab, C, pos)
            emit(dict(check="grouped_equals_padded", workload=work, max_abs_diff=(got - ref).abs().max().item(),
                      bitwise=bool(torch.equal(got, ref))))

            def padded_fwd():
                barycenter.wasserstein_barycenter(xp, wp, pos)

            def padded_bwd():
                xs = xp.detach().requires_grad_(True)
                torch.autograd.grad((up * barycenter.wasserstein_barycenter(xs, wp, pos)).sum(), xs)

            runs.update(padded_fwd=padded_fwd, padded_fwd_bwd=padded_bwd)
            tail = (sizes <= 256).nonzero()[:, 0]
            keep = torch.isin(lab, tail.to(dev))
            t_rows, t_lab = rows[keep].contiguous(), lab[keep].contiguous()

            def eager_tail():
                oracle_groups(t_rows, t_lab, C, pos)

            def grouped_tail():
                barycenter.wasserstein_barycenter_groups(t_rows, t_lab, C, pos)

            runs.update(eager_tail=eager_tail, grouped_tail=grouped_tail)
            tail_rows = int(keep.sum())
        else:
            emit(dict(check="largest_group_entries", workload=work, entries=int(sizes.max()) * n,
                      dense_cap=1 << 24))
        for fn in runs.values():  # warm-up of every shape the timed window uses
            fn()
        for rnd in range(args.rounds):
            for label, fn in runs.items():
                reps = 1 if label == "eager_tail" else args.reps
                t = timed(fn, reps)
                rec = dict(bench=label, workload=work, round=rnd, C=C, largest=int(sizes.max()), seconds=t)
                rec["rows_per_s"] = (tail_rows if label.endswith("tail") else R) / t
                emit(rec)
        if work == "update_c256":
            up256 = barycenter.wasserstein_barycenter_groups(rows, lab, C, pos)
        runs.clear()
        torch.cuda.empty_cache()

    def lloyd():
        cluster.wasserstein_kmeans(rows, 256, pos, init=up256, n_iter=1)

    lloyd()
    for rnd in range(args.rounds):
        t = timed(lloyd, args.reps)
        emit(dict(bench="lloyd_iteration", workload="lloyd_c256", round=rnd, C=256, seconds=t, rows_per_s=R / t))
    if args.out:
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
