"""Exact radius search over spectra (`pairwise.wasserstein_radius`) against blocked `wasserstein_cdist` + `nonzero`, and
`cluster.wasserstein_dbscan`, timed with CUDA events after warm-up, the two search paths alternated in each round.

    python tools/bench_radius.py [--queries 4096] [--db 262144] [--rounds 3] [--out FILE]

Paper-like spectra (synthetic.sot_batch, n_fft 2048: 1025 bins, linear grid, p = 2, square_dist).  Workloads:
  retrieval   the target frames of seed 1 against the targets and predictions of seed 2 (the set of bench_knn.py), at
              the radii where the median query has 1, 10 and 100 rows within (the median k-th value of
              wasserstein_knn); the full contract (indices exactly, values bitwise, against the blocked matrix) is
              checked once
  worst case  cut mode (`dont_normalize`), where no pair can be skipped: the search's overhead over cdist + nonzero
  dbscan      wasserstein_dbscan on 65 536 rows at the eps where the median row has 30 neighbours, min_samples 10:
              the time, the clusters found and the noise fraction
Prints one JSON line per measurement with the card's name and power limit read in the same run, the time, the pairs
per second (P * R / time), the pairs found and the fraction of the pairs walked; `--out` also appends them to a file.
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


def timed(fn):
    import torch
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    out = fn()
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end) / 1e3, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--queries", type=int, default=4096)
    ap.add_argument("--db", type=int, default=262144)
    ap.add_argument("--worst-db", type=int, default=65536)
    ap.add_argument("--dbscan-rows", type=int, default=65536)
    ap.add_argument("--block", type=int, default=1024, help="query rows per cdist block of the baseline")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from sot_b200 import _capi, cluster, pairwise, synthetic as S

    name, power = card()
    dev = "cuda"
    g = S.linear_positions(2048).to(dev)
    lines = []

    def emit(rec):
        rec.update(card=name, power_limit=power)
        lines.append(json.dumps(rec))
        print(lines[-1], flush=True)

    x, _ = S.sot_batch(-(-args.queries // 16), 2048, seed=1, device=dev)
    x = x.reshape(-1, 1025)[:args.queries].contiguous()
    yt, yp = S.sot_batch(-(-args.db // 32), 2048, seed=2, device=dev)
    y = torch.cat([yt.reshape(-1, 1025), yp.reshape(-1, 1025)])[:args.db].contiguous()
    del yt, yp
    P = x.shape[0]

    def radius(a, b, r, cut=False):
        return lambda: pairwise.wasserstein_radius(a, b, r, g, g, p=2, square_dist=True, dont_normalize=cut)

    def cdist_nonzero(a, b, r, cut=False):
        def run():
            idx, vals = [], []
            for q0 in range(0, a.shape[0], args.block):
                D = pairwise.wasserstein_cdist(a[q0:q0 + args.block], b, g, g, p=2, square_dist=True,
                                               dont_normalize=cut)
                mask = D <= torch.tensor(r, dtype=torch.float32)
                hit = mask.nonzero()
                hit[:, 0] += q0
                idx.append(hit)
                vals.append(D[mask])
            return pairwise.RadiusResult(torch.cat(vals), torch.cat(idx))
        return run

    def walked_fraction(a, b, r, flags):
        _, _, _, count, walked = _capi.pairwise_radius(a[None], b[None], g, g, 2.0, flags, r, 0, want_walked=True)
        return walked.item() / (a.shape[0] * b.shape[0]), count.item()

    def median_kth(a, b, k, cut=False):
        v = pairwise.wasserstein_knn(a, b, k, g, g, p=2, square_dist=True, dont_normalize=cut).values[:, k - 1]
        return float(v.nanmedian())

    def run(workload, paths, pairs, extra, flags, r, rounds):
        frac, count = walked_fraction(*pairs, r, flags)
        for fn in paths.values():  # warm-up
            fn()
        for rnd in range(rounds):
            for label, fn in paths.items():
                t, out = timed(fn)
                P_, R_ = pairs[0].shape[0], pairs[1].shape[0]
                rec = dict(bench=workload, path=label, round=rnd, P=P_, R=R_, radius=r, bins=1025, seconds=t,
                           pairs_per_s=P_ * R_ / t, found=int(out.values.numel()), **extra)
                if label == "radius":
                    rec["walked_fraction"] = frac
                    assert count == rec["found"]
                emit(rec)

    with torch.no_grad():
        radii = {k: median_kth(x, y, k) for k in (1, 10, 100)}
        # the contract once at this size, at the k = 10 radius: indices exactly, values bitwise
        got, want = radius(x, y, radii[10])(), cdist_nonzero(x, y, radii[10])()
        ok = torch.equal(got.indices, want.indices) and torch.equal(got.values.view(torch.int32),
                                                                    want.values.view(torch.int32))
        emit(dict(check="contract_vs_cdist_nonzero", P=P, R=y.shape[0], radius=radii[10],
                  found=int(got.values.numel()), equal=bool(ok)))
        del got, want
        for k, r in radii.items():
            run("retrieval", dict(cdist_nonzero=cdist_nonzero(x, y, r), radius=radius(x, y, r)), (x, y),
                dict(median_hits_k=k), _capi.SOT_SQUARE, r, args.rounds)

        yw = y[:args.worst_db]
        rc = median_kth(x, yw, 10, cut=True)
        run("worst_case_cut",
            dict(cdist_nonzero=cdist_nonzero(x, yw, rc, cut=True), radius=radius(x, yw, rc, cut=True)), (x, yw),
            dict(median_hits_k=10), _capi.SOT_SQUARE | _capi.SOT_CUT_SCALE, rc, args.rounds)
        del y, yw

        rows, _ = S.sot_batch(-(-args.dbscan_rows // 16), 2048, seed=3, device=dev)
        rows = rows.reshape(-1, 1025)[:args.dbscan_rows].contiguous()
        eps = median_kth(rows, rows, 30)
        frac, count = walked_fraction(rows, rows, eps, _capi.SOT_SQUARE)
        dbscan = lambda: cluster.wasserstein_dbscan(rows, eps, 10, g, p=2, square_dist=True)  # noqa: E731
        dbscan()
        for rnd in range(args.rounds):
            t, res = timed(dbscan)
            emit(dict(bench="dbscan", round=rnd, R=rows.shape[0], eps=eps, min_samples=10, bins=1025, seconds=t,
                      neighbour_pairs=count, walked_fraction=frac, n_clusters=res.n_clusters,
                      core_fraction=float(res.core.float().mean()),
                      noise_fraction=float((res.labels == -1).float().mean()),
                      largest_cluster=int(torch.bincount(res.labels[res.labels >= 0]).max())
                      if res.n_clusters else 0))
    if args.out:
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
