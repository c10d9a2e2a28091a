"""Exact k-NN of spectra (`pairwise.wasserstein_knn`) against `wasserstein_cdist` + `torch.topk` (and, for the
assignment shape, `cluster._assign`), timed with CUDA events after warm-up, the two paths alternated in each round.

    python tools/bench_knn.py [--queries 4096] [--db 262144] [--rounds 3] [--out FILE]

Paper-like spectra (synthetic.sot_batch, n_fft 2048: 1025 bins, linear grid, p = 2, square_dist).  Workloads:
  retrieval   the target frames of seed 1 against the targets and predictions of seed 2, k in {1, 10, 100}; the full
              contract (values bitwise, indices exactly, against a stable sort of the matrix) is checked once
  assignment  65 536 rows against 256 centroids, k = 1 (the shape of a k-means assignment step)
  worst case  cut mode (`dont_normalize`), where no pair can be skipped: the kNN's overhead over cdist + topk
Prints one JSON line per measurement with the card's name and power limit read in the same run, the time, the pairs
per second (P * R / time) and the fraction of the pairs the kNN walked; `--out` also appends them to a file.
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
    ap.add_argument("--rows", type=int, default=65536)
    ap.add_argument("--centroids", type=int, default=256)
    ap.add_argument("--worst-db", type=int, default=65536)
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
    P, R = x.shape[0], y.shape[0]

    def knn(a, b, k, flags):
        return lambda: _capi.pairwise_knn(a[None], b[None], g, g, 2.0, flags, k, want_walked=True)

    def cdist_topk(a, b, k, cut=False):
        return lambda: torch.topk(pairwise.wasserstein_cdist(a, b, g, g, p=2, square_dist=True, dont_normalize=cut),
                                  k, dim=-1, largest=False)

    # the contract once at this size: k = 100 against the first columns of a stable sort of the matrix
    with torch.no_grad():
        vals, idx, walked = knn(x, y, 100, _capi.SOT_SQUARE)()
        D = pairwise.wasserstein_cdist(x, y, g, g, p=2, square_dist=True)
        sv, si = torch.sort(D, dim=-1, stable=True)
        ok = torch.equal(vals[0].view(torch.int32), sv[:, :100].view(torch.int32)) and torch.equal(idx[0], si[:, :100])
        emit(dict(check="contract_vs_stable_sort", P=P, R=R, k=100, equal=bool(ok)))
        del D, sv, si

    def run(workload, paths, pairs, k, rounds):
        for fn in paths.values():  # warm-up
            fn()
        for rnd in range(rounds):
            for label, fn in paths.items():
                t, out = timed(fn)
                rec = dict(bench=workload, path=label, round=rnd, P=pairs[0], R=pairs[1], k=k, bins=1025, seconds=t,
                           pairs_per_s=pairs[0] * pairs[1] / t)
                if label == "knn":
                    rec["walked_fraction"] = out[2].item() / (pairs[0] * pairs[1])
                emit(rec)

    for k in (1, 10, 100):
        run("retrieval", dict(cdist_topk=cdist_topk(x, y, k), knn=knn(x, y, k, _capi.SOT_SQUARE)), (P, R), k,
            args.rounds)

    rows, _ = S.sot_batch(-(-args.rows // 16), 2048, seed=3, device=dev)
    rows = rows.reshape(-1, 1025)[:args.rows].contiguous()
    cents = y[:args.centroids].contiguous()
    with torch.no_grad():
        _, lab = cluster._assign(rows, cents, g)
        _, i1, _ = knn(rows, cents, 1, 0)()  # (`_assign` is W2^2 of the magnitudes: no square_dist)
        emit(dict(check="assignment_labels_equal", equal=bool(torch.equal(lab, i1[0, :, 0]))))
    run("assignment", dict(cluster_assign=lambda: cluster._assign(rows, cents, g),
                           knn=knn(rows, cents, 1, 0)), (rows.shape[0], cents.shape[0]), 1, args.rounds)

    yw = y[:args.worst_db]
    run("worst_case_cut", dict(cdist_topk=cdist_topk(x, yw, 10, cut=True),
                               knn=knn(x, yw, 10, _capi.SOT_SQUARE | _capi.SOT_CUT_SCALE)), (P, yw.shape[0]), 10,
        args.rounds)
    if args.out:
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
