#!/usr/bin/env python
"""bench.py -- SOT loss forward+backward throughput (frames/s) on 1..8 B200, with roofline, end-to-end (host
buffers through the C ABI), reference-on-the-same-GPU and CPU-baseline legs.  Prints ONE JSON line (rank 0).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--scaling weak|strong] [--graph]
                    [--dump-outputs DIR]
    python bench.py --impl reference ...          (the reference's own CPU implementation, same metric/config)
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

A "step" = one `loss = Wasserstein1D(...)(x, y, x_pos, y_pos); loss.backward()` over this rank's shard of the
workload with BOTH spectra requiring gradients (24*F+8 algorithmic bytes per frame, SURVEY.md section 8d; the one
fused launch that now makes the step moves 16*F of them).  Weak scaling (default): every rank owns `--frames`
frames (65,536 x 1025 bins, BASELINE.json config "SOT-NoCut large sweep"); strong scaling: `--frames` frames in
total, split over the ranks.  Inputs + gradients of one rank are ~1 GiB at the default size, far larger than the
126 MB L2; smaller shards rotate through enough input sets to exceed twice the L2 (`config.l2`).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "SOT loss fwd+bwd frames/s (n_fft=2048)"
WORKLOADS = {
    # name: (n_fft, cut, grid)
    "sot2048-nocut-sweep": (2048, False, "linear"),  # BASELINE.json configs[3] (the multi-GPU sweep)
    "sot2048-cut": (2048, True, "linear"),           # paper config SOT-2048
    "sot512-cut": (512, True, "linear"),             # configs[1]
    "sot512-logf-cut": (512, True, "logf"),          # configs[2]
}
L2_BYTES = 126e6
DUMP_BYTES = 48 << 20  # both sampled gradients of --dump-outputs (+ 4 bytes of loss), within a 64 MB budget


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="sot2048-nocut-sweep", choices=sorted(WORKLOADS))
    ap.add_argument("--frames", type=int, default=65536, help="frames per GPU (weak) or in total (strong)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--mode", default=None, choices=["onepass", "recompute"], help="backward mode (default: onepass)")
    ap.add_argument("--graph", action="store_true", help="replay the step from a CUDA graph (launch-bound shards)")
    ap.add_argument("--tuning", default=None, help="threads_per_frame,bins_per_thread[,chains] kernel override")
    ap.add_argument("--collective", default="auto", choices=["auto", "nccl", "p2p"],
                    help="the one exchange of the sharded mean: NCCL all-reduce or NVLink peer-memory mailboxes")
    ap.add_argument("--no-overlap", action="store_true", help="collect the exchange on the main stream")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-ref-cuda", action="store_true")
    ap.add_argument("--no-check", action="store_true", help="skip the rank-0 recomputation of the sharded value")
    ap.add_argument("--cpu-frames", type=int, default=4096, help="frames per call of the CPU reference")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (loss.npy, grad_x.npy, grad_y.npy, "
                         "float32; rank 0's shard) to DIR, the gradients cut to a fixed sample of frames if larger "
                         f"than {DUMP_BYTES >> 20} MiB: the inputs are seeded, so two builds can be compared file by file")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    return args


def sample_frames(frames, bins):
    """Frames whose gradients `--dump-outputs` writes: all of them when both gradients fit DUMP_BYTES, else a sorted
    sample drawn from a fixed seed, so that the same arguments select the same frames in every run."""
    keep = DUMP_BYTES // (2 * 4 * bins)
    if frames <= keep:
        return None
    return torch.randperm(frames, generator=torch.Generator().manual_seed(0))[:keep].sort().values


def dump_outputs(out_dir, value, grad_x, grad_y):
    """Writes the loss and the two gradients one step returned as float32 .npy files; returns what was written."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    frames, bins = grad_x.shape
    idx = sample_frames(frames, bins)
    if idx is not None:
        idx = idx.to(grad_x.device)
        grad_x, grad_y = grad_x[idx], grad_y[idx]
    for name, t in (("loss", value.detach().reshape(1)), ("grad_x", grad_x), ("grad_y", grad_y)):
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())
    return {"dir": out_dir, "frames_written": frames if idx is None else int(idx.numel()), "frames": frames,
            "sample": None if idx is None else "sorted randperm(frames), torch generator seed 0"}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and throttle reasons WHILE the timed region runs: one `nvidia-smi -lms 50` child process streams a
    line every 50 ms, a thread only reads the pipe (it sleeps in the read; NVML calls from this process -- from a
    polling thread or from the timing loop itself -- were measured to stall the launch path by 10 %).  The summary
    uses the samples that fell between `begin()` and `end()`; when the region was shorter than the sampling period
    it uses the samples of the whole loaded phase (warm-up, timed steps, kernel-alone loops) and says so."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")

    def __init__(self, index):
        self.index, self.samples, self.proc, self.thread = index, [], None, None
        self.t_begin, self.t_end = None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "50"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.strip().split(",")]
            if len(parts) >= 6:
                try:
                    self.samples.append((time.perf_counter(), float(parts[0]), float(parts[1]),
                                         tuple(p.lower().startswith("active") for p in parts[2:6])))
                except ValueError:
                    pass

    def begin(self):
        self.t_begin = time.perf_counter()

    def end(self):
        self.t_end = time.perf_counter()

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        if self.thread is not None:
            self.thread.join(timeout=5)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        inside = [s for s in self.samples if self.t_begin is not None and self.t_begin <= s[0] <= (self.t_end or 1e30)]
        used = inside if inside else self.samples
        sm = sorted(s[1] for s in used)
        reasons = [n for k, n in enumerate(self.NAMES) if any(s[3][k] for s in used)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": used[0][2], "reasons": reasons, "samples": len(used),
                "samples_inside_timed_region": len(inside),
                "window": "timed region" if inside else "loaded phase around the timed region (region < 50 ms)"}


def positions(n_fft, grid):
    from sot_b200 import synthetic as S
    return S.linear_positions(n_fft) if grid == "linear" else S.logf_positions(n_fft)


def cpu_reference_leg(n_fft, cut, grid, total_frames, chunk_frames, steps, warmup, seconds_cap=None, budget_s=None):
    """The reference's CPU implementation timed on this box's host cores, forward + backward, both gradients: the
    UNMODIFIED `losses.Wasserstein1D` when its files are present (`/root/reference`, or the verbatim git-ignored
    copy under baseline/_ref/ that travels to the GPU box: kind "reference"), else the oracle port, which is pinned
    bit-for-bit to it (kind "port").  One step = `total_frames` frames processed in calls of `chunk_frames`."""
    from oracle import reference_loader as RL
    from sot_b200 import synthetic as S
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    signals = max(1, chunk_frames // 16)
    x, y = S.sot_batch(signals, n_fft, seed=42)
    pos = positions(n_fft, grid)
    if RL.available():
        ref = RL.load()
        loss_fn = ref.Wasserstein1D(p=2, square_dist=True, dont_normalize=cut, limit_quantile_range=cut)
        kind, what = "reference", f"unmodified losses.Wasserstein1D from {RL.root()}"

        def call(xr, yr):
            return loss_fn(xr, yr, x_pos=pos, y_pos=pos.clone())
    else:
        from oracle import sot_oracle as O
        kind, what = "port", "oracle/sot_oracle.py (pinned bit-for-bit to the reference in the build container)"

        def call(xr, yr):
            return O.sot_loss(xr, yr, pos, pos.clone(), p=2, square=True, cut_scale=cut, limit=cut)

    per_call = x.shape[0] * x.shape[1]
    calls = max(1, -(-total_frames // per_call))
    if budget_s is not None:
        # bounded sample: as many calls per step as fit `budget_s` seconds for the whole run (one probe call sets the rate)
        xr, yr = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
        call(xr, yr).backward()
        t0 = time.perf_counter()
        xr, yr = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
        call(xr, yr).backward()
        per_call_s = time.perf_counter() - t0
        calls = max(1, min(calls, int(budget_s / (per_call_s * (steps + warmup)))))

    def step():
        for _ in range(calls):
            xr = x.clone().requires_grad_(True)
            yr = y.clone().requires_grad_(True)
            call(xr, yr).backward()

    for _ in range(warmup):
        step()
    times = []
    t_start = time.perf_counter()
    for _ in range(steps):
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
        if seconds_cap is not None and time.perf_counter() - t_start > seconds_cap:
            break
    n = per_call * calls
    total = sum(times)
    return {"value": n * len(times) / total, "unit": "frames/s", "cores": torch.get_num_threads(), "kind": kind,
            "frames_per_step": n,
            "sample": f"{len(times)} steps x {n} frames x {x.shape[-1]} bins in calls of {per_call} frames ({what}; "
                      f"torch CPU ops, fwd+bwd, both grads), median {sorted(times)[len(times) // 2] * 1e3:.1f} ms/step"
            }, total / len(times)


def ref_on_cuda_leg(x, y, pos, cut, steps=5, warmup=2, max_frames=16384):
    """The reference's chain of eager ATen ops (losses.py:172-184, 286-313; ~30 launches forward, as many backward) on
    THIS GPU, same inputs -- what a user of the reference on a B200 has today.  The stock `losses.Wasserstein1D`
    when its files travelled (baseline/_ref/), else the oracle's torch ops, which are the same calls."""
    from oracle import reference_loader as RL
    n = min(x.shape[0], max_frames)  # the chain materialises ~30 temporaries of N x 2F (int64 among them)
    xs, ys = x[:n], y[:n]
    if RL.available():
        loss_fn = RL.load().Wasserstein1D(p=2, square_dist=True, dont_normalize=cut, limit_quantile_range=cut)
        kind = "reference"

        def call(xr, yr):
            return loss_fn(xr, yr, x_pos=pos, y_pos=pos.clone())
    else:
        from oracle import sot_oracle as O
        kind = "port"

        def call(xr, yr):
            return O.sot_loss(xr, yr, pos, pos.clone(), p=2, square=True, cut_scale=cut, limit=cut)

    def step():
        xr = xs.clone().requires_grad_(True)
        yr = ys.clone().requires_grad_(True)
        v = call(xr, yr)
        v.backward()
        return v

    for _ in range(warmup):
        v = step()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        v = step()
    b.record()
    b.synchronize()
    ms = a.elapsed_time(b) / steps
    return {"value": n / (ms * 1e-3), "unit": "frames/s", "ms_per_step": ms, "frames": n, "kind": kind,
            "loss": float(v.item()),
            "what": "reference eager torch ops on the same B200 (fwd+bwd, both grads, CUDA events)"}


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    n_fft, cut, grid = WORKLOADS[args.workload]
    F = n_fft // 2 + 1
    frames = args.frames if args.scaling == "weak" else max(16, args.frames // world)  # this rank's shard
    set_bytes = 16 * F * frames  # u, v, grad_u, grad_v of one input set
    n_sets = 1 if set_bytes >= 2 * L2_BYTES else min(32, int(-(-2 * L2_BYTES // set_bytes)))
    config = {"workload": args.workload, "frames_per_gpu": frames, "frames_total": frames * world, "bins": F, "p": 2,
              "square_dist": True, "cutoff": cut, "positions": grid, "grads": "both spectra",
              "l2": ("inputs+grads per GPU ~%.0f MB >> 126 MB L2, no flush needed" % (set_bytes / 1e6)) if n_sets == 1
              else ("%d input sets of %.1f MB rotated (working set %.0f MB > 2 x 126 MB L2)"
                    % (n_sets, set_bytes / 1e6, n_sets * set_bytes / 1e6)),
              "parallelism": f"frames sharded over {world} rank(s), one exchange of (sum, count)",
              "step": "cuda-graph replay" if args.graph else "eager (public API call)"}

    if args.impl == "reference":
        if rank != 0:
            return
        cb, ms = cpu_reference_leg(n_fft, cut, grid, frames * world, args.cpu_frames, args.steps, max(args.warmup, 1),
                                   budget_s=150.0)
        sample = {"frames_per_step": cb["frames_per_step"], "frames_per_call": args.cpu_frames,
                  "what": ("the whole workload every step" if cb["frames_per_step"] >= frames * world else
                           "a bounded sample of the workload every step (the run is sized to ~150 s)")}
        print(json.dumps({"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "frames/s",
                          "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms * 1e3,
                          "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32",
                          "data": "synthetic", "config": config, "reference_sample": sample, "cpu_baseline": cb,
                          "gpu_launches": 0,
                          "e2e": {"value": cb["value"], "unit": "frames/s", "h2d_bytes_per_step": 0,
                                  "d2h_bytes_per_step": 0}}))
        return

    import torch.distributed as dist
    from sot_b200 import _capi, sharding, synthetic as S

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the SOT kernels have no CPU path)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if args.tuning:
        _capi.set_tuning(*[int(t) for t in args.tuning.split(",")])

    # ---- inputs: synthetic harmonic spectra, resident in HBM ----------------------------------
    def make_set(seed):
        signals = -(-frames // 16)
        x, y = S.sot_batch(signals, n_fft, seed=seed, device=dev)
        return x.reshape(-1, F)[:frames].contiguous(), y.reshape(-1, F)[:frames].contiguous()

    def seed_of(r, k):
        return 42 + r + 1000 * k

    sets = [make_set(seed_of(rank, k)) for k in range(n_sets)]
    x, y = sets[0]
    pos = positions(n_fft, grid).to(dev)
    pos_y = pos.clone()
    kw = dict(p=2, square_dist=True, dont_normalize=cut, limit_quantile_range=cut)
    if args.mode:
        kw["backward_mode"] = args.mode
    overlap = world > 1 and not args.no_overlap and not args.graph
    if args.graph and world > 1 and args.collective != "p2p":
        # the captured step carries the peer-memory exchange (its call numbers live on the device, so the graph can
        # be replayed); an NCCL all-reduce inside the captured step is not supported here
        args.collective = "p2p"
    loss_fn = sharding.ShardedWasserstein1D(collective=args.collective, overlap_exchange=overlap, **kw)
    leaves = [(a.clone().requires_grad_(True), b.clone().requires_grad_(True)) for a, b in sets]

    host_s = [0.0, 0.0, 0]  # host seconds spent issuing the forward calls / the backward calls, number of steps

    def eager_step(k):
        xg, yg = leaves[k % n_sets]
        xg.grad = None
        yg.grad = None
        t0 = time.perf_counter()
        value = loss_fn(xg, yg, x_pos=pos, y_pos=pos_y)
        t1 = time.perf_counter()
        value.backward()
        host_s[0] += t1 - t0
        host_s[1] += time.perf_counter() - t1
        host_s[2] += 1
        return value

    graphs = None
    if args.graph:
        # the whole step (SOT launch, exchange, in-place scale) captured once per input set; replay = 1 host call
        for k in range(n_sets):
            for _ in range(3):
                eager_step(k)
        torch.cuda.synchronize()
        graphs = []
        for k in range(n_sets):
            g = torch.cuda.CUDAGraph()
            xg, yg = leaves[k]
            xg.grad = None
            yg.grad = None
            with torch.cuda.graph(g):
                v = loss_fn(xg, yg, x_pos=pos, y_pos=pos_y)
                v.backward()
            graphs.append((g, v))

    def step(k):
        if graphs is None:
            return eager_step(k)
        g, v = graphs[k % n_sets]
        g.replay()
        return v

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    sampler.start()
    for k in range(max(args.warmup, 3)):
        value = step(k)
    barrier()
    launches0 = _capi.launch_count()
    host_s[:] = [0.0, 0.0, 0]
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.cudart().cudaProfilerStart()  # `ncu --profile-from-start off` sees exactly the timed steps
    if world > 1:
        # the ranks leave the host barrier above milliseconds apart; an in-stream all-reduce lines the GPUs up again
        # right before the first timed step (each rank's stream waits for every peer), so that the max over ranks
        # measures the steps and not the start skew
        dist.all_reduce(torch.zeros(1, device=dev))
    ev0.record()
    sampler.begin()
    for k in range(args.steps):
        value = step(k)
    loss_fn.wait_value(value)  # (overlapped exchange: the last value is part of the timed region)
    ev1.record()
    barrier()
    sampler.end()
    torch.cuda.cudart().cudaProfilerStop()
    launches = _capi.launch_count() - launches0
    last_set = (args.steps - 1) % n_sets
    dumped = None
    if args.dump_outputs and rank == 0:
        # now, before the legs below reuse the leaves (the graph leg clears their gradients)
        xg, yg = leaves[last_set]
        dumped = dump_outputs(args.dump_outputs, value, xg.grad, yg.grad)
    host_issue = None if host_s[2] == 0 else {"forward_us": 1e6 * host_s[0] / host_s[2],
                                              "backward_us": 1e6 * host_s[1] / host_s[2],
                                              "note": "host time to ISSUE one step (no synchronisation)"}
    if graphs is not None:
        launches = 2 * args.steps  # replayed from the graph: the SOT launch + the in-place scale per step
    ms_total = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
    ms_by_rank = [ms_total.item() / args.steps]
    if world > 1:
        every = [torch.zeros_like(ms_total) for _ in range(world)]
        dist.all_gather(every, ms_total)
        ms_by_rank = [t.item() / args.steps for t in every]
        dist.all_reduce(ms_total, op=dist.ReduceOp.MAX)
    ms_step = ms_total.item() / args.steps
    frames_s = frames * world / (ms_step * 1e-3)
    value_last = float(value.item())
    exchange = loss_fn.exchange
    collective = {"used": getattr(exchange, "collective_used", None) if world > 1 else "none (one rank)",
                  "requested": args.collective, "fallback_reason": getattr(exchange, "fallback_reason", None),
                  "overlapped_with_next_step": bool(overlap)}

    # ---- the sharded value, recomputed on ONE GPU by rank 0 (every shard regenerated from its seed) -----------
    value_check = None
    if world > 1 and not args.no_check:
        if rank == 0:
            from sot_b200 import losses as Lm
            single = Lm.Wasserstein1D(**kw)
            acc = 0.0
            for r in range(world):
                xs, ys = make_set(seed_of(r, last_set))
                with torch.no_grad():
                    acc += float(single(xs, ys, x_pos=pos, y_pos=pos_y).item())
                del xs, ys
            want = acc / world  # equal shards
            rel = abs(value_last - want) / max(abs(want), 1e-30)
            value_check = {"distributed": value_last, "recomputed_on_rank0": want, "rel_err": rel, "ok": rel <= 2e-6,
                           "how": "rank 0 regenerates every rank's shard from its seed, one GPU, no exchange"}
            assert value_check["ok"], value_check
        barrier()

    # ---- dominant kernel alone (the fused forward+backward launch the step makes), CUDA events on its stream ----
    flags = _capi.SOT_SQUARE | (_capi.SOT_CUT_SCALE | _capi.SOT_LIMIT if cut else 0)
    if grid == "linear":  # what the module detects for these grids (exact i * 2**-k positions)
        flags |= _capi.SOT_UNIFORM_GRID
    inv = 1.0 / (frames * world)

    def timed(fn, reps):
        """Average duration of `reps` back-to-back launches, CUDA events on the launching stream (one pair around
        the whole train: an event pair per launch would add the launch latency of a ~0.4 ms kernel to each)."""
        for it in range(3):
            fn(*sets[it % n_sets])
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        for it in range(reps):
            fn(*sets[it % n_sets])
        b.record()
        b.synchronize()
        return a.elapsed_time(b) / reps

    k_avg = timed(lambda xs, ys: _capi.mean_step(xs, ys, pos, pos_y, 2.0, flags, grad_scale=inv, mean_scale=1.0 / frames),
                  args.steps)
    f_avg = timed(lambda xs, ys: _capi.mean_step(xs, ys, pos, pos_y, 2.0, flags, grad_scale=inv, mean_scale=1.0 / frames,
                                                 want_gu=False, want_gv=False), args.steps)
    sampler.stop()
    peak, peak_src = peaks()
    bytes_fused = (16 * F + 4) * frames  # reads u, v; writes grad_u, grad_v (+ the frame's share of the sum)
    bytes_fwd = (8 * F + 4) * frames     # reads u, v
    bytes_step = (24 * F + 8) * frames   # SURVEY.md 8(d): what forward + backward as two passes would move
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            traffic = json.load(f).get(args.workload, {}).get("fused_kernel_dram_bytes_per_launch")
    roofline = {"bound": "hbm", "kernel": "sot_frame_kernel<OUT_GRAD> (the one fused forward+backward launch of a step)",
                "achieved": bytes_fused / (k_avg * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                "frac": bytes_fused / (k_avg * 1e-3) / 1e9 / peak, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": bytes_fused, "kernel_ms": k_avg,
                "note": "frac counts the bytes this launch really has to move (16F+4 per frame); `step` uses SURVEY 8(d)'s "
                        "24F+8 per frame for a forward+backward step, which the single launch completes",
                "forward_only_kernel": {"ms": f_avg, "achieved": bytes_fwd / (f_avg * 1e-3) / 1e9,
                                        "frac": bytes_fwd / (f_avg * 1e-3) / 1e9 / peak,
                                        "algorithmic_bytes_per_launch": bytes_fwd},
                "step": {"algorithmic_bytes_per_frame": 24 * F + 8, "ms": ms_step,
                         "achieved": bytes_step / (ms_step * 1e-3) / 1e9,
                         "frac": bytes_step / (ms_step * 1e-3) / 1e9 / peak,
                         "frac_on_moved_bytes": bytes_fused / (ms_step * 1e-3) / 1e9 / peak}}

    # ---- the same step replayed from a CUDA graph / eagerly (whichever the timed region did not use), 1 GPU ----
    other = None
    if world == 1 and graphs is None and frames <= 16384:
        try:
            g = torch.cuda.CUDAGraph()
            xg, yg = leaves[0]
            xg.grad = None
            yg.grad = None
            with torch.cuda.graph(g):
                v = loss_fn(xg, yg, x_pos=pos, y_pos=pos_y)
                v.backward()
            for _ in range(5):
                g.replay()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = max(args.steps, 50)
            a.record()
            for _ in range(reps):
                g.replay()
            b.record()
            b.synchronize()
            other = {"cuda_graph_ms_per_step": a.elapsed_time(b) / reps, "eager_ms_per_step": ms_step,
                     "note": "graph replay re-reads one input set (L2-resident for small shards)"}
        except Exception as exc:  # pragma: no cover
            other = {"error": f"{type(exc).__name__}: {exc}"[:200]}

    # ---- the reference's eager op chain on this GPU ------------------------------------------------------------
    ref_cuda = None
    if rank == 0 and not args.no_ref_cuda:
        try:
            ref_cuda = ref_on_cuda_leg(x, y, pos, cut)
        except Exception as exc:  # pragma: no cover
            ref_cuda = {"error": f"{type(exc).__name__}: {exc}"[:200]}
        torch.cuda.empty_cache()
    if world > 1:
        barrier()

    # ---- end to end through the C ABI with HOST buffers ----------------------------------------
    e2e = None
    if not args.no_e2e:
        bind = _bind_host_side(local)
        up = torch.full((frames,), inv, device=dev)
        hx, hy = x.cpu().pin_memory(), y.cpu().pin_memory()
        hpos = pos.cpu()
        hup = up.cpu().pin_memory()
        out = {"loss": torch.empty(frames).pin_memory(), "grad_u": torch.empty_like(hx).pin_memory(),
               "grad_v": torch.empty_like(hy).pin_memory()}
        for _ in range(2):
            _capi.loss_grad_host(hx, hy, hpos, hpos, 2.0, flags, upstream=hup, device=local, out=out)
        barrier()
        n_e2e = max(3, min(args.steps, 10))
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            _capi.loss_grad_host(hx, hy, hpos, hpos, 2.0, flags, upstream=hup, device=local, out=out)
        t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        # the host path must give the device path's numbers
        check = _capi.forward_backward(x, y, pos, pos_y, 2.0, flags, upstream=up)
        torch.cuda.synchronize()
        assert torch.equal(check[0].cpu(), out["loss"]) and torch.equal(check[1].cpu(), out["grad_u"])
        e2e = {"value": frames * world * n_e2e / t.item(), "unit": "frames/s",
               "h2d_bytes_per_step": 4 * frames * (2 * F + 1) + 8 * F,
               "d2h_bytes_per_step": 4 * frames * (2 * F + 1), "steps": n_e2e,
               "api": "sot_loss_grad_host (C ABI, pinned host buffers, " +
                      ("zero-copy: one launch reads and writes host memory over PCIe)"
                       if os.environ.get("SOT_HOST_ZEROCOPY", "")[:1] == "1" else "chunked 3-stream pipeline)"),
               "host_binding": bind}

    cb = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cb, _ = cpu_reference_leg(n_fft, cut, grid, min(frames, 16384), args.cpu_frames, 30, 1, seconds_cap=20.0)

    if rank == 0:
        line = {"metric": METRIC, "value": frames_s, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "ms_per_step_by_rank": ms_by_rank,
                "higher_is_better": True,
                "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "clocks": sampler.summary(), "gpu_launches": launches, "roofline": roofline, "e2e": e2e,
                "cpu_baseline": cb, "ref_on_cuda": ref_cuda, "collective": collective,
                "collective_used": collective["used"], "value_check": value_check, "step_modes": other,
                "host_issue": host_issue,
                "loss": value_last, "backward_mode": loss_fn.backward_mode}
        if dumped is not None:
            line["dumped_outputs"] = dumped
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def _bind_host_side(local_rank: int):
    """The host-buffer pipeline streams ~1 GB per step each way through pinned memory: keep this rank's thread and
    the pages it is about to pin on the NUMA node of its GPU (the launcher leaves every rank on all cores)."""
    try:
        from sot_b200 import hostbind
        return hostbind.bind_to_gpu_node(local_rank)
    except Exception as exc:  # pragma: no cover
        return {"bound": False, "why": f"{type(exc).__name__}: {exc}"[:120]}


if __name__ == "__main__":
    main()
