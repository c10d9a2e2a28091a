"""Frame sharding across the GPUs of one box: one process per GPU, each owns a contiguous slice of
the frame axis, and the only data-path collective is ONE all-reduce of two scalars (sum of the
per-frame losses, number of frames) -- NCCL over NVLink on the GPUs, gloo in the CPU tests.

The reference is single-process (`devices: 1`, train_config.yaml:155); its `torch.mean` over all
frames (losses.py:211) becomes: local sum -> all-reduce -> / global frame count.  The backward
needs no collective: each rank scales its own rows by 1 / N_global -- inside the one SOT launch of the
step, because N_global depends on the frame counts only (`MeanExchange`).
"""
from __future__ import annotations

import torch
import torch.distributed as dist

from . import _capi, losses


RUN_AHEAD = 4  # steps a rank may run ahead of the collection of its exchanges (mailbox phases = 2 * RUN_AHEAD)


def shard_bounds(n_items: int, rank: int, world: int):
    """Contiguous, balanced split of `n_items` (signals, so a signal's frames stay together)."""
    base, extra = divmod(n_items, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


class PeerReducer:
    """All-reduce (sum) of a handful of float64 scalars through NVLink / NVSwitch peer memory: every rank
    stores its values into a mailbox on each peer and spins on its own (`csrc/sot_p2p.cu`, one 32-thread
    kernel, a few microseconds) instead of an NCCL all-reduce (tens of microseconds of launch + protocol that
    sit between the forward and the backward launch of a 0.75 ms step).  The mailboxes are one symmetric
    allocation (`torch.distributed._symmetric_memory`); construction is collective over `group`."""

    def __init__(self, group=None, device=None):
        import torch.distributed._symmetric_memory as symm
        self.group = group if group is not None else dist.group.WORLD
        self.world, self.rank = dist.get_world_size(self.group), dist.get_rank(self.group)
        device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.box = symm.empty(_capi.p2p_mailbox_doubles(self.world), dtype=torch.float64, device=device)
        self.box.zero_()
        self.handle = symm.rendezvous(self.box, self.group)
        self.ptrs = [int(p) for p in self.handle.buffer_ptrs]
        self.seq = 0
        # call numbers kept on the device for the launches that post / collect themselves (`MeanExchange`):
        # [0] = posts made by the SOT launch, [1] = collections -- a CUDA graph of the step can be replayed
        self.seq_dev = torch.zeros(2, dtype=torch.int64, device=device)
        self.seq_post, self.seq_wait = self.seq_dev[0:1], self.seq_dev[1:2]
        self.ptr_array = _capi.mailbox_array(self.ptrs)  # (built once: the per-step host time matters)
        torch.cuda.synchronize(device)
        dist.barrier(self.group)  # every mailbox is zeroed before anybody writes into it

    def all_reduce(self, values: torch.Tensor) -> torch.Tensor:
        self.seq += 1
        return _capi.p2p_allreduce(values, torch.empty_like(values), self.ptr_array, self.rank, self.seq)

    def global_mean(self, local_sum: torch.Tensor, local_count: float):
        """(sum over ranks of local_sum) / (sum of local_count) and 1 / (sum of local_count), (1,) float32 each."""
        self.seq += 1
        return _capi.p2p_global_mean(local_sum, local_count, self.ptr_array, self.rank, self.seq)


class _GlobalMean(torch.autograd.Function):
    """mean over the frames of ALL ranks of per-rank rows; differentiable w.r.t. the local rows."""

    @staticmethod
    def forward(ctx, rows, group):
        total = rows.sum(dtype=torch.float64)
        count = float(rows.numel())
        ctx.shape, ctx.dtype = rows.shape, rows.dtype
        if dist.is_available() and dist.is_initialized() and _world(group) > 1:
            # (no host->device copy here: `torch.tensor(count, device=...)` would synchronise the stream)
            stats = torch.stack((total, torch.full_like(total, count)))
            if isinstance(group, PeerReducer):
                stats = group.all_reduce(stats)
            else:
                dist.all_reduce(stats, op=dist.ReduceOp.SUM, group=group)
            ctx.save_for_backward(stats[1:2])
            ctx.count = None
            return (stats[0] / stats[1]).to(rows.dtype)
        ctx.count = count
        return (total / count).to(rows.dtype)

    @staticmethod
    def backward(ctx, grad_out):
        if ctx.count is None:
            (count,) = ctx.saved_tensors
            g = (grad_out.to(torch.float64) / count).to(ctx.dtype)
        else:
            g = grad_out / ctx.count
        return g.expand(ctx.shape), None


def _world(group) -> int:
    return group.world if isinstance(group, PeerReducer) else dist.get_world_size(group)


def global_mean(rows: torch.Tensor, group=None) -> torch.Tensor:
    return _GlobalMean.apply(rows, group)


class MeanExchange:
    """How the per-rank sums of one step become the mean over ALL ranks' frames (SURVEY.md 8e) -- the host logic
    of the sharded `Wasserstein1D` around its one SOT launch:

    * 1 / N_global scales the gradients INSIDE that launch, so it must be known before it.  It depends on the frame
      counts only.  `equal_shards=True` (default): every rank holds as many frames as this one (the DDP case:
      same batch size everywhere), N_global = world * N_local, no communication; the exchange below still carries
      the counts, and if they do not add up the returned loss is NaN and the NEXT call raises.  `equal_shards=
      False`: the counts are all-reduced before the launch (one host synchronisation per step).
    * the sums meet in ONE exchange: "p2p" -- the last CTA of the SOT launch stores (sum, count) into every
      peer's mailbox over NVLink / NVSwitch (`csrc/sot_kernels.cuh: finish_mean`) and a 32-thread kernel collects
      (`sot_p2p_wait_mean_device`); "nccl" / "gloo" -- `torch.distributed.all_reduce` of two doubles.
    * `overlap=True` runs the collecting half on a side stream, so neither the backward nor the next step's launch
      ever waits for the slowest rank; the returned tensor is then valid on the current stream only after
      `sharding.wait_value(loss)` (bounded run-ahead: step s waits for the exchange of step s-4)."""

    def __init__(self, process_group=None, collective="auto", overlap=False, equal_shards=True):
        self.group, self.collective, self.overlap, self.equal_shards = process_group, collective, overlap, equal_shards
        self.collective_used, self.fallback_reason = None, None
        self._reducer, self._side, self._status, self._flag, self._events = None, None, None, None, None
        self._done = {}  # seq -> event: "the exchange of call seq has been collected on this rank"
        self._seq = 0

    # ---- set-up (collective over the group: every rank takes the same branch -- same code, same box) ----------
    def world(self) -> int:
        return dist.get_world_size(self.group) if dist.is_available() and dist.is_initialized() else 1

    def _setup(self, device):
        if self.collective_used is not None:
            return
        backend = dist.get_backend(self.group)
        if device.type != "cuda" or backend != "nccl":
            self.collective_used = backend  # gloo on CPU tensors: the CPU tests of this logic
            self._status = torch.zeros(1, dtype=torch.int32)
            return
        if self.collective in ("auto", "p2p"):
            try:
                self._reducer = PeerReducer(self.group, device)
                self.collective_used = "p2p"
            except Exception as exc:  # symmetric memory cannot be set up on this box / build
                if self.collective == "p2p":
                    raise
                self.fallback_reason = f"{type(exc).__name__}: {exc}"[:200]
                import warnings
                warnings.warn(f"sot_b200: peer-memory exchange unavailable ({self.fallback_reason}); using NCCL")
        if self.collective_used is None:
            self.collective_used = "nccl"
        if self.overlap:
            self._side = torch.cuda.Stream(device)
        self._status = torch.zeros(1, dtype=torch.int32).pin_memory()  # written by the device, read by the host
        self._events = [torch.cuda.Event() for _ in range(4 * RUN_AHEAD)]  # rotated: "launch s queued" / "exchange s collected"

    def _check_status(self):
        if self._status is None:
            return
        if self._flag is None:
            import ctypes
            self._flag = ctypes.c_int32.from_address(self._status.data_ptr())  # (a plain host read, no tensor op)
        if self._flag.value != 0:
            code = int(self._flag.value)
            raise RuntimeError(
                "sot_b200: the ranks of the previous step did not hold the same number of frames, so its gradients "
                "were scaled with the wrong 1/N_global (construct with equal_shards=False)" if code == 1 else
                "sot_b200: a peer never arrived at the exchange of the sharded loss")

    # ---- the three steps around the launch ---------------------------------------------------------------------
    def global_count(self, n_local: int, device) -> float:
        self._setup(device)
        self._check_status()
        if self.equal_shards:
            return float(n_local) * self.world()
        t = torch.tensor([float(n_local)], dtype=torch.float64).to(device)
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)
        return float(t.item())

    def launch_kwargs(self, n_local: int, device) -> dict:
        self._seq += 1
        if device.type == "cuda" and self.overlap and (self._seq - RUN_AHEAD) in self._done:
            # bounded run-ahead; also what makes the eight-phase mailboxes safe: a rank that posts call s has
            # collected call s-4, so every peer has posted s-4 and therefore collected s-8 -- the slot s overwrites
            torch.cuda.current_stream(device).wait_event(self._done.pop(self._seq - RUN_AHEAD))
        if self.collective_used == "p2p":
            return dict(post=(self._reducer.ptr_array, self._reducer.rank, self._reducer.seq_post),
                        count_value=float(n_local))
        return dict(total_out=torch.empty(2, dtype=torch.float64, device=device), count_value=float(n_local))

    def finish(self, kw: dict, n_global: float, device) -> torch.Tensor:
        cuda = device.type == "cuda"
        side = self._side if (cuda and self.overlap) else None
        if side is not None:
            queued = self._events[(2 * self._seq) % (4 * RUN_AHEAD)]
            queued.record()  # (on the current stream: the SOT launch of this step is queued)
            side.wait_event(queued)
        if self.collective_used == "p2p":
            mean = torch.empty((), dtype=torch.float32, device=device)
            if side is not None:
                mean.record_stream(side)
            _capi.p2p_wait_mean(self._reducer.ptr_array, self._reducer.rank, self._reducer.seq_wait,
                                expected_count=n_global, status_ptr=self._status.data_ptr(), device=device,
                                stream=side, out=mean)
        else:
            with (torch.cuda.stream(side) if side is not None else _NullContext()):
                stats = kw["total_out"]
                if side is not None:
                    stats.record_stream(side)
                dist.all_reduce(stats, op=dist.ReduceOp.SUM, group=self.group)
                mean = torch.where(stats[1] == n_global, stats[0] / stats[1], float("nan")).to(torch.float32)
                # (the count check reaches the host like the peer-memory kernel's: a flag in pinned memory)
                self._status.copy_((stats[1:2] != n_global).to(torch.int32), non_blocking=True)
            if side is not None:
                mean.record_stream(torch.cuda.current_stream(device))
        if side is not None:
            done = self._events[(2 * self._seq + 1) % (4 * RUN_AHEAD)]
            done.record(side)
            self._done[self._seq] = done
            self._done.pop(self._seq - RUN_AHEAD - 1, None)
        return mean


class _NullContext:
    def __enter__(self):
        return None

    def __exit__(self, *exc):
        return False


def wait_value(loss: torch.Tensor) -> torch.Tensor:
    """Makes the current stream wait until `loss` (returned by a `ShardedWasserstein1D(overlap_exchange=True)`)
    holds the mean over all ranks; a no-op for any other tensor.  Call it before reading or logging the value."""
    ready = getattr(loss, "_sot_ready", None)
    if ready is not None:
        torch.cuda.current_stream(loss.device).wait_event(ready)
    return loss


class ShardedWasserstein1D(losses.Wasserstein1D):
    """`Wasserstein1D` whose inputs are this rank's slice of the batch and whose value is the mean
    over the whole (all-rank) batch.  Same constructor plus `process_group` (None = the default
    group).  `dims` other than None and `return_quantiles` stay local.

    Under DistributedDataParallel: DDP averages the parameter gradients over the ranks again, so a loss that is
    already the GLOBAL mean (gradients scaled by 1/N_global) ends up world_size times too small compared with a
    single-process run on the full batch.  Either multiply this loss by the world size, or use the plain
    `Wasserstein1D` (local mean) under DDP -- the standard DDP convention, and then no exchange is needed at all."""

    def __init__(self, *args, process_group=None, collective="auto", overlap_exchange=False, equal_shards=True,
                 **kwargs):
        """`collective`: "nccl" = `torch.distributed.all_reduce` on `process_group`; "p2p" = the peer-memory
        mailboxes (`PeerReducer`), written by the SOT launch itself; "auto" = p2p when it can be set up (CUDA,
        symmetric memory), else nccl with a warning -- `exchange.collective_used` / `.fallback_reason` say which.
        `overlap_exchange`, `equal_shards`: see `MeanExchange`."""
        super().__init__(*args, **kwargs)
        if collective not in ("auto", "nccl", "p2p"):
            raise ValueError('collective must be "auto", "nccl" or "p2p"')
        self.process_group = process_group
        self.collective = collective
        self.overlap_exchange = overlap_exchange
        self.equal_shards = equal_shards
        self._reducer = None  # the MeanExchange of this process (never pickled)

    @property
    def exchange(self):
        return self._reducer

    def wait_value(self, loss: torch.Tensor) -> torch.Tensor:
        """`overlap_exchange=True`: makes the current stream wait for the exchange of the latest step, after which
        `loss` holds the mean over all ranks.  A no-op otherwise."""
        ex = self._reducer
        if isinstance(ex, MeanExchange) and ex.overlap and ex._seq in ex._done:
            torch.cuda.current_stream(loss.device).wait_event(ex._done[ex._seq])
        return loss

    def __getstate__(self):  # the peer-memory mailboxes belong to this process: never pickled with the module
        state = self.__dict__.copy()
        state["_reducer"] = None
        return state

    def _mean_exchange(self):
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(self.process_group) < 2:
            return None
        if self._reducer is None:
            self._reducer = MeanExchange(self.process_group, self.collective, self.overlap_exchange,
                                         self.equal_shards)
        return self._reducer

    def _reduce_frames(self, loss, dims, as64):
        if dims is not None:  # `dims` stays local
            return super()._reduce_frames(loss, dims, as64)
        return global_mean(loss, self.process_group)  # (float32 even for float64 inputs)
