"""Drop-in for the reference's SOT loss: `Wasserstein1D`, `wasserstein_1d`, `quantile_function`.

Same constructor, `forward(x, y, x_pos=None, y_pos=None, **kwargs)` signature, attribute and
buffer names, error types and return shapes as `/root/reference/losses.py:89-313`, so it drops
into `trainer.py:209-221`, `metrics.py:144-149` and the YAML configs (`class_path:
losses.Wasserstein1D`).  The arithmetic is not torch ops: a `torch.autograd.Function` hands device
pointers to the sm_100a kernels behind the C ABI in `include/sot_b200.h` (one launch forward, one
backward).  PyTorch is only the host layer here (memory, streams, autograd graph).

CUDA float32 only -- there is deliberately no CPU or eager fallback; wrong-device inputs raise.
"""
from __future__ import annotations

import weakref

import torch

from . import _capi

__all__ = ["Wasserstein1D", "wasserstein_1d", "quantile_function", "sot_frames", "sot_mean", "position_term_from_plan"]

BACKWARD_MODES = ("recompute", "fused")       # per-frame values (`sot_frames`: hinge, `dims`, `wasserstein_1d`)
MEAN_BACKWARD_MODES = ("onepass", "recompute")  # the plain mean over all frames (every paper config)
DEFAULT_BACKWARD_MODE = "onepass"


# --------------------------------------------------------------------------------------
# autograd bridge
# --------------------------------------------------------------------------------------
class _SotFrames(torch.autograd.Function):
    """rows (N, n), (N, m) -> per-frame W_p^p (N,).

    backward_mode "recompute": forward launches the loss-only kernel and saves the inputs;
    backward launches the fused forward+backward kernel with the upstream gradient folded in
    (24 F + 8 bytes of HBM traffic per frame in total, nothing extra saved).
    backward_mode "fused": when a gradient is required, forward launches the fused kernel once and
    saves the unit gradients; backward is a row-scaling kernel."""

    @staticmethod
    def forward(ctx, u, v, pos_u, pos_v, p, flags, mode):
        need_u, need_v = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        ctx.p, ctx.flags, ctx.mode = p, flags, mode
        ctx.need = (need_u, need_v)
        if mode == "fused" and (need_u or need_v):
            loss, gu, gv = _capi.forward_backward(u, v, pos_u, pos_v, p, flags, None, True, need_u, need_v)
            ctx.save_for_backward(gu, gv)
        else:
            loss = _capi.forward(u, v, pos_u, pos_v, p, flags)
            ctx.save_for_backward(u, v, pos_u, pos_v)
        return loss

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_loss):
        need_u, need_v = ctx.need
        grad_loss = grad_loss.contiguous().float()
        if ctx.mode == "fused":
            gu, gv = ctx.saved_tensors
            gu = _capi.scale_rows(gu, grad_loss) if need_u else None
            gv = _capi.scale_rows(gv, grad_loss) if need_v else None
        else:
            u, v, pos_u, pos_v = ctx.saved_tensors
            _, gu, gv = _capi.forward_backward(u, v, pos_u, pos_v, ctx.p, ctx.flags, grad_loss, False, need_u, need_v)
        return gu, gv, None, None, None, None, None


# --------------------------------------------------------------------------------------
# host-side canonicalisation (the reference's reshape / expand / sort prologue)
# --------------------------------------------------------------------------------------
_sorted_cache: dict = {}  # id(user tensor) -> (weakref, version, ascending?)


def _require_cuda(t: torch.Tensor, name: str) -> None:
    if not t.is_cuda:
        raise _capi.SotError(f"sot_b200: `{name}` lives on {t.device}; the SOT kernels are CUDA only "
                             "(no CPU fallback exists by design)")


def _rows(t: torch.Tensor, name: str) -> torch.Tensor:
    """(B, T, F) or (N, F) -> contiguous float32 (N, F) (losses.py:158-165).

    complex64 rows (an STFT that has not been through `.abs()`, features.py:236) are kept complex:
    the kernels form the magnitude themselves and return complex gradients."""
    _require_cuda(t, name)
    if t.dtype in (torch.float16, torch.bfloat16, torch.float64):
        t = t.float()  # (float64: the reference accepts it; the kernels compute in float32, the result is cast back)
    elif t.dtype not in (torch.float32, torch.complex64):
        raise TypeError(f"sot_b200: `{name}` must be float32 (half / bfloat16 / float64 are converted) or complex64, "
                        f"got {t.dtype}")
    if t.ndim == 3:
        t = t.reshape(-1, t.shape[-1])
    elif t.ndim != 2:
        raise ValueError(f"sot_b200: `{name}` must be (batch, time, features) or (batch, features), got {tuple(t.shape)}")
    return t.contiguous()


def _support(pos: torch.Tensor, like: torch.Tensor, name: str, attach: bool = False) -> torch.Tensor:
    """1-D -> shared grid (the reference `expand`s it, losses.py:167-170; an expanded view is
    recognised and collapsed back); 2-D / 3-D -> per-frame rows.  `attach` keeps the positions in the
    autograd graph (`_position_term`); the kernels never see them attached."""
    if not attach:
        pos = pos.detach()
    if pos.device != like.device:
        raise ValueError(f"sot_b200: `{name}` is on {pos.device} but the spectra are on {like.device}")
    if pos.dtype != torch.float32:
        pos = pos.float()
    if pos.ndim == 3:
        pos = pos.reshape(-1, pos.shape[-1])
    if pos.ndim == 2 and (pos.shape[0] == 1 or pos.stride(0) == 0):
        pos = pos[0]
    if pos.ndim == 1:
        if pos.shape[0] != like.shape[1]:
            raise ValueError(f"sot_b200: `{name}` has {pos.shape[0]} positions for {like.shape[1]} bins")
        return pos.contiguous()
    if tuple(pos.shape) != tuple(like.shape):
        raise ValueError(f"sot_b200: `{name}` has shape {tuple(pos.shape)}, spectra {tuple(like.shape)}")
    return pos.contiguous()


def _version(t: torch.Tensor):
    """Version counter of a caller tensor, or None for an inference tensor (`torch.inference_mode`, which
    `metrics.wasserstein_distance` runs under, metrics.py:144): those are never cached."""
    try:
        return t._version
    except RuntimeError:
        return None


def _is_ascending(pos: torch.Tensor, owner: torch.Tensor) -> bool:
    """One device->host read per distinct (tensor object, version) of the caller's positions
    tensor `owner`; cached after that (a `fixed_x` buffer or a grid the caller keeps is checked once).

    Callers that build a NEW positions tensor every step (the reference's `trainer.py:187-197` does) pay this read
    -- and the one in `_uniform_grid` -- every step: a host synchronisation with the stream.  Keep the positions
    tensor (hoist it out of the step, as `features.Wasserstein1DWithTransform` does) and the step stays
    synchronisation free; INTEGRATION.md says so."""
    key = id(owner)
    version = _version(owner)
    hit = _sorted_cache.get(key)
    if hit is not None and version is not None and hit[0]() is owner and hit[1] == version:
        return hit[2]
    ok = bool((pos[..., 1:] >= pos[..., :-1]).all().item()) if pos.shape[-1] > 1 else True
    if version is not None:
        try:
            ref = weakref.ref(owner, lambda _, k=key: _sorted_cache.pop(k, None))
            _sorted_cache[key] = (ref, version, ok)
        except TypeError:
            pass
    return ok


def _order(pos: torch.Tensor, w: torch.Tensor, owner: torch.Tensor):
    """`require_sort` (losses.py:286-290) hoisted out of the kernel: supports that are already
    ascending (every linear grid, the log grid at n_fft 512) cost nothing; otherwise positions
    and weights are permuted once with a stable argsort before the launch.  Positions attached to
    the autograd graph stay attached through the sort."""
    if _is_ascending(pos, owner):
        return pos, w
    if pos.ndim == 1:
        pos_sorted, perm = torch.sort(pos, stable=True)
        return pos_sorted.contiguous(), w.index_select(1, perm)
    pos_sorted, perm = torch.sort(pos, dim=1, stable=True)
    return pos_sorted.contiguous(), torch.gather(w, 1, perm)


_uniform_cache: dict = {}  # (id(x_pos), id(y_pos)) -> (weakref, weakref, version, version, uniform?)


def _uniform_grid(pu: torch.Tensor, pv: torch.Tensor, owner_u: torch.Tensor, owner_v: torch.Tensor,
                  sorted_flags=(False, False)) -> bool:
    """Are both supports EXACT uniform grids pos[i] = pos[0] + i*h with one common power-of-two h, so
    that every position and every position difference is exact in float32?  True for rfftfreq / max
    with a power-of-two n_fft (trainer.py:193-197) and for `fixed_x = linspace(0, 1, 2**k + 1)`
    (losses.py:124-125).  The kernels then compute positions instead of loading them -- bit-identical
    results, fewer shared-memory accesses.  One device->host read per distinct pair of caller tensors."""
    if pu.ndim != 1 or pv.ndim != 1 or pu.shape[0] < 2 or pv.shape[0] < 2:
        return False
    key = (id(owner_u), id(owner_v), tuple(sorted_flags))  # (the verdict depends on whether a support was re-sorted)
    ver_u, ver_v = _version(owner_u), _version(owner_v)
    cacheable = ver_u is not None and ver_v is not None
    hit = _uniform_cache.get(key)
    if (hit is not None and cacheable and hit[0]() is owner_u and hit[1]() is owner_v and hit[2] == ver_u
            and hit[3] == ver_v):
        return hit[4]
    h = pu[1] - pu[0]
    ok = (pu == pu[0] + torch.arange(pu.shape[0], device=pu.device) * h).all() & \
         (pv == pv[0] + torch.arange(pv.shape[0], device=pv.device) * h).all()
    h_val, ok_val, u0, v0 = torch.stack((h, ok.to(h.dtype), pu[0], pv[0])).tolist()  # the one sync
    uniform = False
    if ok_val == 1.0 and h_val > 0.0:
        import math
        mant, _ = math.frexp(h_val)
        span = max(pu.shape[0], pv.shape[0]) + abs(u0 / h_val) + abs(v0 / h_val)
        uniform = (mant == 0.5 and float(u0 / h_val).is_integer() and float(v0 / h_val).is_integer()
                   and span < 2 ** 23)
    if cacheable:
        try:
            drop = lambda _, k=key: _uniform_cache.pop(k, None)  # noqa: E731
            _uniform_cache[key] = (weakref.ref(owner_u, drop), weakref.ref(owner_v, drop), ver_u, ver_v, uniform)
        except TypeError:
            pass
    return uniform


def _magnitude(t: torch.Tensor) -> torch.Tensor:
    return t.abs() if t.is_complex() else t


def _canonical(x, y, x_pos, y_pos, require_sort, raw_weights, keep_complex=False, attach_positions=False):
    """The reference's prologue that stays on the host, shared by every launch so that they all see the same rows:
    flatten, canonicalise the supports, hoisted sort.  Returns (u, v, pu, pv, (sorted u?, sorted v?)).

    Complex rows stay complex only for the fused loss launch (`keep_complex`), and only when both sides are complex
    and short enough for its |z| prologue in shared memory; otherwise |z| is taken in torch (the real path takes any
    length).  `attach_positions` keeps the positions in the autograd graph for `_position_term`."""
    if not keep_complex:
        x, y = _magnitude(x), _magnitude(y)
    u, v = _rows(x, "x"), _rows(y, "y")
    if not (u.is_complex() and v.is_complex() and max(u.shape[1], v.shape[1]) <= _capi.MAX_COMPLEX_BINS):
        u, v = _magnitude(u), _magnitude(v)
    if u.is_complex() and raw_weights:
        raise TypeError("sot_b200: `wasserstein_1d` weights must be real")
    if u.shape[0] != v.shape[0]:
        raise ValueError(f"sot_b200: x has {u.shape[0]} frames, y has {v.shape[0]}")
    pu, pv = _support(x_pos, u, "x_pos", attach_positions), _support(y_pos, v, "y_pos", attach_positions)
    sort_u, sort_v = require_sort if isinstance(require_sort, tuple) else (require_sort, require_sort)
    if sort_u:
        pu, u = _order(pu, u, x_pos)
    if sort_v:
        pv, v = _order(pv, v, y_pos)
    return u, v, pu, pv, (bool(sort_u), bool(sort_v))


def _flags(square, cut_scale, raw_weights, limit=False, uniform=False) -> int:
    return ((_capi.SOT_SQUARE if square else 0) | (_capi.SOT_CUT_SCALE if cut_scale else 0) |
            (_capi.SOT_LIMIT if limit else 0) | (_capi.SOT_RAW_WEIGHTS if raw_weights else 0) |
            (_capi.SOT_UNIFORM_GRID if uniform else 0))


def _prepare(x, y, x_pos, y_pos, p, square, cut_scale, limit, require_sort, raw_weights):
    """Rows, supports and flags of the loss and gradient launches."""
    assert p >= 1, f"The OT loss is only valid for p>=1, {p} was given"  # losses.py:271
    u, v, pu, pv, sort = _canonical(x, y, x_pos, y_pos, require_sort, raw_weights, keep_complex=True)
    return u, v, pu, pv, _flags(square, cut_scale, raw_weights, limit, _uniform_grid(pu, pv, x_pos, y_pos, sort))


# --------------------------------------------------------------------------------------
# gradients w.r.t. the support positions
# --------------------------------------------------------------------------------------
def _wants_position_grad(x_pos, y_pos) -> bool:
    return torch.is_grad_enabled() and (x_pos.requires_grad or y_pos.requires_grad)


def position_term_from_plan(qs, iu, iv, pu, pv, p, limit) -> torch.Tensor:
    """Per-frame loss (N,) as a function of the SORTED support positions `pu`, `pv` (1-D shared rows or (N, F)), the
    transport plan held fixed: `qs` (N, K) merged quantile grid, `iu` / `iv` (N, K) un-clamped `searchsorted` indices.
    This is losses.py:301-313 with `quantile_function`'s `xs[idx]` (losses.py:219-220) as the only place the positions
    enter -- which is also the only way they enter the reference's autograd graph, so the gradients w.r.t. the
    positions are the reference's.  Plain torch ops (runs wherever the tensors live; the CPU tests use it as is)."""
    def take(pos, idx):
        idx = idx.long().clamp(max=pos.shape[-1] - 1)  # losses.py:220
        return pos[idx] if pos.ndim == 1 else torch.gather(pos, 1, idx)
    delta = qs - torch.nn.functional.pad(qs, pad=(1, 0))[..., :-1]  # losses.py:301-304
    if limit:
        delta = torch.where(qs > 1, torch.zeros_like(delta), delta)  # losses.py:306-307
    diff = torch.abs(take(pu, iu) - take(pv, iv))
    return torch.sum(delta * (diff if p == 1 else diff.pow(p)), 1)  # losses.py:311-313


def _position_term(x, y, x_pos, y_pos, p, square, cut_scale, limit, require_sort, raw_weights) -> torch.Tensor:
    """Per-frame loss attached to the autograd graph of x_pos / y_pos only (the spectra are constants here): the plan
    kernel (`OUT_PLAN`) finds the merged grid and the indices, `position_term_from_plan` is differentiated by torch.
    A path the paper's configurations never take (trainer.py:187-197 builds the positions without gradients): an extra
    plan launch and ATen-sized temporaries, only when a position tensor requires a gradient."""
    u, v, pu, pv, _ = _canonical(x.detach(), y.detach(), x_pos, y_pos, require_sort, raw_weights,
                                 attach_positions=True)
    _, _, qs, _, _, iu, iv = _capi.quantiles(u, v, pu.detach(), pv.detach(), _flags(square, cut_scale, raw_weights),
                                             want_indices=True)
    return position_term_from_plan(qs, iu, iv, pu, pv, p, limit)


def sot_frames(x, y, x_pos, y_pos, p=1, square=False, cut_scale=False, limit=False, require_sort=True,
               raw_weights=False, backward_mode="recompute") -> torch.Tensor:
    """Per-frame W_p^p, shape (N,), differentiable w.r.t. x and y (and, through `_position_term`, the positions)."""
    if backward_mode not in BACKWARD_MODES:
        raise ValueError(f"backward_mode must be one of {BACKWARD_MODES}")
    u, v, pu, pv, flags = _prepare(x, y, x_pos, y_pos, p, square, cut_scale, limit, require_sort, raw_weights)
    rows = _SotFrames.apply(u, v, pu, pv, float(p), flags, backward_mode)
    if _wants_position_grad(x_pos, y_pos):  # value unchanged (+ exactly 0); the gradient w.r.t. the positions rides on it
        term = _position_term(x, y, x_pos, y_pos, p, square, cut_scale, limit, require_sort, raw_weights)
        rows = rows + (term - term.detach())
    return rows


class _SotMean(torch.autograd.Function):
    """rows (N, n), (N, m) -> mean over the frames of ALL ranks of W_p^p, a 0-dim tensor.

    The mean the reference takes at the end (losses.py:211) and the whole backward folded into ONE launch
    (mode "onepass"): when a gradient is required the forward launches the fused forward+backward kernel, which
    writes the gradient rows of the mean (already scaled by 1/N_global) and whose last CTA writes the float mean --
    no memset, division, cast or reduction kernel, no host synchronisation.  The backward is an in-place
    `rows *= dL/dmean` that leaves at once when the upstream gradient is exactly 1 (trainer.py:220,233-238: the
    loss enters the total with weight 1).  Mode "recompute" keeps nothing between the passes: loss-only launch
    forward, fused launch backward.  With an `exchange` (sharding.MeanExchange) the per-rank sums meet in ONE
    exchange that the backward never waits for: 1/N_global depends on the frame counts only."""

    @staticmethod
    def forward(ctx, u, v, pos_u, pos_v, p, flags, exchange, mode):
        need_u, need_v = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        n_local = u.shape[0]
        kw = {}
        n_global = float(n_local)
        if exchange is not None:
            n_global = exchange.global_count(n_local, u.device)
            kw = exchange.launch_kwargs(n_local, u.device)
        onepass = mode == "onepass" and (need_u or need_v)
        mean, _, gu, gv = _capi.mean_step(u, v, pos_u, pos_v, p, flags, grad_scale=1.0 / n_global,
                                          mean_scale=1.0 / n_local, want_gu=onepass and need_u,
                                          want_gv=onepass and need_v, **kw)
        if exchange is not None:
            mean = exchange.finish(kw, n_global, u.device)
        ctx.p, ctx.flags, ctx.need, ctx.n_global = p, flags, (need_u, need_v), n_global
        ctx.gu, ctx.gv = gu, gv  # taken (and dropped) by the first backward
        ctx.save_for_backward(u, v, pos_u, pos_v)  # references only; a repeated backward recomputes from them
        return mean

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_out):
        need_u, need_v = ctx.need
        g = grad_out.detach().to(torch.float32).reshape(1)
        gu, gv = ctx.gu, ctx.gv
        ctx.gu = ctx.gv = None
        if gu is not None or gv is not None:
            _capi.scale_inplace(gu, gv, g)  # leaves at once for an upstream gradient of exactly 1
        else:  # "recompute" mode, or a second backward through a retained graph
            u, v, pos_u, pos_v = ctx.saved_tensors
            _, _, gu, gv = _capi.mean_step(u, v, pos_u, pos_v, ctx.p, ctx.flags, grad_scale=1.0 / ctx.n_global,
                                           mean_scale=0.0, want_gu=need_u, want_gv=need_v, grad_scale_device=g,
                                           want_mean=False)
        return gu, gv, None, None, None, None, None, None


def sot_mean(x, y, x_pos, y_pos, p=1, square=False, cut_scale=False, limit=False, require_sort=True,
             raw_weights=False, exchange=None, backward_mode="onepass") -> torch.Tensor:
    """mean_n W_p^p(frame n) over this rank's frames -- and over all ranks' when `exchange` (a
    `sharding.MeanExchange`) spans more than one -- differentiable w.r.t. x and y.  One SOT launch a step plus the
    in-place scaling of the backward."""
    if backward_mode not in MEAN_BACKWARD_MODES:
        raise ValueError(f"backward_mode must be one of {MEAN_BACKWARD_MODES}")
    u, v, pu, pv, flags = _prepare(x, y, x_pos, y_pos, p, square, cut_scale, limit, require_sort, raw_weights)
    value = _SotMean.apply(u, v, pu, pv, float(p), flags, exchange, backward_mode)
    if _wants_position_grad(x_pos, y_pos):
        if exchange is not None:
            raise NotImplementedError("sot_b200: gradients w.r.t. support positions are not available for the sharded "
                                      "mean (use the plain Wasserstein1D and reduce the position gradients yourself)")
        term = _position_term(x, y, x_pos, y_pos, p, square, cut_scale, limit, require_sort, raw_weights).mean()
        value = value + (term - term.detach())
    return value


# --------------------------------------------------------------------------------------
# the reference's public surface
# --------------------------------------------------------------------------------------
class Wasserstein1D(torch.nn.Module):
    def __init__(self, p=1, fixed_x=None, require_sort=True, log_scaled_x=False, **kwargs):
        """Same arguments as the reference (losses.py:90-127).  `kwargs` read: dont_normalize,
        limit_quantile_range, hinge, square_dist -- plus `backward_mode`, which only this implementation knows:
        "onepass" (default: ONE fused launch per step, gradients produced by the forward launch), "recompute"
        (nothing kept between the passes: loss-only launch forward, fused launch backward) or "fused" (alias of
        "onepass" for the mean; per-frame outputs: unit gradients saved, row scaling backward).  Any other key is
        ignored like the reference does."""
        super().__init__()
        self.p = p
        self.require_sort = require_sort
        self.log_scaled_x = log_scaled_x  # inert in the reference too (losses.py:117)
        self.dont_normalize = kwargs.get("dont_normalize", False)
        self.limit_quantile_range = kwargs.get("limit_quantile_range", False)
        self.hinge = kwargs.get("hinge", False)
        self.square_dist = kwargs.get("square_dist", False)
        self.backward_mode = kwargs.get("backward_mode", DEFAULT_BACKWARD_MODE)
        if self.backward_mode not in ("onepass", "recompute", "fused"):
            raise ValueError('backward_mode must be "onepass", "recompute" or "fused"')
        if fixed_x is not None:
            self.register_buffer("fixed_x", torch.linspace(0, 1, fixed_x))
        else:
            self.register_buffer("fixed_x", None)

    def _mean_exchange(self):
        """How the ranks' sums meet for the final mean; the single-process reference has no ranks (None).
        `sharding.ShardedWasserstein1D` overrides this."""
        return None

    def forward(self, x, y, x_pos=None, y_pos=None, **kwargs):
        if (x_pos is None or y_pos is None) and self.fixed_x is None:
            raise ValueError("If fixed_x is not provided, x_pos and y_pos must be provided")
        x_pos_ = self.fixed_x if x_pos is None else x_pos
        y_pos_ = self.fixed_x if y_pos is None else y_pos
        if x_pos_.device != x.device:  # a `fixed_x` buffer left behind by `MixOfLosses` (plain list)
            x_pos_ = x_pos_.to(x.device)
        if y_pos_.device != y.device:
            y_pos_ = y_pos_.to(y.device)

        # the `fixed_x` grid is a linspace: ascending by construction, no check needed
        need_sort = (bool(self.require_sort) and x_pos is not None, bool(self.require_sort) and y_pos is not None)
        original_shape = x.shape[:-1]
        cut_scale = bool(kwargs.get("dont_normalize", False) or self.dont_normalize)
        limit = bool(kwargs.get("limit_quantile_range", False) or self.limit_quantile_range)

        if kwargs.get("return_quantiles", False):
            out = _quantiles(x, y, x_pos_, y_pos_, bool(self.square_dist), cut_scale, need_sort)
            return [t.reshape(original_shape + (-1,)) for t in out]  # losses.py:198-201

        mode = getattr(self, "backward_mode", DEFAULT_BACKWARD_MODE)
        as64 = x.dtype == torch.float64 or y.dtype == torch.float64  # the reference returns float64 then
        if not self.hinge and kwargs.get("dims", None) is None and x.numel() > 0:
            # plain mean over all frames (every paper config): folded into the one kernel launch
            value = sot_mean(x, y, x_pos_, y_pos_, p=self.p, square=bool(self.square_dist), cut_scale=cut_scale,
                             limit=limit, require_sort=need_sort, exchange=self._mean_exchange(),
                             backward_mode="recompute" if mode == "recompute" else "onepass")
            return value.double() if as64 else value
        loss = sot_frames(x, y, x_pos_, y_pos_, p=self.p, square=bool(self.square_dist), cut_scale=cut_scale,
                          limit=limit, require_sort=need_sort,
                          backward_mode="recompute" if mode == "recompute" else "fused")
        if self.hinge:  # losses.py:203-205: the ctor flag gates, the call kwarg is the threshold
            loss = torch.nn.functional.relu(loss - kwargs.get("hinge", 0.0))
        return self._reduce_frames(loss.reshape(original_shape), kwargs.get("dims", None), as64)

    def _reduce_frames(self, loss, dims, as64):
        """The reference's final `torch.mean(loss, dim=dims)` (losses.py:211) of the per-frame values, cast back to
        float64 when an input was.  `sharding.ShardedWasserstein1D` overrides this."""
        return torch.mean(loss.double() if as64 else loss, dim=dims)


def _quantiles(x, y, x_pos, y_pos, square, cut_scale, require_sort, raw_weights=False):
    u, v, pu, pv, _ = _canonical(x.detach(), y.detach(), x_pos, y_pos, require_sort, raw_weights)
    return _capi.quantiles(u, v, pu, pv, _flags(square, cut_scale, raw_weights))


def quantile_function(qs, cws, xs):
    """losses.py:214-220: positions `xs` at the first CDF entry >= each level of `qs`."""
    return _capi.quantile_lookup(qs.contiguous().float(), cws.contiguous().float(), xs.contiguous().float())


def wasserstein_1d(u_values, v_values, u_weights=None, v_weights=None, p=1, require_sort=True,
                   return_quantiles=False, limit_quantile_range=False):
    """Module-level entry of the reference (losses.py:223-313): positions `*_values` (batch, n),
    weights used as given (uniform 1/n if None).  Returns (batch,) W_p^p, or the five quantile
    tensors when `return_quantiles`."""
    assert p >= 1, f"The OT loss is only valid for p>=1, {p} was given"
    n, m = u_values.shape[1], v_values.shape[1]
    if u_weights is None:
        u_weights = torch.full(u_values.shape, 1.0 / n, device=u_values.device, dtype=u_values.dtype)
    if v_weights is None:
        v_weights = torch.full(v_values.shape, 1.0 / m, device=v_values.device, dtype=v_values.dtype)
    if return_quantiles:
        return tuple(_quantiles(u_weights, v_weights, u_values, v_values, False, False, require_sort,
                                raw_weights=True))
    return sot_frames(u_weights, v_weights, u_values, v_values, p=p, limit=limit_quantile_range,
                      require_sort=require_sort, raw_weights=True)
