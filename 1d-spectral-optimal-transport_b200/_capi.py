"""ctypes binding of `libsot_b200.so` (C ABI declared in include/sot_b200.h).

This is the only way the Python layer reaches the kernels.  There is no fallback: if the library
cannot be loaded (or built) every entry point raises.
"""
from __future__ import annotations

import ctypes
import os
import threading

import torch

from . import build as _build

SOT_SQUARE, SOT_CUT_SCALE, SOT_LIMIT, SOT_RAW_WEIGHTS, SOT_UNIFORM_GRID, SOT_COMPLEX_INPUT = 1, 2, 4, 8, 16, 32
ABI_VERSION = 3
MAX_COMPLEX_BINS = 4352  # longest SOT_COMPLEX_INPUT row (include/sot_b200.h: sot_max_bins); real rows take 2^24 - 1

_c_float_p = ctypes.c_void_p  # device pointers travel as integers


class SotProblem(ctypes.Structure):
    """`struct sot_problem` of include/sot_b200.h."""
    _fields_ = [
        ("n_frames", ctypes.c_int64),
        ("n_u", ctypes.c_int32),
        ("n_v", ctypes.c_int32),
        ("u", ctypes.c_void_p),
        ("v", ctypes.c_void_p),
        ("pos_u", ctypes.c_void_p),
        ("pos_v", ctypes.c_void_p),
        ("pos_u_stride", ctypes.c_int64),
        ("pos_v_stride", ctypes.c_int64),
        ("p", ctypes.c_float),
        ("flags", ctypes.c_int32),
    ]


class SotMeanPlan(ctypes.Structure):
    """`struct sot_mean_plan` of include/sot_b200.h."""
    _fields_ = [
        ("workspace", ctypes.c_void_p),
        ("mean_out", ctypes.c_void_p),
        ("mean_scale", ctypes.c_double),
        ("total_out", ctypes.c_void_p),
        ("count_value", ctypes.c_double),
        ("post_mailboxes", ctypes.POINTER(ctypes.c_void_p)),
        ("post_world", ctypes.c_int32),
        ("post_rank", ctypes.c_int32),
        ("post_seq", ctypes.c_uint64),
        ("post_seq_device", ctypes.c_void_p),
        ("grad_scale", ctypes.c_float),
        ("grad_scale_device", ctypes.c_void_p),
    ]


class SotPairwiseProblem(ctypes.Structure):
    """`struct sot_pairwise_problem` of include/sot_b200.h."""
    _fields_ = [
        ("batch", ctypes.c_int64),
        ("rows_u", ctypes.c_int64),
        ("rows_v", ctypes.c_int64),
        ("n_u", ctypes.c_int32),
        ("n_v", ctypes.c_int32),
        ("u", ctypes.c_void_p),
        ("v", ctypes.c_void_p),
        ("pos_u", ctypes.c_void_p),
        ("pos_v", ctypes.c_void_p),
        ("p", ctypes.c_float),
        ("flags", ctypes.c_int32),
    ]


class SotBarycenterProblem(ctypes.Structure):
    """`struct sot_barycenter_problem` of include/sot_b200.h."""
    _fields_ = [
        ("count", ctypes.c_int64),
        ("k", ctypes.c_int32),
        ("n", ctypes.c_int32),
        ("n_out", ctypes.c_int32),
        ("x", ctypes.c_void_p),
        ("weights", ctypes.c_void_p),
        ("weights_stride", ctypes.c_int64),
        ("pos", ctypes.c_void_p),
        ("pos_out", ctypes.c_void_p),
        ("flags", ctypes.c_int32),
    ]


# name -> (restype, argtypes); kept in one place so tests can check the exported symbol table
_P = ctypes.POINTER(SotProblem)
_PP = ctypes.POINTER(SotPairwiseProblem)
_PB = ctypes.POINTER(SotBarycenterProblem)
_V = ctypes.c_void_p
SIGNATURES = {
    "sot_forward_device": (ctypes.c_int, [_P, _V, _V]),
    "sot_forward_backward_device": (ctypes.c_int, [_P, _V, _V, _V, _V, _V]),
    "sot_scale_rows_device": (ctypes.c_int, [_V, _V, _V, ctypes.c_int64, ctypes.c_int32, _V]),
    "sot_mean_step_device": (ctypes.c_int, [_P, ctypes.POINTER(SotMeanPlan), _V, _V, _V, _V]),
    "sot_scale_inplace_device": (ctypes.c_int, [_V, ctypes.c_int64, _V, ctypes.c_int64, _V, _V]),
    "sot_quantiles_device": (ctypes.c_int, [_P, _V, _V, _V, _V, _V, _V, _V, _V]),
    "sot_quantile_lookup_device": (ctypes.c_int, [_V, _V, _V, _V, ctypes.c_int64, ctypes.c_int32,
                                                  ctypes.c_int32, _V]),
    "sot_plan_from_cdf_device": (ctypes.c_int, [_P, _V, _V, _V, _V, _V, _V]),
    "sot_loss_from_cdf_device": (ctypes.c_int, [_P, _V, _V, _V, _V]),
    "sot_loss_grad_host": (ctypes.c_int, [_P, _V, _V, _V, _V, ctypes.c_int32]),
    "sot_pairwise_device": (ctypes.c_int, [_PP, _V, _V]),
    "sot_pairwise_backward_device": (ctypes.c_int, [_PP, _V, _V, _V, _V]),
    "sot_barycenter_device": (ctypes.c_int, [_PB, _V, _V]),
    "sot_barycenter_backward_device": (ctypes.c_int, [_PB, _V, _V, _V]),
    "sot_host_release": (ctypes.c_int, [ctypes.c_int32]),
    "sot_abi_version": (ctypes.c_int, []),
    "sot_last_error": (ctypes.c_char_p, []),
    "sot_max_bins": (ctypes.c_int, [ctypes.c_int32, ctypes.c_int32]),
    "sot_set_tuning": (ctypes.c_int, [ctypes.c_int32, ctypes.c_int32, ctypes.c_int32]),
    "sot_launch_count": (ctypes.c_int64, []),
    "sot_mss_forward_device": (ctypes.c_int, [_V, _V, ctypes.c_int64, ctypes.c_float, ctypes.c_float, ctypes.c_int32,
                                              ctypes.c_float, _V, _V]),
    "sot_mss_backward_device": (ctypes.c_int, [_V, _V, ctypes.c_int64, ctypes.c_float, ctypes.c_float, ctypes.c_int32,
                                               ctypes.c_float, _V, _V, _V, _V]),
}
SIGNATURES["sot_p2p_mailbox_doubles"] = (ctypes.c_int, [ctypes.c_int32])
SIGNATURES["sot_p2p_allreduce_device"] = (ctypes.c_int, [_V, _V, ctypes.c_int32, ctypes.POINTER(ctypes.c_void_p),
                                                         ctypes.c_int32, ctypes.c_int32, ctypes.c_uint64, _V])
SIGNATURES["sot_p2p_global_mean_device"] = (ctypes.c_int, [_V, ctypes.c_double, _V, _V, ctypes.POINTER(ctypes.c_void_p),
                                                           ctypes.c_int32, ctypes.c_int32, ctypes.c_uint64, _V])
SIGNATURES["sot_p2p_wait_mean_device"] = (ctypes.c_int, [_V, ctypes.c_double, _V, ctypes.POINTER(ctypes.c_void_p),
                                                         ctypes.c_int32, ctypes.c_int32, ctypes.c_uint64, _V,
                                                         ctypes.c_uint32, _V])
SOT_MSS_L1, SOT_MSS_L2 = 0, 1

_lib = None
_lock = threading.Lock()


class SotError(RuntimeError):
    pass


def library_path() -> str:
    """The in-tree library; SOT_B200_LIBRARY points developers' tuning experiments at another build of it."""
    return os.environ.get("SOT_B200_LIBRARY") or _build.LIB_PATH


def load(build_if_needed: bool = True):
    """Load (building first if the in-tree library is missing or stale) and return the CDLL."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = library_path()
        if path == _build.LIB_PATH and build_if_needed and _build.is_stale():
            _build.build()
        if not os.path.exists(path):
            raise SotError(f"{path} is missing: build it with `python -m sot_b200.build` "
                           "(this package has no CPU or eager fallback)")
        lib = ctypes.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError here = header / library mismatch
            fn.restype, fn.argtypes = res, args
        if lib.sot_abi_version() != ABI_VERSION:
            raise SotError("libsot_b200.so ABI version mismatch: rebuild with `python -m sot_b200.build --force`")
        _lib = lib
        return lib


def _check(rc: int):
    if rc == 0:
        return
    msg = load().sot_last_error().decode("utf-8", "replace")
    if rc == -3:
        raise AssertionError(msg)  # p < 1: the reference asserts (losses.py:271)
    if rc < 0:
        raise ValueError(f"sot_b200: {msg}")
    raise SotError(f"sot_b200 CUDA error {rc}: {msg}")


def _dev_tensor(t: torch.Tensor, name: str, complex_ok: bool = False) -> torch.Tensor:
    if not t.is_cuda:
        raise SotError(f"sot_b200: `{name}` lives on {t.device}; the SOT kernels are CUDA only "
                       "(no CPU fallback exists by design)")
    if t.dtype != torch.float32 and not (complex_ok and t.dtype == torch.complex64):
        raise TypeError(f"sot_b200: `{name}` must be float32{' or complex64' if complex_ok else ''}, got {t.dtype}")
    return t


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream(device) -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


class _on_device:
    """`torch.cuda.device(dev)` only when `dev` is not the current device already (the guard costs ~10 us of host
    time per call, which matters for launch-bound shards)."""

    def __init__(self, device):
        self.guard = None if device.index is None or device.index == torch.cuda.current_device() else \
            torch.cuda.device(device)

    def __enter__(self):
        if self.guard is not None:
            self.guard.__enter__()

    def __exit__(self, *exc):
        if self.guard is not None:
            return self.guard.__exit__(*exc)
        return False


def _launch(name: str, device, *args, stream=None) -> None:
    """Calls the C entry point `name` with `args` and the current stream of `device` (or `stream`, a
    `torch.cuda.Stream`) on that device; raises on a non-zero return code."""
    fn = getattr(load(), name)
    handle = _stream(device) if stream is None else ctypes.c_void_p(stream.cuda_stream)
    with _on_device(device):
        _check(fn(*args, handle))


def make_problem(u, v, pos_u, pos_v, p: float, flags: int) -> SotProblem:
    """u: (N, n), v: (N, m) contiguous CUDA float32; pos_*: (n,) shared or (N, n) per frame.

    u and v may both be complex64 STFT rows instead: the magnitude is then formed inside the kernel
    (SOT_COMPLEX_INPUT is added to the flags) and the gradients come back as complex64 rows."""
    _dev_tensor(u, "x", True), _dev_tensor(v, "y", True), _dev_tensor(pos_u, "x_pos"), _dev_tensor(pos_v, "y_pos")
    if u.dtype != v.dtype:
        raise TypeError(f"sot_b200: `x` and `y` must have the same dtype, got {u.dtype} and {v.dtype}")
    if u.is_complex():
        flags = int(flags) | SOT_COMPLEX_INPUT
    return _problem(u, v, pos_u, pos_v, p, flags)


def _problem(u, v, pos_u, pos_v, p: float, flags: int) -> SotProblem:
    """The shape and stride rules shared by the device entry points and the host-buffer one."""
    if u.ndim != 2 or v.ndim != 2 or u.shape[0] != v.shape[0]:
        raise ValueError(f"sot_b200: expected (N, n) and (N, m) rows, got {tuple(u.shape)} and {tuple(v.shape)}")
    if not (u.is_contiguous() and v.is_contiguous() and pos_u.is_contiguous() and pos_v.is_contiguous()):
        raise ValueError("sot_b200: tensors must be contiguous")
    if len({u.device, v.device, pos_u.device, pos_v.device}) != 1:
        raise ValueError("sot_b200: all tensors must be on the same CUDA device")
    N, n = u.shape
    m = v.shape[1]
    strides = []
    for pos, width, name in ((pos_u, n, "x_pos"), (pos_v, m, "y_pos")):
        if pos.ndim == 1 and pos.shape[0] == width:
            strides.append(0)
        elif pos.ndim == 2 and tuple(pos.shape) == (N, width):
            strides.append(width)
        else:
            raise ValueError(f"sot_b200: `{name}` has shape {tuple(pos.shape)}, expected ({width},) or ({N}, {width})")
    return SotProblem(N, n, m, u.data_ptr(), v.data_ptr(), pos_u.data_ptr(), pos_v.data_ptr(),
                      strides[0], strides[1], float(p), int(flags))


def forward(u, v, pos_u, pos_v, p, flags) -> torch.Tensor:
    prob = make_problem(u, v, pos_u, pos_v, p, flags)
    loss = torch.empty(u.shape[0], dtype=torch.float32, device=u.device)
    _launch("sot_forward_device", u.device, ctypes.byref(prob), _ptr(loss))
    return loss


def forward_backward(u, v, pos_u, pos_v, p, flags, upstream=None, want_loss=True, want_gu=True, want_gv=True):
    prob = make_problem(u, v, pos_u, pos_v, p, flags)
    if upstream is not None:
        _dev_tensor(upstream, "upstream")
        if upstream.shape != (u.shape[0],) or not upstream.is_contiguous():
            raise ValueError("sot_b200: upstream gradient must be a contiguous (N,) tensor")
    loss = torch.empty(u.shape[0], dtype=torch.float32, device=u.device) if want_loss else None
    gu = torch.empty_like(u) if want_gu else None
    gv = torch.empty_like(v) if want_gv else None
    _launch("sot_forward_backward_device", u.device, ctypes.byref(prob), _ptr(upstream), _ptr(loss), _ptr(gu),
            _ptr(gv))
    return loss, gu, gv


_workspaces: dict = {}  # (device index, stream handle) -> 2 zeroed doubles the mean-step kernel keeps zero


def mean_workspace(device) -> torch.Tensor:
    """The (sum, ticket) accumulator of `sot_mean_step_device` for the current stream of `device`: allocated and
    zeroed once, left zero by every launch (its last CTA resets it)."""
    key = (torch.device(device).index, torch.cuda.current_stream(device).cuda_stream)
    ws = _workspaces.get(key)
    if ws is None:
        ws = torch.zeros(2, dtype=torch.float64, device=device)
        _workspaces[key] = ws
    return ws


def mean_step(u, v, pos_u, pos_v, p, flags, grad_scale: float, mean_scale: float, want_gu=True, want_gv=True,
              want_rows=False, total_out=None, count_value: float = 0.0, post=None, grad_scale_device=None,
              want_mean=None):
    """ONE launch: mean over this launch's frames (times `mean_scale` * N, i.e. sum * mean_scale) as a 0-dim float32
    tensor, and the gradient rows of `grad_scale * sum_n loss_n`.  `total_out`: (2,) float64 tensor that receives
    (sum, count_value) instead of / besides the mean; `post` = (mailbox pointers, rank, seq): the last CTA also
    stores (sum, count_value, seq) into every peer's mailbox (seq: an int, or a one-element int64 DEVICE tensor
    holding the previous call number).  Returns (mean or None, rows or None, gu, gv)."""
    prob = make_problem(u, v, pos_u, pos_v, p, flags)
    dev = u.device
    if want_mean is None:
        want_mean = total_out is None and post is None
    if grad_scale_device is not None:
        _dev_tensor(grad_scale_device, "grad_scale_device")
    mean = torch.empty((), dtype=torch.float32, device=dev) if want_mean else None
    rows = torch.empty(u.shape[0], dtype=torch.float32, device=dev) if want_rows else None
    gu = torch.empty_like(u) if want_gu else None
    gv = torch.empty_like(v) if want_gv else None
    plan = SotMeanPlan()
    plan.workspace = mean_workspace(dev).data_ptr()
    plan.mean_out = None if mean is None else mean.data_ptr()
    plan.mean_scale = float(mean_scale)
    plan.total_out = None if total_out is None else total_out.data_ptr()
    plan.count_value = float(count_value)
    plan.grad_scale = float(grad_scale)
    plan.grad_scale_device = None if grad_scale_device is None else grad_scale_device.data_ptr()
    keep = None
    if post is not None:
        ptrs, rank, seq = post
        keep = mailbox_array(ptrs)
        plan.post_mailboxes, plan.post_world, plan.post_rank = keep, len(keep), int(rank)
        if isinstance(seq, torch.Tensor):
            plan.post_seq, plan.post_seq_device = 0, seq.data_ptr()
        else:
            plan.post_seq = int(seq)
    _launch("sot_mean_step_device", dev, ctypes.byref(prob), ctypes.byref(plan), _ptr(rows), _ptr(gu), _ptr(gv))
    return mean, rows, gu, gv


def mailbox_array(ptrs):
    """ctypes array of the peers' mailbox pointers (build it once, pass it to every call); an array is returned as
    it is."""
    if isinstance(ptrs, ctypes.Array):
        return ptrs
    return (ctypes.c_void_p * len(ptrs))(*[ctypes.c_void_p(int(q)) for q in ptrs])


def scale_inplace(a, b, scale) -> None:
    """a *= scale; b *= scale in place (either may be None); `scale` = one-element float32 DEVICE tensor.  The
    kernel leaves at once when the scalar is exactly 1."""
    _dev_tensor(scale, "scale")
    if scale.numel() != 1:
        raise ValueError("sot_b200: the scale must hold one element")
    dev = scale.device
    views = []
    for t in (a, b):
        if t is None:
            views.append(None)
            continue
        if not t.is_contiguous() or t.device != dev:
            raise ValueError("sot_b200: rows to scale must be contiguous and on the scale's device")
        views.append(torch.view_as_real(t) if t.is_complex() else t)
    va, vb = views
    _launch("sot_scale_inplace_device", dev, _ptr(va), 0 if va is None else va.numel(), _ptr(vb),
            0 if vb is None else vb.numel(), _ptr(scale))


def scale_rows(unit, scale) -> torch.Tensor:
    """unit (N, F) float32 or complex64 rows times scale (N,): a new tensor."""
    _dev_tensor(unit, "unit", True), _dev_tensor(scale, "scale")
    out = torch.empty_like(unit)
    width = 2 * unit.shape[1] if unit.is_complex() else unit.shape[1]  # (interleaved re, im pairs)
    _launch("sot_scale_rows_device", unit.device, _ptr(unit), _ptr(scale), _ptr(out), unit.shape[0], width)
    return out


def quantiles(u, v, pos_u, pos_v, flags, from_cdf=False, want_indices=False):
    """(uq, vq, qs, cu, cv[, iu, iv]); with `from_cdf` the rows ARE the CDFs (parity harness)."""
    prob = make_problem(u, v, pos_u, pos_v, 2.0, flags)
    N, n = u.shape
    m = v.shape[1]
    f32 = dict(dtype=torch.float32, device=u.device)
    uq, vq, qs = (torch.empty(N, n + m, **f32) for _ in range(3))
    iu = torch.empty(N, n + m, dtype=torch.int32, device=u.device) if want_indices else None
    iv = torch.empty(N, n + m, dtype=torch.int32, device=u.device) if want_indices else None
    if from_cdf:
        cu, cv = u, v
        _launch("sot_plan_from_cdf_device", u.device, ctypes.byref(prob), _ptr(uq), _ptr(vq), _ptr(qs), _ptr(iu),
                _ptr(iv))
    else:
        cu, cv = torch.empty(N, n, **f32), torch.empty(N, m, **f32)
        _launch("sot_quantiles_device", u.device, ctypes.byref(prob), _ptr(uq), _ptr(vq), _ptr(qs), _ptr(cu),
                _ptr(cv), _ptr(iu), _ptr(iv))
    return (uq, vq, qs, cu, cv, iu, iv) if want_indices else (uq, vq, qs, cu, cv)


MAX_PAIRWISE_BINS = 8448  # longest row of the pairwise entry points (include/sot_b200.h)


def pairwise_problem(u, v, pos_u, pos_v, p: float, flags: int) -> SotPairwiseProblem:
    """u: (B, P, n), v: (B, R, m) contiguous CUDA float32; pos_u (n,), pos_v (m,) ascending."""
    for t, name in ((u, "x"), (v, "y"), (pos_u, "x_pos"), (pos_v, "y_pos")):
        _dev_tensor(t, name)
        if not t.is_contiguous():
            raise ValueError("sot_b200: tensors must be contiguous")
    if u.ndim != 3 or v.ndim != 3 or u.shape[0] != v.shape[0]:
        raise ValueError(f"sot_b200: expected (B, P, n) and (B, R, m) rows, got {tuple(u.shape)} and {tuple(v.shape)}")
    if pos_u.shape != (u.shape[2],) or pos_v.shape != (v.shape[2],):
        raise ValueError(f"sot_b200: positions of shape {tuple(pos_u.shape)} / {tuple(pos_v.shape)} for rows of "
                         f"{u.shape[2]} / {v.shape[2]} bins")
    if len({u.device, v.device, pos_u.device, pos_v.device}) != 1:
        raise ValueError("sot_b200: all tensors must be on the same CUDA device")
    return SotPairwiseProblem(u.shape[0], u.shape[1], v.shape[1], u.shape[2], v.shape[2], u.data_ptr(), v.data_ptr(),
                              pos_u.data_ptr(), pos_v.data_ptr(), float(p), int(flags))


def pairwise(u, v, pos_u, pos_v, p, flags) -> torch.Tensor:
    """(B, P, R) float32: W_p^p of every (u[b, i], v[b, j])."""
    prob = pairwise_problem(u, v, pos_u, pos_v, p, flags)
    dist = torch.empty(u.shape[0], u.shape[1], v.shape[1], dtype=torch.float32, device=u.device)
    _launch("sot_pairwise_device", u.device, ctypes.byref(prob), _ptr(dist))
    return dist


def pairwise_backward(u, v, pos_u, pos_v, p, flags, upstream, want_gu=True, want_gv=True):
    """Gradients of sum_{b,i,j} upstream[b, i, j] * dist[b, i, j] w.r.t. u and v (None where not wanted)."""
    prob = pairwise_problem(u, v, pos_u, pos_v, p, flags)
    _dev_tensor(upstream, "upstream")
    if upstream.shape != (u.shape[0], u.shape[1], v.shape[1]) or not upstream.is_contiguous():
        raise ValueError("sot_b200: the upstream gradient must be a contiguous (B, P, R) tensor")
    alloc = torch.zeros_like if upstream.numel() == 0 else torch.empty_like  # (no pairs: nothing is launched)
    gu = alloc(u) if want_gu else None
    gv = alloc(v) if want_gv else None
    _launch("sot_pairwise_backward_device", u.device, ctypes.byref(prob), _ptr(upstream), _ptr(gu), _ptr(gv))
    return gu, gv


MAX_BARYCENTER_ENTRIES = 1 << 24  # K x n per barycenter (include/sot_b200.h)


def barycenter_problem(x, weights, pos, pos_out, flags: int) -> SotBarycenterProblem:
    """x: (N, K, n) contiguous CUDA float32; weights (K,) shared or (N, K); pos (n,), pos_out (M,) ascending."""
    for t, name in ((x, "x"), (weights, "weights"), (pos, "pos"), (pos_out, "out_pos")):
        _dev_tensor(t, name)
        if not t.is_contiguous():
            raise ValueError("sot_b200: tensors must be contiguous")
    if x.ndim != 3:
        raise ValueError(f"sot_b200: expected (N, K, n) rows, got {tuple(x.shape)}")
    N, K, n = x.shape
    if weights.shape not in ((K,), (N, K)):
        raise ValueError(f"sot_b200: weights of shape {tuple(weights.shape)} for {K} rows per barycenter")
    if pos.shape != (n,) or pos_out.ndim != 1:
        raise ValueError(f"sot_b200: positions of shape {tuple(pos.shape)} / {tuple(pos_out.shape)} for rows of {n} bins")
    if len({x.device, weights.device, pos.device, pos_out.device}) != 1:
        raise ValueError("sot_b200: all tensors must be on the same CUDA device")
    return SotBarycenterProblem(N, K, n, pos_out.shape[0], x.data_ptr(), weights.data_ptr(),
                                0 if weights.ndim == 1 else K, pos.data_ptr(), pos_out.data_ptr(), int(flags))


def barycenter(x, weights, pos, pos_out, flags) -> torch.Tensor:
    """(N, M) float32: the W2 barycenter of each x[b] as mass per point of `pos_out`."""
    prob = barycenter_problem(x, weights, pos, pos_out, flags)
    out = torch.empty(x.shape[0], pos_out.shape[0], dtype=torch.float32, device=x.device)
    _launch("sot_barycenter_device", x.device, ctypes.byref(prob), _ptr(out))
    return out


def barycenter_backward(x, weights, pos, pos_out, flags, upstream) -> torch.Tensor:
    """Gradient of sum_{b,m} upstream[b, m] * out[b, m] w.r.t. x, (N, K, n)."""
    prob = barycenter_problem(x, weights, pos, pos_out, flags)
    _dev_tensor(upstream, "upstream")
    if upstream.shape != (x.shape[0], pos_out.shape[0]) or not upstream.is_contiguous():
        raise ValueError("sot_b200: the upstream gradient must be a contiguous (N, M) tensor")
    grad = torch.empty_like(x)
    _launch("sot_barycenter_backward_device", x.device, ctypes.byref(prob), _ptr(upstream), _ptr(grad))
    return grad


def loss_from_cdf(cu, cv, pos_u, pos_v, p, flags, want_grads=True):
    """Parity harness: per-frame loss and dL/dcu, dL/dcv from injected CDF rows."""
    prob = make_problem(cu, cv, pos_u, pos_v, p, flags)
    loss = torch.empty(cu.shape[0], dtype=torch.float32, device=cu.device)
    g_cu = torch.empty_like(cu) if want_grads else None
    g_cv = torch.empty_like(cv) if want_grads else None
    _launch("sot_loss_from_cdf_device", cu.device, ctypes.byref(prob), _ptr(loss), _ptr(g_cu), _ptr(g_cv))
    return loss, g_cu, g_cv


def quantile_lookup(qs, cws, xs) -> torch.Tensor:
    for t, name in ((qs, "qs"), (cws, "cws"), (xs, "xs")):
        _dev_tensor(t, name)
        if t.ndim != 2 or not t.is_contiguous():
            raise ValueError(f"sot_b200: `{name}` must be a contiguous 2-D tensor")
    if cws.shape != xs.shape or qs.shape[0] != cws.shape[0]:
        raise ValueError("sot_b200: quantile_function shape mismatch")
    out = torch.empty_like(qs)
    _launch("sot_quantile_lookup_device", qs.device, _ptr(qs), _ptr(cws), _ptr(xs), _ptr(out), qs.shape[0],
            qs.shape[1], cws.shape[1])
    return out


def loss_grad_host(u, v, pos_u, pos_v, p, flags, upstream=None, want_loss=True, want_gu=True, want_gv=True,
                   device=0, out=None):
    """Host-buffer entry point: CPU tensors in (ideally pinned), CPU tensors out; all copies and
    kernels happen inside the one C call.  `out` may carry preallocated (pinned) result tensors."""
    for t, name in ((u, "x"), (v, "y"), (pos_u, "x_pos"), (pos_v, "y_pos")):
        if t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous():
            raise ValueError(f"sot_b200: `{name}` must be a contiguous float32 CPU tensor for the host entry point")
    prob = _problem(u, v, pos_u, pos_v, p, flags)
    N = u.shape[0]
    out = out or {}
    loss = out.get("loss", torch.empty(N) if want_loss else None)
    gu = out.get("grad_u", torch.empty_like(u) if want_gu else None)
    gv = out.get("grad_v", torch.empty_like(v) if want_gv else None)
    _check(load().sot_loss_grad_host(ctypes.byref(prob), _ptr(upstream), _ptr(loss), _ptr(gu), _ptr(gv), int(device)))
    return loss, gu, gv


def set_tuning(threads_per_frame: int = 0, bins_per_thread: int = 0, chains_per_thread: int = 0):
    """Select a kernel configuration (benchmarks, tests); (0, 0, 0) restores the built-in choice and (-1, 0, 0)
    routes every real-row loss / gradient request through the split-frame path of long rows."""
    _check(load().sot_set_tuning(threads_per_frame, bins_per_thread, chains_per_thread))


def launch_count() -> int:
    return int(load().sot_launch_count())


def max_bins(with_grad: bool = True, shared_positions: bool = True) -> int:
    return int(load().sot_max_bins(int(with_grad), int(shared_positions)))


def _mss_check(zt, zv):
    for t, name in ((zt, "target spectrogram"), (zv, "spectrogram")):
        if not t.is_cuda:
            raise SotError(f"sot_b200: the {name} lives on {t.device}; the kernels are CUDA only "
                           "(no CPU fallback exists by design)")
        if t.dtype != torch.complex64:
            raise TypeError(f"sot_b200: the {name} must be complex64, got {t.dtype}")
    if zt.shape != zv.shape or zt.device != zv.device:
        raise ValueError(f"sot_b200: spectrogram shapes differ: {tuple(zt.shape)} vs {tuple(zv.shape)}")
    if zt.stride() != zv.stride():
        raise ValueError("sot_b200: the two spectrograms must have the same (dense) memory layout")


def mss_forward(zt, zv, mag_weight, logmag_weight, loss_type, post_scale, total=None):
    """total (1,) float64 += post_scale * sum_i [mag_w d(|zt|,|zv|) + logmag_w d(safe_log|zt|, safe_log|zv|)]."""
    _mss_check(zt, zv)
    if total is None:
        total = torch.zeros(1, dtype=torch.float64, device=zt.device)
    _launch("sot_mss_forward_device", zt.device, _ptr(zt), _ptr(zv), zt.numel(), float(mag_weight),
            float(logmag_weight), int(loss_type), float(post_scale), _ptr(total))
    return total


def mss_backward(zt, zv, mag_weight, logmag_weight, loss_type, post_scale, scale, want_t=True, want_v=True):
    """Complex gradients of scale * post_scale * S w.r.t. zt / zv (same layout as the inputs)."""
    _mss_check(zt, zv)
    _dev_tensor(scale, "scale")
    gt = torch.empty_like(zt) if want_t else None
    gv = torch.empty_like(zv) if want_v else None
    _launch("sot_mss_backward_device", zt.device, _ptr(zt), _ptr(zv), zt.numel(), float(mag_weight),
            float(logmag_weight), int(loss_type), float(post_scale), _ptr(scale), _ptr(gt), _ptr(gv))
    return gt, gv


def p2p_mailbox_doubles(world: int) -> int:
    return load().sot_p2p_mailbox_doubles(int(world))


def p2p_allreduce(values, out, mailbox_ptrs, rank: int, seq: int):
    """out[:] = sum over ranks of `values` (float64, <= 8 elements) through peer-mapped mailboxes."""
    if values.dtype != torch.float64 or out.dtype != torch.float64 or not values.is_cuda or not out.is_cuda:
        raise TypeError("sot_b200: p2p_allreduce works on CUDA float64 tensors")
    arr = mailbox_array(mailbox_ptrs)
    _launch("sot_p2p_allreduce_device", values.device, _ptr(values), _ptr(out), values.numel(), arr, len(arr),
            int(rank), int(seq))
    return out


def p2p_wait_mean(mailbox_ptrs, rank: int, seq, expected_count: float = 0.0, status_ptr: int = 0,
                  timeout_ms: int = 0, device=None, stream=None, out=None) -> torch.Tensor:
    """Collects call `seq` of every rank from this rank's mailbox (the stores were made by the last CTA of
    `mean_step(..., post=...)` on every rank) and returns the global mean, a 0-dim float32 tensor.  `stream`: a
    `torch.cuda.Stream` to launch on (default: the current one); `out`: where to write (default: a new tensor)."""
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if out is None:
        out = torch.empty((), dtype=torch.float32, device=dev)
    arr = mailbox_array(mailbox_ptrs)
    on_device = isinstance(seq, torch.Tensor)  # one-element int64 device tensor: the previous call number
    _launch("sot_p2p_wait_mean_device", dev, _ptr(out), float(expected_count),
            ctypes.c_void_p(status_ptr) if status_ptr else None, arr, len(arr), int(rank),
            0 if on_device else int(seq), _ptr(seq) if on_device else None, int(timeout_ms), stream=stream)
    return out


def p2p_global_mean(local_sum, local_count: float, mailbox_ptrs, rank: int, seq: int):
    """(mean, 1 / count) over all ranks as two (1,) float32 tensors from this rank's (1,) float64 sum and its count."""
    if local_sum.dtype != torch.float64 or not local_sum.is_cuda or local_sum.numel() != 1:
        raise TypeError("sot_b200: p2p_global_mean takes a (1,) CUDA float64 sum")
    out = torch.empty(2, dtype=torch.float32, device=local_sum.device)
    arr = mailbox_array(mailbox_ptrs)
    _launch("sot_p2p_global_mean_device", local_sum.device, _ptr(local_sum), float(local_count), _ptr(out),
            ctypes.c_void_p(out.data_ptr() + 4), arr, len(arr), int(rank), int(seq))
    return out[0:1], out[1:2]
