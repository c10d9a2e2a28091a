"""Stand-ins with the oracle's arithmetic for the CUDA entry points `sot_b200.losses` calls, so that the HOST logic
around the launches (canonicalisation, hoisted sort, autograd bridges, the position-gradient path) can be driven on
CPU tensors.  Test infrastructure only -- the product has no CPU path."""
import torch

from oracle import sot_oracle as O

SQUARE, CUT, LIMIT, RAW = 1, 2, 4, 8


def _weights(u, v, flags):
    if flags & RAW:
        return u, v
    return O.spectra_to_weights(u, v, bool(flags & SQUARE), bool(flags & CUT))


def _expand(pos, like):
    return pos.unsqueeze(0).expand_as(like) if pos.ndim == 1 else pos


def _rows(u, v, pos_u, pos_v, p, flags):
    wu, wv = _weights(u, v, flags)
    return O.w1d_rows(_expand(pos_u, u), _expand(pos_v, v), wu, wv, p=p, require_sort=False,
                      limit=bool(flags & LIMIT), stable=True)


def install(monkeypatch, capi, losses):
    def forward(u, v, pos_u, pos_v, p, flags):
        return _rows(u, v, pos_u, pos_v, p, flags).detach()

    def forward_backward(u, v, pos_u, pos_v, p, flags, upstream=None, want_loss=True, want_gu=True, want_gv=True):
        with torch.enable_grad():
            ur, vr = u.detach().clone().requires_grad_(True), v.detach().clone().requires_grad_(True)
            rows = _rows(ur, vr, pos_u, pos_v, p, flags)
            total = rows.sum() if upstream is None else (rows * upstream).sum()
            gu, gv = torch.autograd.grad(total, (ur, vr))
        return rows.detach(), (gu if want_gu else None), (gv if want_gv else None)

    def mean_step(u, v, pos_u, pos_v, p, flags, grad_scale, mean_scale, want_gu=True, want_gv=True, **kw):
        rows, gu, gv = forward_backward(u, v, pos_u, pos_v, p, flags)
        scale = grad_scale * (float(kw["grad_scale_device"]) if kw.get("grad_scale_device") is not None else 1.0)
        mean = (rows.sum() * mean_scale).float()
        return mean, None, (gu * scale if want_gu else None), (gv * scale if want_gv else None)

    def scale_inplace(a, b, scale):
        for t in (a, b):
            if t is not None:
                t.mul_(float(scale))

    def scale_rows(unit, scale):
        return unit * scale[:, None]

    def quantiles(u, v, pos_u, pos_v, flags, from_cdf=False, want_indices=False):
        wu, wv = _weights(u, v, flags)
        out = O.transport_plan(_expand(pos_u, u), _expand(pos_v, v), wu, wv, require_sort=False, stable=True)
        out = tuple(t.int() if i >= 5 else t for i, t in enumerate(out))
        return out if want_indices else out[:5]

    for name, fn in dict(forward=forward, forward_backward=forward_backward, mean_step=mean_step,
                         scale_inplace=scale_inplace, scale_rows=scale_rows, quantiles=quantiles).items():
        monkeypatch.setattr(capi, name, fn)

    allow_cpu_rows(monkeypatch, losses)
    monkeypatch.setattr(losses, "_uniform_grid", lambda *a, **k: False)


def allow_cpu_rows(monkeypatch, losses):
    """Lets the host prologue of `losses` take CPU tensors: its CUDA-only check becomes a no-op."""
    monkeypatch.setattr(losses, "_require_cuda", lambda t, name: None)
