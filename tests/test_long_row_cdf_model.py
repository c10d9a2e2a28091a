"""CPU model of the split-frame path's CDF stage (csrc/sot_long.cu, pass 1) on rows longer than shared memory holds.

Thread t of a tile owns E = 16 consecutive bins; its local prefixes are packed-fp32 sums (x^2 fused into the add), its
offset is the fp64 sum of the local totals before it -- the in-tile scan plus the carry of the tiles before -- and an
entry is fl32(head + fl32(prefix * inv32 + tail)), (head, tail) the fp32 split of offset * inv64, capped by the next
thread's head (for a tile's last thread: the next tile's first head).  The row end is fl32(mass * inv64).  Checked at
every tile border and over the row: non-decreasing, row end exact, and within 4 ulp (harmonic spectra at n_fft 32768)
or 10 ulp (log-normal magnitudes over 12 decades, 65 536 bins) of the float64 CDF -- the CDF gate of DESIGN §2.
"""
import numpy as np
import pytest

F32 = np.float32
TPB, E = 256, 16
TILE = TPB * E
EPS = 1e-7


def tiled_cdf(x, square=True):
    x64 = np.asarray(x, np.float32).astype(np.float64)
    n = len(x64)
    threads = -(-n // E)
    xs = np.zeros(threads * E)
    xs[:n] = x64
    xs = xs.reshape(threads, E)
    local = np.zeros((threads, E), np.float32)
    acc = np.zeros(threads, np.float32)
    for c in range(E):  # one rounding per fused add (x*x is exact in float64)
        acc = (xs[:, c] * xs[:, c] + acc.astype(np.float64) if square else xs[:, c] + acc.astype(np.float64)).astype(F32)
        local[:, c] = acc
    totals = local[:, -1].astype(np.float64)
    # exclusive fp64 offsets: in-tile prefix plus the carry of the tiles before (added in that order)
    offsets = np.zeros(threads + 1)
    carry = 0.0
    for t0 in range(0, threads, TPB):
        tt = totals[t0:t0 + TPB]
        excl = np.concatenate(([0.0], np.cumsum(tt)))
        offsets[t0:t0 + len(tt) + 1] = carry + excl
        carry = carry + excl[-1]
    mass = carry
    m32 = F32(mass)
    inv64 = 1.0 / np.float64(m32 if m32 > EPS else F32(EPS))
    inv32 = F32(inv64)
    base = offsets[:-1] * inv64
    head = base.astype(F32)
    tail = (base - head.astype(np.float64)).astype(F32)
    cap = (offsets[1:] * inv64).astype(F32)
    inner = (local.astype(np.float64) * np.float64(inv32) + tail[:, None].astype(np.float64)).astype(F32)
    out = np.minimum((head[:, None].astype(np.float64) + inner.astype(np.float64)).astype(F32), cap[:, None])
    out = out.reshape(-1)[:n].copy()
    out[-1] = max(F32(mass * inv64), out[-2])
    return out, mass, inv64


def _ulps(a, b):
    return np.abs(a.view(np.int32).astype(np.int64) - b.view(np.int32).astype(np.int64))


def _check(rows, square, max_ulp):
    worst = 0
    for x in rows:
        cdf, mass, inv64 = tiled_cdf(x, square)
        w = np.asarray(x, np.float32).astype(np.float64)
        ref = (np.cumsum(w * w if square else w) * inv64).astype(F32)
        assert (np.diff(cdf) >= 0).all(), "non-decreasing"
        borders = np.arange(TILE, len(x), TILE)
        assert (cdf[borders] >= cdf[borders - 1]).all(), "non-decreasing across tile borders"
        assert cdf[-1] == F32(mass * inv64), "row end exact"
        worst = max(worst, int(_ulps(cdf, ref).max()))
    assert worst <= max_ulp, worst
    return worst


def test_harmonic_spectra_at_n_fft_32768():
    from sot_b200 import synthetic as S
    x, _ = S.sot_batch(1, 32768, seed=11)  # 16 frames x 16385 bins
    rows = x.reshape(-1, x.shape[-1]).numpy()
    assert rows.shape[1] == 16385
    _check(rows, square=True, max_ulp=4)


@pytest.mark.parametrize("square", [False, True])
def test_log_normal_magnitudes_over_twelve_decades(square):
    rng = np.random.default_rng(12)
    rows = (10.0 ** np.clip(rng.normal(0.0, 2.0, (4, 65536)), -6, 6)).astype(np.float32)
    _check(rows, square=square, max_ulp=10)
