"""The CDF-stage model (tests/kernel_model.py) as the split-frame path runs it (csrc/sot_long.cu, pass 1), on rows
longer than shared memory holds.

Thread t of a tile owns E = 16 consecutive bins; its local prefixes are packed-fp32 sums (x^2 fused into the add), its
offset is the fp64 sum of the local totals before it -- the in-tile scan plus the carry of the tiles before -- and an
entry is fl32(head + fl32(prefix * inv32 + tail)), (head, tail) the fp32 split of offset * inv64, capped by the next
thread's head (for a tile's last thread: the next tile's first head).  The row end is fl32(mass * inv64).  Checked at
every tile border and over the row: non-decreasing, row end exact, and within 4 ulp (harmonic spectra at n_fft 32768)
or 10 ulp (log-normal magnitudes over 12 decades, 65 536 bins) of the float64 CDF -- the CDF gate of DESIGN §2.
"""
import numpy as np
import pytest

from tests import kernel_model as KM

F32 = np.float32
TPB, E = 256, 16
TILE = TPB * E


def _ulps(a, b):
    return np.abs(a.view(np.int32).astype(np.int64) - b.view(np.int32).astype(np.int64))


def _check(rows, square, max_ulp):
    worst = 0
    for x in rows:
        cdf, inv64, mass = KM.cdf_stage_model(x, -(-len(x) // E), E, square=square, tile=TPB, exact_end=True,
                                              return_inv=True)
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
