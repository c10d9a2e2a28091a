"""Row-length limits of the C ABI (no GPU needed): refusals happen before anything is launched."""
import ctypes


def test_row_length_limits_are_checked_before_any_launch():
    from sot_b200 import _capi
    lib = _capi.load()
    before = _capi.launch_count()
    assert lib.sot_max_bins(1, 1) == 2 ** 24 - 1
    # longer than the split-frame path takes
    prob = _capi.SotProblem(4, 2 ** 24, 9, 16, 16, 16, 16, 0, 0, 2.0, 0)
    assert lib.sot_forward_device(ctypes.byref(prob), ctypes.c_void_p(16), None) == -2
    assert b"16777215" in lib.sot_last_error()
    # shared memory still bounds the quantile taps: 8449-bin rows are refused there
    prob = _capi.SotProblem(4, 8449, 8449, 16, 16, 16, 16, 0, 0, 2.0, 0)
    assert lib.sot_quantiles_device(ctypes.byref(prob), *([None] * 7), None) == -2
    # the split-frame path takes rows only in memory the device can reach
    prob = _capi.SotProblem(4, 9000, 9000, 16, 16, 16, 16, 0, 0, 2.0, 0)
    assert lib.sot_forward_device(ctypes.byref(prob), ctypes.c_void_p(16), None) == -2
    assert b"device-accessible" in lib.sot_last_error()
    assert _capi.launch_count() == before
