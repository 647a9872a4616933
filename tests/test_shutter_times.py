"""rrt_shutter_times / shutter_times: the sub-frame times of a centred shutter.  Pure host code (no GPU needed); every
operation is one float32 operation, so numpy float32 reproduces the times bit for bit."""
import ctypes as C

import numpy as np
import pytest


def _numpy_times(t, shutter, fps, n):
    f = np.float32
    d = f(shutter) / f(fps)
    return np.array([f(t) + d * ((f(i) + f(0.5)) / f(n) - f(0.5)) for i in range(n)], np.float32)


@pytest.mark.parametrize("n", [1, 2, 3, 4, 7, 8, 16, 63, 64])
@pytest.mark.parametrize("t,shutter,fps", [(0.0, 0.5, 24.0), (1.0, 0.5, 24.0), (12.345, 1.0, 30.0), (123.5, 0.25, 60.0),
                                           (-3.0, 0.75, 23.976), (1e4, 0.5, 24.0)])
def test_bitwise_numpy_float32(built, t, shutter, fps, n):
    from relativisticraytracer_b200 import shutter_times
    got = np.array(shutter_times(t, shutter, fps, n), np.float32)
    want = _numpy_times(t, shutter, fps, n)
    assert got.shape == (n,)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (got, want)


@pytest.mark.parametrize("t", [0.0, 1.0, 0.1, 7.25, 123.456, -5.5, 3.4e38])
def test_n1_is_t_and_closed_shutter_is_t(built, t):
    from relativisticraytracer_b200 import shutter_times
    t32 = np.float32(t)
    assert np.array(shutter_times(t, 0.5, 24.0, 1), np.float32).view(np.uint32) == t32.view(np.uint32)
    for n in (1, 2, 5, 64):
        got = np.array(shutter_times(t, 0.0, 24.0, n), np.float32)
        assert (got.view(np.uint32) == t32.view(np.uint32)).all(), n


@pytest.mark.parametrize("n", [2, 3, 4, 5, 8, 13, 64])
def test_symmetric_about_t(built, n):
    """Centred: out[i] - t = -(out[n-1-i] - t), exactly at t = 0 when n is a power of two (every step is exact), to within
    an ulp of the times otherwise; the times increase and span shutter/fps * (1 - 1/n)."""
    from relativisticraytracer_b200 import shutter_times
    for t, shutter, fps in ((0.0, 0.5, 24.0), (5.0, 0.5, 24.0), (100.25, 1.0, 30.0)):
        got = np.array(shutter_times(t, shutter, fps, n), np.float64)
        off = got - np.float32(t)
        ulp = float(np.spacing(np.float32(abs(t) + shutter / fps)))
        assert np.all(np.abs(off + off[::-1]) <= 2 * ulp), (t, off)
        if t == 0.0 and n & (n - 1) == 0:
            assert np.array_equal(off, -off[::-1])
        assert np.all(np.diff(got) > 0)
        span = shutter / fps * (1 - 1 / n)
        assert abs((got[-1] - got[0]) - span) <= 4 * ulp


def test_argument_errors(built):
    import relativisticraytracer_b200 as rrt
    from relativisticraytracer_b200 import _capi
    lib = _capi.load()
    out = (C.c_float * 64)()
    for t, shutter, fps, n in ((1.0, -0.1, 24.0, 4), (1.0, 1.01, 24.0, 4), (1.0, float("nan"), 24.0, 4), (1.0, 0.5, 0.0, 4),
                               (1.0, 0.5, -24.0, 4), (1.0, 0.5, float("nan"), 4), (1.0, 0.5, 24.0, 0), (1.0, 0.5, 24.0, 65),
                               (1.0, 0.5, 24.0, -1)):
        assert lib.rrt_shutter_times(t, shutter, fps, n, out) == _capi.ERR_BAD_ARG, (shutter, fps, n)
        with pytest.raises(rrt.RrtError):
            rrt.shutter_times(t, shutter, fps, n)
    assert lib.rrt_shutter_times(1.0, 0.5, 24.0, 4, None) == _capi.ERR_BAD_ARG
    assert lib.rrt_shutter_times(1.0, 0.0, 24.0, 64, out) == 0 and lib.rrt_shutter_times(1.0, 1.0, 24.0, 1, out) == 0
