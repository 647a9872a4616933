"""rrt_lens_cameras / lens_cameras: the camera table of a thin lens.  Pure host code (no GPU needed).  The lens points are the
concentric map of the stratified cell centres evaluated in double and rounded once; the cameras are built from them with
one float32 operation per step, so numpy float32 reproduces every camera bit for bit."""
import ctypes as C
import math

import numpy as np
import pytest

CAMS = [((0.0, 10.0, -60.0), 0.0, -10.0), ((25.0, 3.0, -40.0), -32.0, -4.0), ((-7.5, 1.0, 35.0), 171.0, 2.5),
        ((0.0, -20.0, 0.0), 0.0, 89.0)]


def _disk(ss):
    """(x, y) on the unit disk of every lens cell (i, j), k = j*ss + i, in float64: Shirley & Chiu's concentric map of the
    cell centre (a, b) = (2(i+0.5)/ss - 1, 2(j+0.5)/ss - 1)."""
    out = []
    for j in range(ss):
        for i in range(ss):
            a, b = 2 * (i + 0.5) / ss - 1, 2 * (j + 0.5) / ss - 1
            if a == 0 and b == 0:
                out.append((0.0, 0.0))
            elif abs(a) > abs(b):
                phi = math.pi / 4 * (b / a)
                out.append((a * math.cos(phi), a * math.sin(phi)))
            else:   # phi = pi/2 - pi/4 (a/b), written with cos(phi) = sin(pi/4 (a/b)) so that a = 0 gives x = 0 exactly
                t = math.pi / 4 * (a / b)
                out.append((b * math.sin(t), b * math.cos(t)))
    return np.array(out, np.float64)


def _arr(cam):
    return np.array([list(cam.pos), list(cam.forward), list(cam.right), list(cam.up)], np.float32)


def _want(cam, aperture, focus, ss):
    """numpy float32 cameras in the order rrt.h states, from the float64 lens points rounded to float32 once."""
    f = np.float32
    c = _arr(cam)
    pos, fwd, right, up = c
    out = []
    for k, (x, y) in enumerate(_disk(ss)):
        if aperture == 0 or (x == 0 and y == 0):
            out.append(c.copy())
            continue
        ox, oy = f(float(f(aperture)) * x), f(float(f(aperture)) * y)
        o = (right * ox) + (up * oy)
        out.append(np.array([pos + o, fwd - o / f(focus), right, up], np.float32))
    return out


@pytest.mark.parametrize("cam", range(len(CAMS)))
@pytest.mark.parametrize("ss", [1, 2, 3, 4, 5, 8])
@pytest.mark.parametrize("aperture,focus", [(0.5, 60.0), (0.1, 35.0), (2.0, 12.5), (1e-3, 1000.0)])
def test_bitwise_numpy_float32(built, cam, ss, aperture, focus):
    from relativisticraytracer_b200 import camera_state_from, lens_cameras
    c = camera_state_from(*CAMS[cam])
    got = lens_cameras(c, aperture, focus, ss)
    assert len(got) == ss * ss
    for k, (g, w) in enumerate(zip(got, _want(c, aperture, focus, ss))):
        assert np.array_equal(_arr(g).view(np.uint32), w.view(np.uint32)), (k, _arr(g), w)


@pytest.mark.parametrize("ss", [1, 2, 3, 4, 7, 8])
def test_aperture_zero_and_ss1_are_copies(built, ss):
    """Exact copies, -0 fields included; so is the centre lens point of an odd ss."""
    from relativisticraytracer_b200 import Camera, lens_cameras
    from relativisticraytracer_b200.renderer import camera_state_from
    cams = [camera_state_from(*c) for c in CAMS]
    neg = Camera()
    neg.pos[:] = [-0.0, 3.0, -50.0]
    neg.forward[:] = [-0.0, -0.0, 1.0]
    neg.right[:] = [1.0, -0.0, 0.0]
    neg.up[:] = [0.0, 1.0, -0.0]
    for c in cams + [neg]:
        assert all(bytes(x) == bytes(c) for x in lens_cameras(c, 0.0, 60.0, ss))
        assert bytes(lens_cameras(c, 0.5, 60.0, 1)[0]) == bytes(c)
        if ss % 2:
            assert bytes(lens_cameras(c, 0.5, 60.0, ss)[(ss * ss) // 2]) == bytes(c)


@pytest.mark.parametrize("ss", [2, 3, 4, 6, 8])
def test_lens_points(built, ss):
    """The offsets lie in the right / up plane within the aperture, one per stratified cell in k = j*ss + i order, at the
    float64 concentric map's points.  (That the library's lens points are those points rounded once, within 0.5 ulp, is
    what test_bitwise_numpy_float32 checks: it builds the expected cameras from them.)"""
    from relativisticraytracer_b200 import camera_state_from, lens_cameras
    aperture = 0.5
    for cc in CAMS:
        c = camera_state_from(*cc)
        pos, fwd, right, up = _arr(c).astype(np.float64)
        got = lens_cameras(c, aperture, 60.0, ss)
        disk = _disk(ss) * np.float64(np.float32(aperture))
        for k, g in enumerate(got):
            d = _arr(g)[0].astype(np.float64) - pos
            tol = 4 * float(np.spacing(np.float32(np.abs(pos).max() + aperture)))
            assert abs(d @ fwd) <= tol                                       # in the right / up plane
            assert np.linalg.norm(d) <= aperture + tol                       # inside the lens
            ox, oy = d @ right, d @ up
            assert abs(ox - disk[k, 0]) <= tol and abs(oy - disk[k, 1]) <= tol, (k, ox, oy, disk[k])
            i, j = k % ss, k // ss
            # the concentric map keeps each cell's quadrant / wedge: sign of x from i, of y from j
            if 2 * i + 1 != ss:
                assert np.sign(disk[k, 0]) == np.sign(2 * i + 1 - ss)
            if 2 * j + 1 != ss:
                assert np.sign(disk[k, 1]) == np.sign(2 * j + 1 - ss)
        pts = np.array([[ox, oy] for ox, oy in
                        (((_arr(g)[0].astype(np.float64) - pos) @ right, (_arr(g)[0].astype(np.float64) - pos) @ up) for g in got)])
        assert len({(round(x, 9), round(y, 9)) for x, y in pts}) == ss * ss   # one distinct point per cell


@pytest.mark.parametrize("ss", [2, 4, 8])
@pytest.mark.parametrize("focus", [12.5, 60.0, 400.0])
def test_focal_plane_is_shared(built, ss, focus):
    """Every camera's ray for image-plane coordinate (u, v) passes through pos + focus * (F + R u + U v)."""
    from relativisticraytracer_b200 import camera_state_from, lens_cameras
    for cc in CAMS:
        c = camera_state_from(*cc)
        pos, fwd, right, up = _arr(c).astype(np.float64)
        for g in lens_cameras(c, 0.5, focus, ss):
            p2, f2, r2, u2 = _arr(g).astype(np.float64)
            assert np.array_equal(r2, right) and np.array_equal(u2, up)
            for u, v in ((0.0, 0.0), (-1.3, 0.7), (0.9, -1.0), (1.7, 1.0)):
                a = p2 + focus * (f2 + r2 * u + u2 * v)
                b = pos + focus * (fwd + right * u + up * v)
                assert np.abs(a - b).max() <= 1e-6 * (np.abs(b).max() + focus), (u, v, a, b)


def test_argument_errors(built):
    import relativisticraytracer_b200 as rrt
    from relativisticraytracer_b200 import _capi
    lib = _capi.load()
    cam = rrt.camera_state_from(*CAMS[0])
    out = (rrt.Camera * 64)()
    inf, nan = float("inf"), float("nan")
    for aperture, focus, ss in ((-0.1, 60.0, 2), (nan, 60.0, 2), (inf, 60.0, 2), (0.5, 0.0, 2), (0.5, -1.0, 2), (0.5, nan, 2),
                                (0.5, inf, 2), (0.5, 60.0, 0), (0.5, 60.0, 9), (0.5, 60.0, -1), (-0.0 - 1e-30, 60.0, 2)):
        assert lib.rrt_lens_cameras(C.byref(cam), aperture, focus, ss, out) == _capi.ERR_BAD_ARG, (aperture, focus, ss)
        with pytest.raises(rrt.RrtError):
            rrt.lens_cameras(cam, aperture, focus, ss)
    assert lib.rrt_lens_cameras(None, 0.5, 60.0, 2, out) == _capi.ERR_BAD_ARG
    assert lib.rrt_lens_cameras(C.byref(cam), 0.5, 60.0, 2, None) == _capi.ERR_BAD_ARG
    assert lib.rrt_lens_cameras(C.byref(cam), 0.0, 60.0, 8, out) == 0 and lib.rrt_lens_cameras(C.byref(cam), -0.0, 1e-30, 1, out) == 0
