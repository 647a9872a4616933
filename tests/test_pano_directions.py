"""rrt_pano_directions / pano_directions: the direction of every pixel of an equirectangular panorama (render_pano).  Pure
host code (no GPU needed).  Longitude and latitude are evaluated in double with exactly opposite angles for mirrored
columns and rows, their cosines and sines rounded to float32 once, and the direction is built from them with one float32
operation per step, so the symmetries below hold bit for bit."""
import numpy as np
import pytest

CAMS = [((0.0, 10.0, -60.0), 0.0, -10.0), ((25.0, 3.0, -40.0), -32.0, -4.0), ((-7.5, 1.0, 35.0), 171.0, 2.5),
        ((0.0, -20.0, 0.0), 0.0, 89.0)]
SIZES = [(48, 24), (37, 19), (1, 1), (2, 1), (7, 3), (4096, 2048)]


def _axis_camera():
    """forward = +z, right = +x, up = +y: each term of d lands in its own component."""
    from relativisticraytracer_b200 import Camera
    c = Camera()
    c.pos[:] = [1.0, 2.0, 3.0]
    c.forward[:] = [0.0, 0.0, 1.0]
    c.right[:] = [1.0, 0.0, 0.0]
    c.up[:] = [0.0, 1.0, 0.0]
    return c


@pytest.mark.parametrize("cam", range(len(CAMS)))
@pytest.mark.parametrize("w,h", [(1, 1), (37, 19), (5, 3), (1001, 999)])
def test_centre_of_odd_panorama_is_forward(built, cam, w, h):
    from relativisticraytracer_b200 import camera_state_from, pano_directions
    c = camera_state_from(*CAMS[cam])
    d = pano_directions(c, w, h)
    assert d.shape == (h, w, 3) and d.dtype == np.float32
    assert np.array_equal(d[h // 2, w // 2], np.array(c.forward, np.float32))


@pytest.mark.parametrize("w,h", SIZES)
def test_mirrored_rows_flip_up_and_mirrored_columns_flip_right(built, w, h):
    from relativisticraytracer_b200 import pano_directions
    d = pano_directions(_axis_camera(), w, h)          # d = (b, sin phi, a): right, up and forward terms
    flip_rows, flip_cols = d[::-1], d[:, ::-1]
    assert np.array_equal(flip_rows[..., 1], -d[..., 1]) and np.array_equal(flip_rows[..., [0, 2]], d[..., [0, 2]])
    assert np.array_equal(flip_cols[..., 0], -d[..., 0]) and np.array_equal(flip_cols[..., [1, 2]], d[..., [1, 2]])


@pytest.mark.parametrize("cam", range(len(CAMS)))
@pytest.mark.parametrize("w,h", SIZES)
def test_mirror_symmetry_on_survey_cameras(built, cam, w, h):
    """Any camera: d is (a*forward + b*right) + sin(phi)*up in float32 from the axis camera's exact a, b and sin(phi), and
    the mirrored row (column) is the same sum with the up (right) term's factor negated."""
    from relativisticraytracer_b200 import camera_state_from, pano_directions
    c = camera_state_from(*CAMS[cam])
    d = pano_directions(c, w, h)
    ax = pano_directions(_axis_camera(), w, h)         # (b, sin phi, a) of every pixel, exact
    f = np.float32
    F, R, U = (np.array(v, f) for v in (c.forward, c.right, c.up))
    b, s, a = ax[..., 0:1], ax[..., 1:2], ax[..., 2:3]
    want = (a * F + b * R) + s * U                     # float32, one rounding per operation, the rrt.h order
    assert np.array_equal(d, want)
    assert np.array_equal(d[::-1], (a * F + b * R) + (-s) * U)
    assert np.array_equal(d[:, ::-1], (a * F + (-b) * R) + s * U)


@pytest.mark.parametrize("cam", range(len(CAMS)))
@pytest.mark.parametrize("w,h", SIZES + [(1001, 999)])
def test_within_two_ulp_of_float64(built, cam, w, h):
    """Every vector within 2 float32 ulp (2 FLT_EPSILON of its length) of the float64 evaluation of the projection."""
    from relativisticraytracer_b200 import camera_state_from, pano_directions
    c = camera_state_from(*CAMS[cam])
    d = pano_directions(c, w, h).astype(np.float64)
    lam = 2 * np.pi * ((np.arange(w) + 0.5) / w - 0.5)
    phi = np.pi * ((np.arange(h) + 0.5) / h - 0.5)
    F, R, U = (np.array(v, np.float64) for v in (c.forward, c.right, c.up))
    cp, sp = np.cos(phi)[:, None, None], np.sin(phi)[:, None, None]
    want = (cp * np.cos(lam)[None, :, None]) * F + (cp * np.sin(lam)[None, :, None]) * R + sp * U
    err = np.abs(d - want).max(-1) / (np.finfo(np.float32).eps * np.linalg.norm(want, axis=-1))
    assert err.max() <= 2.0, err.max()


def test_projection_orientation(built):
    """Column 0 looks backwards (longitude -pi), the middle column forward, column 3w/4 right; the first row is near the
    nadir and the last near the zenith."""
    from relativisticraytracer_b200 import pano_directions
    w, h = 64, 32
    d = pano_directions(_axis_camera(), w, h)
    assert d[h // 2, 0, 2] < -0.99 and d[h // 2, 3 * w // 4, 0] > 0.99 and d[h // 2, w // 4, 0] < -0.99
    assert d[0, :, 1].max() < -0.99 and d[-1, :, 1].min() > 0.99


def test_bad_arguments_are_refused(built):
    import ctypes as C
    from relativisticraytracer_b200 import RrtError, _capi, camera_state_from, pano_directions
    c = camera_state_from(*CAMS[0])
    for w, h in [(0, 4), (4, 0), (-1, 4), (4, -3)]:
        with pytest.raises(RrtError):
            pano_directions(c, w, h)
    lib = _capi.load()
    buf = (C.c_float * 12)()
    assert lib.rrt_pano_directions(None, 2, 2, buf) == _capi.ERR_BAD_ARG
    assert lib.rrt_pano_directions(C.byref(c), 2, 2, None) == _capi.ERR_BAD_ARG
    assert lib.rrt_pano_directions(C.byref(c), 2, 2, buf) == 0


@pytest.mark.parametrize("kw", [dict(projection="fisheye"), dict(projection="equirect", aperture=0.5, focus=60.0),
                                dict(projection="equirect", samples=4, shutter=0.5), dict(projection="")])
def test_path_sequence_argument_errors(built, kw):
    from relativisticraytracer_b200.parallel import PathSequence
    with pytest.raises(ValueError):
        PathSequence(None, 64, 32, **kw)
