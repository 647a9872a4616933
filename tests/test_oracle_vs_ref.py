"""Pins the oracle port to the reference itself: every entry point of oracle/librrt_oracle.so against
oracle/_ref/libref_host.so (the reference's unmodified headers compiled for the host), bit for bit, on
fresh seeded inputs and at parameter sets the golden files do not cover.  Skipped where the reference
library was not built (it needs /root/reference at build time; the built .so travels with the snapshot)."""
import numpy as np
import pytest

from inputs import disk_points, noise_points, phase_space
from parity import CAMERAS


def same(a, b):
    return np.array_equal(np.asarray(a).view(np.uint8), np.asarray(b).view(np.uint8))


def test_defaults_match_reference_macros(ora, ref):
    assert bytes(ora.default_params()) == bytes(ref.default_params())      # include/config.h
    assert bytes(ora.default_effects()) == bytes(ref.default_effects())    # camera_settings.h


# the hole and disk of tests/test_gpu_params.py's big-hole and disk-past-escape regimes
BIG_HOLE = dict(event_horizon=20.0, isco_radius=22.0, disk_out=60.0, cloud_out=60.0)
DISK_PAST_ESCAPE = dict(disk_out=300.0)


@pytest.mark.parametrize("kw", [pytest.param(dict(spin_a=a), id=str(a)) for a in (0.0, 0.3, 0.99)] +
                         [pytest.param(dict(spin_a=0.99, **BIG_HOLE), id="big-hole"),
                          pytest.param(dict(spin_a=0.99, **DISK_PAST_ESCAPE), id="disk-past-escape")])
def test_functions(ora, ref, kw):
    q, v = phase_space(seed=7, n=4096)
    po, pr = ora.default_params(**kw), ref.default_params(**kw)
    assert same(ora.geodesic_acc(po, q, v), ref.geodesic_acc(pr, q, v))
    h = np.random.Generator(np.random.PCG64(3)).choice(np.float32([0.3, 0.03, 0.09, 0.15]), size=len(q))
    a, b = ora.rk4_step(po, q, v, h), ref.rk4_step(pr, q, v, h)
    assert same(a[0], b[0]) and same(a[1], b[1])
    a, b = ora.euler_step(po, q, v, h), ref.euler_step(pr, q, v, h)
    assert same(a[0], b[0]) and same(a[1], b[1])
    assert same(ora.redshift(po, q, v), ref.redshift(pr, q, v))


def test_noise_and_density(ora, ref):
    p = noise_points(seed=8)
    assert same(ora.hash31(p), ref.hash31(p)) and same(ora.noise3d(p), ref.noise3d(p))
    for o in (1, 2, 5, 7):
        assert same(ora.fbm(p, o), ref.fbm(p, o))
    d = disk_points(seed=9)
    for prm_kw in ({}, {"isco_radius": 6.0, "disk_out": 30.0, "disk_h": 1.2, "cloud_h": 0.9}):
        po, pr = ora.default_params(**prm_kw), ref.default_params(**prm_kw)
        for t in (0.0, 3.7):
            assert same(ora.disk_density(po, d, t), ref.disk_density(pr, d, t))
            assert same(ora.dust_density(po, d, t), ref.dust_density(pr, d, t))
        r = np.linspace(1, 50, 999).astype(np.float32)
        assert same(ora.disk_temperature(po, r), ref.disk_temperature(pr, r))


def test_camera_and_paths(ora, ref):
    rng = np.random.Generator(np.random.PCG64(11))
    for _ in range(200):
        pos, yaw, pitch = rng.uniform(-80, 80, 3), rng.uniform(-400, 400), rng.uniform(-89, 89)
        assert bytes(ora.camera_from(pos, yaw, pitch)) == bytes(ref.camera_from(pos, yaw, pitch))
    for pi in range(3):
        for t in rng.uniform(-2, 35, 300):
            a, pa = ora.path_state(pi, t)
            b, pb = ref.path_state(pi, t)
            assert bytes(a) == bytes(b) and same(pa, pb)


@pytest.mark.parametrize("cam", ["C0", "C3"])
@pytest.mark.parametrize("kw", [dict(spin_a=0.99, flags=3), dict(spin_a=0.0, flags=1),
                                dict(spin_a=0.6, flags=3, max_steps=600, step_size=0.25, cloud_h=3.0, event_horizon=1.5),
                                dict(spin_a=0.99, flags=3, **BIG_HOLE), dict(spin_a=0.99, flags=3, **DISK_PAST_ESCAPE)])
def test_frames(ora, ref, sky_small, cam, kw):
    for fxo, fxr in ((ora.default_effects(use_ca=1), ref.default_effects(use_ca=1)), (ora.effects_off(), ref.effects_off())):
        a = ora.render(ora.default_params(**kw), ora.camera_from(*CAMERAS[cam]), fxo, sky_small, 2.5, 80, 45)
        b = ref.render(ref.default_params(**kw), ref.camera_from(*CAMERAS[cam]), fxr, sky_small, 2.5, 80, 45)
        for k in ("rgba", "hdr", "dir", "emis", "pos", "vel", "cls", "steps"):
            assert same(getattr(a, k), getattr(b, k)), k
        assert a.counters == b.counters
