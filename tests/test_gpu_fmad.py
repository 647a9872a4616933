"""The RRT_FLAG_FMAD rounding contract: the arithmetic of the reference's OWN CUDA build (nvcc default
-fmad=true), fused operation by operation like nvcc 12.9 fuses the reference's sources on sm_100a.

Two witnesses:
* the CPU twin -- the oracle port with ORA_FLAG_FMAD, the same schedule written with fmaf(): everything that
  only involves + - * / sqrt and FMA must agree bit for bit (integrator, RHS, noise, whole trajectories,
  termination class); emission within north_star's 1e-3;
* the reference's own kernel -- oracle/_ref/libref_cuda.so is src/raymarcher.cu, unmodified, built with nvcc's
  defaults: on every pixel that never touched a medium (pure geodesic + sky lookup + effects + tonemap) our
  uchar4 output must be byte-identical to it.
"""
import numpy as np
import pytest

from inputs import noise_points, phase_space
from parity import CAMERAS, DIR_TOL_RAD, RGB_TOL_REL, assert_reference_digests, census
from test_gpu_frames import render_pair
from test_gpu_probes import bits_equal

pytestmark = pytest.mark.gpu

FMAD = 4   # RRT_FLAG_FMAD == ORA_FLAG_FMAD


@pytest.mark.parametrize("spin", [0.0, 0.99, 0.5])
def test_fmad_rhs_and_integrators_match_twin(gpu, ora, spin):
    import relativisticraytracer_b200 as rrt
    q, v = phase_space(seed=21)
    pg, po = rrt.default_params(spin_a=spin, flags=3 | FMAD), ora.default_params(spin_a=spin, flags=3 | FMAD)
    assert bits_equal(gpu.geodesic_acc(pg, q, v), ora.geodesic_acc(po, q, v))
    for h in (np.float32(0.3), np.float32(0.3) * np.float32(0.1), np.float32(0.3) * np.float32(0.3)):
        p1, v1 = gpu.rk4_step(pg, q, v, h)
        p2, v2 = ora.rk4_step(po, q, v, h)
        assert bits_equal(p1, p2) and bits_equal(v1, v2)
        p1, v1 = gpu.euler_step(pg, q, v, h)
        p2, v2 = ora.euler_step(po, q, v, h)
        assert bits_equal(p1, p2) and bits_equal(v1, v2)
    # and the fused schedule really is a different rounding from the strict one
    ps, _ = gpu.rk4_step(rrt.default_params(spin_a=spin, flags=3), q, v, np.float32(0.3))
    pf, _ = gpu.rk4_step(pg, q, v, np.float32(0.3))
    assert not np.array_equal(ps, pf)


def test_fmad_trajectory_matches_twin(gpu, ora):
    import relativisticraytracer_b200 as rrt
    q, v = phase_space(seed=22, n=512)
    pg, po = rrt.default_params(spin_a=0.99, flags=3 | FMAD), ora.default_params(spin_a=0.99, flags=3 | FMAD)
    p1, v1, p2, v2 = q.copy(), v.copy(), q.copy(), v.copy()
    for _ in range(200):
        p1, v1 = gpu.rk4_step(pg, p1, v1, np.float32(0.03))
        p2, v2 = ora.rk4_step(po, p2, v2, np.float32(0.03))
    assert bits_equal(p1, p2) and bits_equal(v1, v2)


def test_fmad_noise_matches_twin(gpu, ora):
    pts = noise_points(seed=23)
    gpu.set_probe_contract(True)
    ora.set_probe_contract(True)
    try:
        assert bits_equal(gpu.hash31(pts), ora.hash31(pts))
        assert bits_equal(gpu.noise3d(pts), ora.noise3d(pts))
        for octaves in (2, 5):
            assert bits_equal(gpu.fbm(pts, octaves), ora.fbm(pts, octaves))
        fused = gpu.noise3d(pts)
        gpu.set_probe_contract(False)
        strict = gpu.noise3d(pts)
    finally:
        gpu.set_probe_contract(True)     # the library's default
        ora.set_probe_contract(False)    # the oracle port's default
    assert not np.array_equal(fused, strict)   # strict noise differs in some last bits


@pytest.mark.parametrize("cam", ["C0", "C1", "C2", "C3"])
@pytest.mark.parametrize("spin", [0.0, 0.99])
def test_fmad_frames_match_twin(gpu, ora, sky_smooth, cam, spin):
    f, g = render_pair(gpu, ora, sky_smooth, cam, spin, 3 | FMAD, 160, 90)
    for k in ("steps", "pos", "vel", "dir"):
        assert np.array_equal(g[k], getattr(f, k)), k
    c = census(f, g)
    assert c["class_flips"] == 0, c
    assert c["dir_max_rad"] <= DIR_TOL_RAD
    assert g["counters"]["rk4_steps"] == f.counters["rk4_steps"]
    assert g["counters"]["disk_evals"] == f.counters["disk_evals"] and g["counters"]["dust_evals"] == f.counters["dust_evals"]
    assert c["rgb_frac_over_tol"] == 0.0, c
    e_rel = np.abs(g["emis"][..., :3].astype(np.float64) - f.emis[..., :3]) / np.maximum(np.abs(f.emis[..., :3]), 1e-3)
    assert e_rel.max() < RGB_TOL_REL
    assert np.abs(g["rgba"].astype(int) - f.rgba.astype(int)).max() <= 1


def test_fmad_geodesic_only_and_effects(gpu, ora, sky_smooth):
    f, g = render_pair(gpu, ora, sky_smooth, "C1", 0.99, FMAD, 200, 117, fx="default")
    for k in ("cls", "steps", "pos", "vel", "dir"):
        assert np.array_equal(g[k], getattr(f, k)), k
    assert g["counters"] == f.counters
    d = np.abs(g["rgba"].astype(int) - f.rgba.astype(int))
    assert d.max() <= 1 and np.mean(d > 0) < 0.02


def fmad_bytes_case(gpu, sky_np, cam, spin, w, h):
    """our uchar4 frame with the reference's default effects, and the class plane row-flipped like the frame"""
    import relativisticraytracer_b200 as rrt
    import torch
    sky = gpu.create_sky(sky_np)
    planes = gpu.alloc_planes(w, h, names=("cls",))
    out = gpu.render(rrt.default_params(spin_a=spin, flags=3 | FMAD), rrt.camera_state_from(*CAMERAS[cam]),
                     rrt.default_effects(), sky, 1.0, w, h, planes=planes)
    torch.cuda.synchronize()
    ours = out.cpu().numpy()
    cls = np.ascontiguousarray(planes["cls"].cpu().numpy()[::-1])   # planes are [y][x]; the uchar4 frame is row-flipped (:168)
    sky.close()
    return f"fmad_bytes/{cam}/{spin}/{w}x{h}", {"rgba": ours, "cls": cls}


def fmad_bytes_exact(rgba, untouched):
    """the exact part of the comparison: the 8-bit frame on every pixel whose ray touched no medium"""
    return {"rgba_untouched": np.ascontiguousarray(rgba[untouched], dtype=np.uint8)}


def _ours_vs(gpu, sky_np, ref_rgba, cam, spin, w, h):
    import relativisticraytracer_b200 as rrt
    _, g = fmad_bytes_case(gpu, sky_np, cam, spin, w, h)
    untouched = (g["cls"] & rrt.CLSF_TOUCHED) == 0
    diff = np.abs(g["rgba"].astype(int) - ref_rgba.astype(int)).max(axis=-1)
    return untouched, diff


@pytest.mark.parametrize("cam", ["C0", "C1", "C2", "C3"])
@pytest.mark.parametrize("spin", [0.0, 0.99])
def test_fmad_bytes_equal_reference_cuda_kernel(gpu, sky_small, cam, spin):
    """Against the reference's own CUDA kernel (unmodified src/raymarcher.cu, nvcc defaults, same GPU): every
    pixel whose ray never touched a medium is byte-identical; of the pixels that did (there the density code is
    left to nvcc's own fusion in both builds, which need not coincide) at most a handful differ, by one count.
    Measured at 960x540 with the 4096x2048 star-field sky, 8 camera/spin cases (tests/tools/refcuda_census.py):
    0 of 3.66 M untouched and 2 of 0.49 M touched pixels differ.  Where that build is absent, the untouched pixels are
    checked against committed digests of the reference kernel's bytes (tests/parity.py)."""
    import relativisticraytracer_b200 as rrt
    from oracle import RefCuda
    w, h = 320, 180
    if not RefCuda.available():
        key, g = fmad_bytes_case(gpu, sky_small, cam, spin, w, h)
        untouched = (g["cls"] & rrt.CLSF_TOUCHED) == 0
        assert untouched.mean() > 0.3
        assert_reference_digests(key, fmad_bytes_exact(g["rgba"], untouched))
        return
    ref_rgba, _, _ = RefCuda().render(spin, rrt.camera_state_from(*CAMERAS[cam]), rrt.default_effects(), sky_small, 1.0, w, h)
    untouched, diff = _ours_vs(gpu, sky_small, ref_rgba, cam, spin, w, h)
    assert untouched.mean() > 0.3
    assert diff[untouched].max() == 0, f"{int((diff[untouched] > 0).sum())} untouched pixels differ from the reference kernel"
    assert diff[~untouched].max() <= 1 and (diff[~untouched] > 0).sum() <= 3, \
        f"{int((diff[~untouched] > 0).sum())} touched pixels differ, by up to {diff[~untouched].max()} counts"


@pytest.mark.parametrize("cam", ["C0", "C1", "C2", "C3"])
@pytest.mark.parametrize("tag,spin", [("a000", 0.0), ("a099", 0.99)])
def test_fmad_bytes_equal_committed_reference_cuda_frames(gpu, sky_small, cam, tag, spin):
    """Same check against frames of the reference kernel committed under tests/golden/ (generated on a B200 by
    tests/tools/make_golden_refcuda.py), so the pin does not depend on the reference tree being present."""
    import os
    path = os.path.join(os.path.dirname(__file__), "golden", "refcuda_frames.npz")
    if not os.path.exists(path):
        pytest.skip("tests/golden/refcuda_frames.npz not generated yet")
    ref_rgba = np.load(path)[f"{cam}_{tag}"]
    h, w = ref_rgba.shape[:2]
    untouched, diff = _ours_vs(gpu, sky_small, ref_rgba, cam, spin, w, h)
    assert diff[untouched].max() == 0
    assert diff[~untouched].max() <= 1 and (diff[~untouched] > 0).sum() <= 3
