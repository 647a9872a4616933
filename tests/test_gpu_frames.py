"""Whole-frame parity, CUDA (through the C ABI) vs the oracle port, at sizes the oracle finishes in seconds."""
import numpy as np
import pytest

from parity import CAMERAS, DIR_TOL_RAD, RGB_TOL_REL, census

pytestmark = pytest.mark.gpu


def render_pair(gpu, ora, sky_np, cam_key, spin, flags, w, h, time=1.0, fx="off", cam=None, **over):
    """The frame with all its planes and counters from the GPU and from the oracle port.  cam_key names a survey camera;
    `cam` (a Camera, e.g. of a path or a lens table) replaces it.  fx is "off", "default" or an Effects."""
    import relativisticraytracer_b200 as rrt
    import torch
    from oracle import Camera as OraCamera, Effects as OraEffects
    pg = rrt.default_params(spin_a=spin, flags=flags, **over)
    po = ora.default_params(spin_a=spin, flags=flags, **over)
    if cam is None:
        pos, yaw, pitch = CAMERAS[cam_key]
        cg = rrt.camera_state_from(pos, yaw, pitch)
        co = ora.camera_from(pos, yaw, pitch)
    else:
        cg, co = cam, OraCamera.from_buffer_copy(bytes(cam))
    assert bytes(cg) == bytes(co)
    if isinstance(fx, str):
        fg = rrt.effects_off() if fx == "off" else rrt.default_effects()
        fo = ora.effects_off() if fx == "off" else ora.default_effects()
    else:
        fg, fo = fx, OraEffects.from_buffer_copy(bytes(fx))
    sky = gpu.create_sky(sky_np)
    planes = gpu.alloc_planes(w, h)
    gpu.read_counters(reset=True)
    out = gpu.render(pg, cg, fg, sky, time, w, h, planes=planes)
    torch.cuda.synchronize()
    cnt = gpu.read_counters()
    new = {k: v.cpu().numpy() for k, v in planes.items()}
    new["rgba"] = out.cpu().numpy()
    new["counters"] = cnt
    sky.close()
    f = ora.render(po, co, fo, sky_np, time, w, h)
    return f, new


def test_config1_schwarzschild_256(gpu, ora, sky_small):
    """BASELINE config 1: 256x256, a=0, geodesic only, default camera.  Known answers from the reference
    headers (SURVEY.md 7.2): 69,585,851 steps; 374 captured / 63,208 escaped / 1,954 exhausted (lens
    distortion on, as in the survey probe)."""
    f, g = render_pair(gpu, ora, sky_small, "C0", 0.0, 0, 256, 256, fx="default")
    assert g["counters"]["rk4_steps"] == 69585851 == f.counters["rk4_steps"]
    assert (g["counters"]["n_captured"], g["counters"]["n_escaped"], g["counters"]["n_exhausted"]) == (374, 63208, 1954)
    for k in ("cls", "steps", "pos", "vel", "dir"):
        assert np.array_equal(g[k], getattr(f, k)), k


@pytest.mark.parametrize("cam", ["C0", "C1", "C2", "C3"])
@pytest.mark.parametrize("spin", [0.0, 0.99])
def test_geodesic_only_bit_exact(gpu, ora, sky_smooth, cam, spin):
    f, g = render_pair(gpu, ora, sky_smooth, cam, spin, 0, 160, 90)
    for k in ("cls", "steps", "pos", "vel", "dir"):
        assert np.array_equal(g[k], getattr(f, k)), k
    c = census(f, g)
    assert c["class_flips"] == 0 and c["dir_max_rad"] == 0.0
    assert c["rgb_max_rel"] < RGB_TOL_REL, c          # sky lookup: texture unit vs host emulation
    assert g["counters"] == f.counters


@pytest.mark.parametrize("cam", ["C0", "C1", "C2", "C3"])
@pytest.mark.parametrize("flags", [1, 3])
def test_volumetric_parity(gpu, ora, sky_smooth, cam, flags):
    """a=0.99 with the disk (flags=1, BASELINE config 2 reading) and disk+dust (flags=3, config 3)."""
    f, g = render_pair(gpu, ora, sky_smooth, cam, 0.99, flags, 160, 90)
    # the trajectory never depends on the media: still bit-exact
    for k in ("steps", "pos", "vel", "dir"):
        assert np.array_equal(g[k], getattr(f, k)), k
    c = census(f, g)
    assert c["class_flips"] == 0, c
    assert c["dir_max_rad"] <= DIR_TOL_RAD
    assert g["counters"]["rk4_steps"] == f.counters["rk4_steps"]
    assert g["counters"]["disk_evals"] == f.counters["disk_evals"]
    assert g["counters"]["dust_evals"] == f.counters["dust_evals"]
    assert c["rgb_frac_over_tol"] == 0.0, c
    # emission and transmittance alone (no texture unit involved)
    e_rel = np.abs(g["emis"][..., :3].astype(np.float64) - f.emis[..., :3]) / np.maximum(np.abs(f.emis[..., :3]), 1e-3)
    assert e_rel.max() < RGB_TOL_REL
    assert np.abs(g["rgba"].astype(int) - f.rgba.astype(int)).max() <= 1


def test_star_field_sky_outliers_are_texture_quantisation(gpu, ora, sky_small):
    """With a high-contrast star field the only pixels past 1e-3 are sky taps whose texture coordinate
    differs by an ulp between libdevice and glibc atan2f/asinf (glibc 2.39's are themselves not correctly
    rounded in 16 % / 7 % of arguments) and therefore lands in a neighbouring 1/256 filter-weight bucket of
    the texture unit: error <= contrast/256.  Trajectory, class and emission stay exact / in tolerance."""
    f, g = render_pair(gpu, ora, sky_small, "C0", 0.99, 3, 240, 135)
    c = census(f, g)
    assert c["class_flips"] == 0 and c["dir_max_rad"] == 0.0
    assert np.array_equal(g["vel"], f.vel)
    assert c["rgb_frac_over_tol"] < 2e-3 and c["rgb_max_rel"] < 1e-2, c
    e_rel = np.abs(g["emis"][..., :3].astype(np.float64) - f.emis[..., :3]) / np.maximum(np.abs(f.emis[..., :3]), 1e-3)
    assert e_rel.max() < RGB_TOL_REL


def test_default_effects_bytes(gpu, ora, sky_small):
    """reference default CameraEffects (bloom, vignette, lens on): final uchar4 within one count."""
    f, g = render_pair(gpu, ora, sky_small, "C1", 0.99, 3, 160, 90, fx="default")
    d = np.abs(g["rgba"].astype(int) - f.rgba.astype(int))
    assert d.max() <= 1 and np.mean(d > 0) < 0.02
    assert np.array_equal(g["rgba"][..., 3], f.rgba[..., 3])


def test_nondefault_params(gpu, ora, sky_smooth):
    """run-time parameters really are run-time: smaller step budget, thicker dust, other step size."""
    f, g = render_pair(gpu, ora, sky_smooth, "C2", 0.7, 3, 96, 54, max_steps=700, step_size=0.25, cloud_h=3.0, disk_h=0.5)
    for k in ("steps", "pos", "vel"):
        assert np.array_equal(g[k], getattr(f, k)), k
    c = census(f, g)
    assert c["class_flips"] == 0 and c["rgb_frac_over_tol"] == 0.0, c


def test_bands_equal_full_frame(gpu, sky_small):
    """cyclic row bands (multi-GPU partition) reproduce the single-launch frame bit for bit."""
    import relativisticraytracer_b200 as rrt
    import torch
    w, h = 200, 117     # ragged: not a multiple of tile, group or rank count
    prm = rrt.default_params(spin_a=0.99)
    cam = rrt.camera_state_from(*CAMERAS["C1"])
    fx = rrt.default_effects()
    sky = gpu.create_sky(sky_small)
    full = gpu.render(prm, cam, fx, sky, 1.0, w, h)
    for nranks, group in [(2, 8), (4, 16), (8, 1), (3, 5)]:
        rows = max(gpu.band_rows(rrt.Band(r, nranks, group), h) for r in range(nranks))
        packed = torch.zeros((nranks, rows, w, 4), dtype=torch.uint8, device=gpu.device)
        frame = torch.zeros((h, w, 4), dtype=torch.uint8, device=gpu.device)
        for r in range(nranks):
            b = rrt.Band(r, nranks, group)
            gpu.render(prm, cam, fx, sky, 1.0, w, h, band=b, out=packed[r], layout=rrt.OUT_PACKED)
            gpu.render(prm, cam, fx, sky, 1.0, w, h, band=b, out=frame, layout=rrt.OUT_FRAME)
        asm = gpu.assemble_bands(packed, rows, w, h, nranks, group)
        torch.cuda.synchronize()
        assert torch.equal(asm, full), (nranks, group)
        assert torch.equal(frame, full), (nranks, group)
    sky.close()


def test_launch_raymarch_mirror(gpu, sky_small):
    """the reference-named entry point renders into a caller-owned buffer like the C ABI does."""
    import relativisticraytracer_b200 as rrt
    import torch
    w, h = 128, 72
    sky = gpu.create_sky(sky_small)
    cam = rrt.camera_state_from(*CAMERAS["C0"])
    fx = rrt.CameraEffects()
    rrt._capi.load().rrt_default_effects(fx)
    d_out = torch.zeros((h, w, 4), dtype=torch.uint8, device="cuda")
    rrt.launch_raymarch(d_out, w, h, 1.0, cam, sky.texture, fx)
    ref = gpu.render(rrt.default_params(), cam, fx, sky, 1.0, w, h)
    torch.cuda.synchronize()
    assert torch.equal(d_out, ref)
    host = np.zeros((h, w, 4), np.uint8)
    gpu.render_host(rrt.default_params(), cam, fx, sky, 1.0, w, h, host)
    assert np.array_equal(host, ref.cpu().numpy())
    sky.close()


def test_bad_arguments(gpu, sky_small):
    import relativisticraytracer_b200 as rrt
    sky = gpu.create_sky(sky_small)
    cam = rrt.camera_state_from(*CAMERAS["C0"])
    with pytest.raises(rrt.RrtError):
        gpu.render(rrt.default_params(), cam, rrt.effects_off(), 0, 1.0, 64, 64)          # null texture
    with pytest.raises(rrt.RrtError):
        gpu.render(rrt.default_params(), cam, rrt.effects_off(), sky, 1.0, 64, 64, band=rrt.Band(3, 2, 4))
    sky.close()
