"""Edge cases of the path, CUDA (through the C ABI) vs the oracle port, in both rounding contracts: the step
budget's ends, one-pixel frames, a camera inside the horizon, the general-domain fallback of the render loop (a
camera so far out that the branch-free div/sqrt domain does not apply; a horizon so large that a single RK4 stage
can jump inside r < Rs/2, where getGeodesicAcc returns zero, geodesics.h:33)."""
import numpy as np
import pytest

from parity import census

pytestmark = pytest.mark.gpu

CONTRACTS = [3, 7]   # strict, FMAD (flags: disk | dust [| RRT_FLAG_FMAD]); ORA_FLAG_* == RRT_FLAG_*


def pair(gpu, ora, sky_np, pos, yaw, pitch, w, h, flags, spin=0.99, **over):
    import relativisticraytracer_b200 as rrt
    import torch
    pg = rrt.default_params(spin_a=spin, flags=flags, **over)
    po = ora.default_params(spin_a=spin, flags=flags, **over)
    cg, co = rrt.camera_state_from(pos, yaw, pitch), ora.camera_from(pos, yaw, pitch)
    sky = gpu.create_sky(sky_np)
    planes = gpu.alloc_planes(w, h)
    gpu.read_counters(reset=True)
    out = gpu.render(pg, cg, rrt.effects_off(), sky, 1.0, w, h, planes=planes)
    torch.cuda.synchronize()
    g = {k: v.cpu().numpy() for k, v in planes.items()}
    g["rgba"], g["counters"] = out.cpu().numpy(), gpu.read_counters()
    sky.close()
    return ora.render(po, co, ora.effects_off(), sky_np, 1.0, w, h), g


def same_trajectories(f, g):
    for k in ("cls", "steps", "pos", "vel", "dir"):
        assert np.array_equal(g[k], getattr(f, k), equal_nan=True), k
    assert g["counters"] == f.counters


@pytest.mark.parametrize("flags", CONTRACTS)
@pytest.mark.parametrize("max_steps", [0, 1, 2, 37])
def test_step_budget_ends(gpu, ora, sky_smooth, flags, max_steps):
    f, g = pair(gpu, ora, sky_smooth, (15.0, 3.0, -30.0), -26.6, -5.1, 64, 36, flags, max_steps=max_steps)
    same_trajectories(f, g)
    assert int(g["steps"].max()) <= max_steps
    assert census(f, g)["rgb_frac_over_tol"] == 0.0


@pytest.mark.parametrize("flags", CONTRACTS)
@pytest.mark.parametrize("w,h", [(1, 1), (1, 7), (9, 1), (33, 5)])
def test_tiny_and_ragged_frames(gpu, ora, sky_smooth, flags, w, h):
    f, g = pair(gpu, ora, sky_smooth, (0.0, 10.0, -60.0), 0.0, -10.0, w, h, flags)
    same_trajectories(f, g)
    assert np.abs(g["rgba"].astype(int) - f.rgba.astype(int)).max() <= 1


@pytest.mark.parametrize("flags", CONTRACTS)
def test_camera_inside_the_horizon(gpu, ora, sky_smooth, flags):
    f, g = pair(gpu, ora, sky_smooth, (0.5, 1.0, 1.2), 30.0, 5.0, 40, 24, flags)
    same_trajectories(f, g)
    assert g["counters"]["n_captured"] == 40 * 24 and g["counters"]["rk4_steps"] == 0
    assert not g["rgba"][..., :3].any()          # black: T = 0 and nothing emitted (raymarcher.cu:47-51, 128)


@pytest.mark.parametrize("flags", CONTRACTS)
def test_far_camera_takes_the_general_path(gpu, ora, sky_smooth, flags):
    """|p|^2 >= 1e8: every step is redone with the guarded division / square root (rk4_step_general)"""
    f, g = pair(gpu, ora, sky_smooth, (0.0, 500.0, -20000.0), 0.0, -1.4, 48, 27, flags, max_steps=300)
    same_trajectories(f, g)
    assert g["counters"]["n_exhausted"] + g["counters"]["n_escaped"] == 48 * 27


@pytest.mark.parametrize("flags", CONTRACTS)
def test_stage_inside_half_horizon(gpu, ora, sky_smooth, flags):
    """event_horizon = 20 and a 30-unit step: RK4 stages land inside r < 10 = Rs/2, where the acceleration is
    defined as zero (geodesics.h:33) -- the branch-free loop must notice and redo those steps."""
    f, g = pair(gpu, ora, sky_smooth, (0.0, 2.0, -45.0), 0.0, -2.0, 64, 36, flags, event_horizon=20.0, step_size=100.0,
                disk_out=60.0, isco_radius=22.0, cloud_out=60.0)
    same_trajectories(f, g)
    assert g["counters"]["n_captured"] > 0 and g["counters"]["n_escaped"] + g["counters"]["n_exhausted"] > 0
    assert census(f, g)["rgb_frac_over_tol"] == 0.0

