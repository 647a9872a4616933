"""Every tracer against the oracle port and against each other at parameter sets that move the thresholds the render
kernels' unchecked step runs (bursts) are validated against.

The kernels take runs of kBurst steps without their per-step checks -- vacuum bursts in every tracer, zone bursts (near
the hole, in the disk zone) in the split pipeline's packed tracer -- and check afterwards that none of the skipped checks
would have fired.  Those checks compare radii with horizon_r = 1.01 event_horizon, acc_rmin = 0.5 event_horizon (the
branch-free domain), disk_zone_r = disk_out + 5, disk_zone_y = 5 disk_h, dust_zone_r = cloud_out, the near-hole radius 18
and the escape radius 250, and how these are ordered decides which checks a burst can skip.  The default parameters give
one order; each regime below gives another, with cameras whose rays reach the boundary in question, and asserts on the
oracle's frame that they do (so that a later change of camera or default cannot leave the case empty).

Three kinds of check:
  * each tracer against the oracle port: exact trajectories (steps, pos, vel, dir), CAPTURED / EXHAUSTED and the
    counters rk4_steps, disk_evals, dust_evals, n_captured, n_exhausted; emission and hdr within the tolerances of
    test_gpu_oracle_reach.py;
  * each split-pipeline tracer against the fused kernel of the same contract, bit for bit: every plane, the frame and
    every counter;
  * max_steps at the limits that choose the tracer, and the other users of the packed trace kernel (rrt_capture and the
    lens instance behind rrt_render_dof), exactly against fused renders.

tests/tools/params_census.py imports the cases and the rendering from this file."""
import numpy as np
import pytest

from parity import CAMERAS
from test_gpu_dof import _dof, _expected_hi, _renderer, _resolve, _same
from test_gpu_oracle_reach import EMIS_TOL, EXACT_COUNTERS, _frame_dicts, check

pytestmark = pytest.mark.gpu

W, H, TIME, SPIN = 96, 54, 1.0, 0.99
SLAB_BIG = ((0.0, 0.2, -26.0), 0.0, -0.5)      # r = 26, inside the disk slab, looking at the hole
SLAB_HUGE = ((0.0, 0.2, -50.0), 0.0, -0.5)
SLAB_FAR = ((0.0, 0.3, 235.0), 0.0, 0.0)       # r = 235, inside the disk slab, looking outward (+z)
BIG_HOLE = dict(event_horizon=20.0, isco_radius=22.0, disk_out=60.0, cloud_out=60.0)
HUGE_HOLE = dict(event_horizon=40.0, isco_radius=45.0, disk_out=80.0, cloud_out=80.0)
DISK_PAST_ESCAPE = dict(disk_out=300.0)


def _escaped(f):
    return ((f.cls & 3) != 0) & ((f.cls & 4) == 0)


def _captured(f):
    return (f.cls & 3) == 0


def _r(f):
    return np.linalg.norm(f.pos[..., :3].astype(np.float64), axis=-1)


def _in_slab(f, p):
    return np.abs(f.pos[..., 1].astype(np.float64)) < 5.0 * p.disk_h


# name: (parameter overrides, cameras (survey name or (pos, yaw, pitch)), what the oracle's disk + dust FMAD frame of at
# least one camera shows: the regime reaches its boundary)
REGIMES = {
    # control
    "defaults": ({}, ["C1", "C3"], lambda f, p: f.counters["disk_evals"] > 0 and f.counters["n_captured"] > 0),
    # horizon_r = 20.2 > 18: the disk zone reaches down to the horizon
    "big-hole": (BIG_HOLE, [SLAB_BIG, "C0"], lambda f, p: (_captured(f) & _in_slab(f, p) & (_r(f) >= 18.0)).sum() > 100),
    # acc_rmin = 20 > 18 as well: the branch-free domain ends inside the disk zone
    "huge-hole": (HUGE_HOLE, [SLAB_HUGE], lambda f, p: (_captured(f) & _in_slab(f, p) & (_r(f) >= 18.0)).sum() > 100),
    # disk_zone_r = 305 > 250: rays escape from inside the disk zone
    "disk-past-escape": (DISK_PAST_ESCAPE, [SLAB_FAR, "C0"], lambda f, p: (_escaped(f) & _in_slab(f, p)).sum() > 100),
    # horizon_r = 0: no fast step anywhere (fast_ok false) while the media are on
    "flat": (dict(event_horizon=0.0), ["C0", "C1"], lambda f, p: f.counters["n_captured"] == 0 and f.counters["disk_evals"] > 0),
    # disk_zone_r = 17 < 18: the disk lies inside the near-hole zone, the disk-zone window is empty
    "disk-in-near-zone": (dict(disk_out=12.0, isco_radius=3.0, cloud_out=15.0), ["C3"], lambda f, p: f.counters["disk_evals"] > 0),
    # dust_zone_r = 60 sets the zone radius, dust far outside the disk zone
    "wide-dust": (dict(cloud_out=60.0, cloud_h=3.0), ["C1"], lambda f, p: f.counters["dust_evals"] > f.counters["disk_evals"] > 0),
    # disk_zone_y = 0.25 < the disk-zone burst margin: no disk bursts at all
    "thin-disk": (dict(disk_h=0.05), ["C0"], lambda f, p: f.counters["disk_evals"] > 0),
    # margins much smaller / larger than the windows
    "step0.05": (dict(step_size=0.05), ["C1"], lambda f, p: f.counters["n_exhausted"] > 0 and f.counters["disk_evals"] > 0),
    "step2": (dict(step_size=2.0), ["C1"], lambda f, p: f.counters["n_captured"] > 0 and f.counters["disk_evals"] > 0),
    # negative frame drag; the SPIN instance at another value
    "spin-0.99": (dict(spin_a=-0.99), ["C1", "C3"], lambda f, p: f.counters["n_captured"] > 0),
    "spin0.5": (dict(spin_a=0.5), ["C1", "C3"], lambda f, p: f.counters["n_captured"] > 0),
    # the fold / transmittance arithmetic away from the default media constants
    "media-dense": (dict(disk_opacity=40.0, disk_luminosity=50.0, cloud_luminosity=0.0, disk_temp_ref=4.0e6), ["C3"],
                    lambda f, p: f.counters["dense_samples"] > 0),
    "media-clear": (dict(disk_opacity=0.0), ["C3"], lambda f, p: f.counters["dense_samples"] > 0),
}
# Emission bounds of the regimes that exceed test_gpu_oracle_reach.EMIS_TOL, from profiles/params_census_b200.jsonl
# (NVIDIA B200, 1000 W power limit; every tracer of the regime, t = 1).  The exact part held in all 180 cases of the census,
# no TOUCHED flag differed and the hdr stayed within HDR_TOL everywhere.
REGIME_EMIS_TOL = {
    # six times the samples of the default step, each with the libdevice / glibc rounding of the noise: census max 4.86e-4,
    # p99.9 3.71e-4, p99 1.39e-4 (fused_strict / split_strict).  Margins 1.34x, 1.29x, 1.29x.
    "step0.05": {"max": (6.5e-4, 0.0), "p999": (4.8e-4, 0.0), "p99": (1.8e-4, 0.0)},
    # a disk of zero opacity emits nothing, so a pixel's emission is the dust's alone, without the disk's larger terms to
    # dilute its rounding: census max 2.94e-4, p99.9 1.99e-4 (strict), p99 1.41e-5.  Margins 1.29x, 1.31x; p99 as EMIS_TOL.
    "media-clear": {"max": (3.8e-4, 0.0), "p999": (2.6e-4, 0.0), "p99": EMIS_TOL["p99"]},
}
# (context, pipeline, flags, the fused tracer a split one must equal bit for bit)
TRACERS = {
    "scalar_fused": ("auto", "auto", 0, None),          # strict, no medium: render_kernel
    "packed_fused": ("auto", "auto", 4, None),          # FMAD, no medium: render_kernel_p
    "fused_media": ("auto", "fused", 7, None),          # render_kernel with the media inline
    "fused_disk": ("auto", "fused", 5, None),
    "fused_strict": ("auto", "fused", 3, None),
    "split_packed": ("auto", "split", 7, "fused_media"),         # trace_kernel_p + media + fold
    "split_packed_disk": ("auto", "split", 5, "fused_disk"),
    "split_scalar": ("scalar", "split", 7, "fused_media"),       # trace_kernel under the FMAD contract
    "split_strict": ("auto", "split", 3, "fused_strict"),        # trace_kernel under the strict contract
}


def cases():
    """(regime, camera index) of every regime camera"""
    return [(name, k) for name, (_, cams, _) in REGIMES.items() for k in range(len(cams))]


def case_id(regime, k):
    return f"{regime}-{k}"


def params_of(mod, regime, flags, **more):
    """rrt.default_params / Oracle.default_params with the regime's overrides (spin 0.99 unless it sets one)"""
    return mod.default_params(**{"spin_a": SPIN, "flags": flags, **REGIMES[regime][0], **more})


def camera_of(rrt, regime, k):
    cam = REGIMES[regime][1][k]
    return rrt.camera_state_from(*(CAMERAS[cam] if isinstance(cam, str) else cam))


def tiles_of(packed, w=W, h=H):
    """tickets of a split-pipeline frame: 16x4 tiles for the packed tracer, 8x4 for the scalar one"""
    return -(-w // (16 if packed else 8)) * -(-h // 4)


def gpu_frame(r, prm, cam, sky, w=W, h=H, time=TIME):
    """every plane, the frame and the counters of one rrt_render, as numpy"""
    import relativisticraytracer_b200 as rrt
    import torch
    planes = r.alloc_planes(w, h)
    r.read_counters(reset=True)
    out = r.render(prm, cam, rrt.effects_off(), sky, time, w, h, planes=planes)
    torch.cuda.synchronize()
    g = {k: v.cpu().numpy() for k, v in planes.items()}
    g["rgba"] = out.cpu().numpy()
    g["counters"] = r.read_counters(reset=True)
    return g


def render_tracer(ctxs, skies, tracer, regime, k, **more):
    """(GPU dict, the context it ran in) of one tracer on one regime camera"""
    import relativisticraytracer_b200 as rrt
    ctx, pipeline, flags, _ = TRACERS[tracer]
    r = ctxs[ctx]
    r.set_pipeline(pipeline)
    return gpu_frame(r, params_of(rrt, regime, flags, **more), camera_of(rrt, regime, k), skies[ctx]), r


def oracle_frame(ora, sky_np, regime, k, flags, **more):
    from oracle import Camera as OraCamera
    import relativisticraytracer_b200 as rrt
    cam = camera_of(rrt, regime, k)
    co = OraCamera.from_buffer_copy(bytes(cam))
    return ora.render(params_of(ora, regime, flags, **more), co, ora.effects_off(), sky_np, TIME, W, H)


def case_dict(cid):
    return {"id": cid, "section": 0, "time": TIME, "mask": "all"}


def same_bits(a, b, tag):
    """every plane, the frame and every counter of two GPU dicts"""
    for key in a:
        if key == "counters":
            assert a[key] == b[key], f"{tag}: counters {a[key]} != {b[key]}"
        else:
            x, y = a[key], b[key]
            assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), \
                f"{tag}: {key} differs at {int(np.sum(np.any((x != y).reshape(x.shape[0], x.shape[1], -1), axis=-1)))} pixels"


# ---- fixtures ------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def env(built, sky_smooth):
    """Contexts of their own (RRT_TRACE is read when a context is created; pipeline and counters are per context) with
    the smooth sky."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    ctxs = {"auto": _renderer("auto"), "scalar": _renderer("scalar")}
    skies = {k: r.create_sky(sky_smooth) for k, r in ctxs.items()}
    yield ctxs, skies
    for k, r in ctxs.items():
        skies[k].close()
        r.close()


@pytest.fixture(scope="module")
def oracle_frames(ora, sky_smooth):
    """the oracle's frame of each (regime, camera, flags), rendered once for the module"""
    memo = {}

    def get(regime, k, flags, **more):
        key = (regime, k, flags, tuple(sorted(more.items())))
        if key not in memo:
            memo[key] = oracle_frame(ora, sky_smooth, regime, k, flags, **more)
        return memo[key]
    return get


# ---- 1. every tracer in every regime -----------------------------------------------------------------------------------
@pytest.mark.parametrize("tracer", list(TRACERS))
@pytest.mark.parametrize("regime,k", [pytest.param(*c, id=case_id(*c)) for c in cases()])
def test_tracer(env, oracle_frames, regime, k, tracer):
    ctxs, skies = env
    flags, fused = TRACERS[tracer][2], TRACERS[tracer][3]
    tag = f"{case_id(regime, k)} {tracer}"
    g, r = render_tracer(ctxs, skies, tracer, regime, k)
    if TRACERS[tracer][1] == "split":
        packed = TRACERS[tracer][0] == "auto" and flags & 4 != 0
        assert r.split_stats()["tiles"] == tiles_of(packed), f"{tag}: not the expected split tracer"
        same_bits(g, render_tracer(ctxs, skies, fused, regime, k)[0], f"{tag} vs {fused}")
    fo, go = _frame_dicts(oracle_frames(regime, k, flags), g)
    check(case_dict(tag), fo, go, emis=REGIME_EMIS_TOL.get(regime, EMIS_TOL))


@pytest.mark.parametrize("regime", list(REGIMES))
def test_regime_reaches_its_boundary(ora, oracle_frames, regime):
    _, cams, reach = REGIMES[regime]
    frames = [oracle_frames(regime, k, 7) for k in range(len(cams))]
    assert any(reach(f, params_of(ora, regime, 7)) for f in frames), [f.counters for f in frames]


# ---- 2. max_steps at the limits that choose the tracer -----------------------------------------------------------------
# rrt_b200.cu: the packed split tracer takes 2 (max_steps + 1) + 2 <= 128 (kDescChunks - 2) rows, the split pipeline
# max_steps + 2 <= 128 (kDescChunks - 2); beyond, the scalar split tracer and then the fused kernel trace the frame.
MAX_STEPS = {2430: "split packed", 2431: "split scalar", 4862: "split scalar", 4863: "fused"}


@pytest.mark.parametrize("max_steps", list(MAX_STEPS))
def test_max_steps_at_the_tracer_limits(env, oracle_frames, max_steps):
    ctxs, skies = env
    r = ctxs["auto"]
    l0 = r.kernel_launches()
    g, _ = render_tracer(ctxs, skies, "split_packed", "defaults", 1, max_steps=max_steps)
    launches = r.kernel_launches() - l0
    side = MAX_STEPS[max_steps]
    if side == "fused":
        assert launches == 1, launches
    else:
        st = r.split_stats()
        assert launches == 3 * st["passes_enqueued"] + 1, (launches, st)
        assert st["tiles"] == tiles_of(side == "split packed"), (side, st)
    same_bits(g, render_tracer(ctxs, skies, "fused_media", "defaults", 1, max_steps=max_steps)[0], f"max_steps {max_steps}")
    assert g["steps"].max() >= min(max_steps, 2431)     # rays use the budget up to the packed tracer's limit
    fo, go = _frame_dicts(oracle_frames("defaults", 1, 7, max_steps=max_steps), g)
    check(case_dict(f"max_steps {max_steps}"), fo, go)


def test_capture_max_steps_limit(env):
    import relativisticraytracer_b200 as rrt
    ctxs, skies = env
    r = ctxs["auto"]
    cam = camera_of(rrt, "defaults", 1)
    cap = r.capture(params_of(rrt, "defaults", 7, max_steps=4862), cam, rrt.effects_off(), skies["auto"], 32, 16)
    assert not cap.info()["packed"]
    cap.close()
    with pytest.raises(rrt.RrtError):
        r.capture(params_of(rrt, "defaults", 7, max_steps=4863), cam, rrt.effects_off(), skies["auto"], 32, 16)


# ---- 3. the other users of the packed trace kernel ---------------------------------------------------------------------
def _hdr(r, w=W, h=H):
    import torch
    return torch.zeros((h, w, 4), dtype=torch.float32, device=r.device)


@pytest.mark.parametrize("regime", ["big-hole", "disk-past-escape"])
def test_capture_equals_fused_render(env, regime):
    """rrt_capture traces with trace_kernel_p: its trace counts the fused kernel's steps, classes and zone entries, and its
    render at any time is the fused kernel's frame at that time.  (At big-hole the frame alone cannot tell: the steps a
    ray takes below the horizon lie inside isco, where no sample is kept.)"""
    import relativisticraytracer_b200 as rrt
    import torch
    ctxs, skies = env
    r, sky, fx = ctxs["auto"], skies["auto"], rrt.effects_off()
    prm, cam = params_of(rrt, regime, 7), camera_of(rrt, regime, 0)
    r.read_counters(reset=True)
    cap = r.capture(prm, cam, fx, sky, W, H)
    try:
        traced = r.read_counters(reset=True)
        assert cap.info()["packed"]
        r.set_pipeline("fused")
        for t in (1.0, 7.5):
            got_hdr, want_hdr = _hdr(r), _hdr(r)
            got = cap.render(prm, fx, sky, t, hdr_out=got_hdr)
            r.read_counters(reset=True)
            want = r.render(prm, cam, fx, sky, t, W, H, planes={"hdr": want_hdr})
            torch.cuda.synchronize()
            fused = r.read_counters(reset=True)
            assert {k: traced[k] for k in EXACT_COUNTERS} == {k: fused[k] for k in EXACT_COUNTERS}, (regime, traced, fused)
            for name, a, b in (("frame", got, want), ("hdr", got_hdr, want_hdr)):
                a, b = a.cpu().numpy(), b.cpu().numpy()
                assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), f"{regime} t={t}: {name} differs on {np.sum(a != b)} elements"
    finally:
        cap.close()
        r.set_pipeline("auto")


@pytest.mark.parametrize("pipeline", ["auto", "fused"])
@pytest.mark.parametrize("regime", ["big-hole", "disk-past-escape"])
def test_render_dof_on_the_slab_camera(env, regime, pipeline):
    """rrt_render_dof (the lens instance of the tracers) equals the ss*w x ss*h composition of fused plain renders, the
    way test_gpu_dof._check builds it, and counts the steps and classes of the pixels each render contributes: the split
    pipeline's render_dof must give the fused pipeline's bytes and counts"""
    import relativisticraytracer_b200 as rrt
    ctxs, skies = env
    r, sky = ctxs["auto"], skies["auto"]
    prm, fx = params_of(rrt, regime, 7), rrt.default_effects()
    ss = 2
    cams = rrt.lens_cameras(camera_of(rrt, regime, 0), 0.5, 20.0, ss)
    r.set_pipeline("fused")
    hi, pl = _expected_hi(r, prm, cams, fx, sky, W, H, ss, planes=("steps", "cls"))
    want = _resolve(r, prm, fx, hi, ss, W, H)
    steps = np.concatenate([pl["steps"][k].cpu().numpy()[k // ss::ss, k % ss::ss].ravel() for k in range(ss * ss)])
    cls = np.concatenate([pl["cls"][k].cpu().numpy()[k // ss::ss, k % ss::ss].ravel() for k in range(ss * ss)])
    r.set_pipeline(pipeline)
    r.read_counters(reset=True)
    _same(_dof(r, prm, cams, fx, sky, W, H, ss), want, f"{regime} {pipeline}")
    got = r.read_counters(reset=True)
    r.set_pipeline("auto")
    assert got["rk4_steps"] == int(steps.astype(np.int64).sum()), (regime, pipeline)
    assert got["n_captured"] == int(((cls & rrt.CLS_MASK) == rrt.CLS_CAPTURED).sum()), (regime, pipeline)
    assert got["n_exhausted"] == int(((cls & rrt.CLSF_EXHAUSTED) != 0).sum()), (regime, pipeline)
