"""rrt_render against the oracle port at the inputs the re-timing, motion-blur, supersampling and depth-of-field features
feed it, which the other oracle-comparing files do not reach: frame times other than 1.0, path and lens cameras, camera
positions inside the media, next to the horizon and looking along the spin axis, every post effect at non-default
settings, and sampled rows of 1080p and 4K frames (the split pipeline's tiling at full size).

What does not depend on time or effects is exact in every case: the trajectory planes (steps, pos, vel, dir), the CAPTURED
class and EXHAUSTED flag, and the counters rk4_steps, disk_evals, dust_evals, n_captured and n_exhausted (a ray ends only at
the horizon, on escape or at max_steps; disk_evals / dust_evals count zone entries).  What passes through a medium, a
transcendental or the texture unit (emis, hdr, rgba, dense_samples, n_touched, the TOUCHED flag) is compared within
tolerances measured on a B200 by tests/tools/oracle_reach_census.py (profiles/oracle_reach_census_b200.jsonl).

tests/tools/oracle_reach_census.py imports the cases and the comparison from this file."""
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from parity import CAMERAS
from test_gpu_frames import render_pair

pytestmark = pytest.mark.gpu

FMAD = 4                                       # RRT_FLAG_FMAD == ORA_FLAG_FMAD
CONTRACTS = {"strict": 3, "fmad": 3 | FMAD}    # disk + dust
TIMES = (-2.0, 0.0, 0.5, 12.5, 50.0, 123.5)    # the times the motion-blur and re-time tests render at
PATH_TIMES = (0.0, 3.3, 12.0, 20.7, 40.0)      # a keyframe, between keyframes, past the last key of every path
LENS_CAMS = [((0.0, 10.0, -60.0), 0.0, -10.0), ((25.0, 3.0, -40.0), -32.0, -4.0), ((-7.5, 1.0, 35.0), 171.0, 2.5),
             ((0.0, -20.0, 0.0), 0.0, 89.0)]   # the cameras of test_lens_cameras.py
LENS = (2.0, 12.5, 2)                          # aperture, focus, ss: forward - o/focus is ~1 % off unit length
# Camera positions the survey cameras never take (default parameters: isco 10, disk_out 25, disk_h 0.8, cloud_h 0.5).
POSES = {
    "in-disk-slab": ((3.0, 0.2, -17.0), 40.0, 2.0),       # r = 17.3, |y| < disk_h: every ray's first step samples the disk
    "in-dust-layer": ((12.0, 0.6, -16.0), -20.0, -3.0),    # r = 20, y = 0.6 < 1.5 cloud_h: in the dust zone, above the disk
    "near-horizon": ((0.0, 0.3, -2.03), 90.0, 0.0),        # r = 2.052, just outside the 2.02 capture radius, looking along +x
    "pole-down": ((0.0, 40.0, -5.0), 0.0, -89.0),          # along the spin axis
    "pole-up": ((0.0, -40.0, 5.0), 180.0, 89.0),
}
POLE_POSES = ("pole-down", "pole-up")
EXACT_COUNTERS = ("rk4_steps", "disk_evals", "dust_evals", "n_captured", "n_exhausted")
ROW_COUNTERS = ("rk4_steps", "n_captured", "n_exhausted")   # the ones the GPU's planes give per row
# evenly spaced rows of a full-size frame: with the first / last / middle rows and a tile-row boundary pair, about 21 rows,
# rendered by the oracle one row per core.  Fixed rather than taken from the host's core count, so that every host compares
# the rows the census measured.
EVEN_ROWS = 16


# ---- tolerances, from profiles/oracle_reach_census_b200.jsonl ----------------------------------------------------------
# Measured on an NVIDIA B200 (1000 W power limit), all 122 cases of this file: the exact part held in every case, no TOUCHED
# flag differed, n_touched was equal everywhere and dense_samples differed by at most 4.  Each bound below is written as
# a + b |t| (t = frame time) and clears the worst census value by the margin stated with it.
#
# Emission relative error |g - f| / max(|f|, 1e-3), per pixel the worst channel.  The noise's sensitivity to the libdevice /
# glibc rounding of powf (omega), sinf / cosf (rotation) and atan2f grows with |t|.  Census: p99 <= 5.8e-5 up to t = 50 and
# 1.0e-4 at t = 123.5; p99.9 <= 1.14e-4 up to t = 50 and 2.0e-4 at 123.5; max <= 1.8e-4 at t = 1 and 5.2e-4 at 123.5 (the
# 96x54 default-effects case).  Smallest margin of each bound over the census's cases: p99 1.13x (C3 at t = 123.5, and the
# 1080p C3 rows), p99.9 1.15x (C3 at t = 123.5), max 1.26x (C1 at t = 50).
EMIS_TOL = {"max": (2.5e-4, 5e-6), "p999": (1.3e-4, 8e-7), "p99": (6.0e-5, 4.5e-7)}
# hdr relative error: mostly the texture unit's 1/256 filter weights on the smooth sky (1.3e-4 at every time, effects and
# camera), plus the emission at large |t|: census p99 <= 8.8e-5, p99.9 <= 1.29e-4, max <= 2.6e-4 (5.0e-4 at t = 123.5 in the
# 96x54 default-effects case).  Smallest margin 1.24x.
HDR_TOL = {"max": (2.5e-4, 3e-6), "p999": (1.6e-4, 0.0), "p99": (1.1e-4, 0.0)}
# |dense_samples difference| (samples past the 0.001 density gate): census <= 1 at t = 1, 2 at 12.5, 4 at 50 and 3 at 123.5.
# Bound 4 + 0.04 |t| (>= 1.5x where the census saw a difference).
DENSE_TOL = (4, 0.04)
# A TOUCHED flag can differ only where a sample sits at the density gate, which also moves dense_samples: the count of such
# pixels gets the dense_samples bound (the census saw none).
TOUCHED_TOL = DENSE_TOL
# A pixel whose TOUCHED flag differs has no dense sample on one side, so on the other every dense sample is within the
# rounding noise of the 0.001 gate.  Such a sample emits at most g^4 * 0.001 * disk_luminosity * (1 - exp(-0.001 opacity h))
# ~ 5 * 0.001 * 6 * 0.001 * 0.4 * 0.09 ~ 1e-6 (disk; dust is smaller): the floor allows 100 of them.
FLIP_EMIS_FLOOR = 1e-4


def emis_tol(t, q):
    return EMIS_TOL[q][0] + EMIS_TOL[q][1] * abs(t)


# ---- cases -----------------------------------------------------------------------------------------------------------
def _case(cid, sec, cam, flags, w, h, time=1.0, fx="off", prm=None, mask="all"):
    return {"id": cid, "section": sec, "cam": cam, "flags": flags, "w": w, "h": h, "time": time, "fx": fx,
            "prm": prm or {}, "mask": mask}


def time_cases():
    out = [_case(f"{cam}-{con}-t{t:g}", 1, cam, flags, 160, 90, time=t)
           for cam in ("C1", "C3") for con, flags in CONTRACTS.items() for t in TIMES]
    out.append(_case("C1-fmad-t123.5-default-effects-96x54", 1, "C1", CONTRACTS["fmad"], 96, 54, time=123.5, fx="default"))
    return out


def camera_cases():
    out = []
    for con, flags in CONTRACTS.items():
        for path in range(3):
            for t in PATH_TIMES:   # each path camera at its own clock as the frame time, as PathSequence couples them
                out.append(_case(f"path{path}-t{t:g}-{con}", 2, ("path", path, t), flags, 96, 54, time=t))
        for k in range(len(LENS_CAMS)):
            for j in range(LENS[2] ** 2):
                out.append(_case(f"lens{k}.{j}-{con}", 2, ("lens", k, j), flags, 96, 54))
        for name in POSES:
            out.append(_case(f"{name}-{con}", 2, ("pose", name), flags, 96, 54,
                             mask="medium" if name in POLE_POSES else "all"))
    return out


def effects_cases():
    f7 = CONTRACTS["fmad"]
    out = [_case(f"ca{a:g}", 3, "C2", f7, 160, 90, fx={"use_ca": 1, "ca_amount": a}) for a in (0.005, 0.01, 0.2)]
    out += [_case(f"vignette{v:g}", 3, "C1", f7, 160, 90, fx={"use_vignette": 1, "vignette_intensity": v}) for v in (0.4, 0.7, 2.0)]
    out += [_case(f"bloom{b:g}x{i:g}", 3, "C1", f7, 160, 90, fx={"use_bloom": 1, "bloom_threshold": b, "bloom_intensity": i})
            for b in (0.3, 0.8, 5.0) for i in (0.5, 2.0)]
    out += [_case(f"exposure{e:g}", 3, "C1", f7, 160, 90, prm={"exposure": e}) for e in (0.5, 1.7, 10.0)]
    out += [_case("lens-off", 3, "C1", f7, 160, 90, fx={"use_lens": 0, "distortion_amount": 0.6})]
    out += [_case(f"lens{k:g}", 3, "C1", f7, 160, 90, fx={"use_lens": 1, "distortion_amount": k}) for k in (0.0, 0.15, -0.3, 0.6)]
    return out


def fullsize_cases():
    out = []
    for (w, h, tag) in ((1920, 1080, "1080p"), (3840, 2160, "4k")):
        for cam in ("C0", "C3"):
            out.append(_case(f"{tag}-{cam}-fmad", 4, cam, CONTRACTS["fmad"], w, h, fx="default"))
    out.append(_case("4k-C3-strict", 4, "C3", CONTRACTS["strict"], 3840, 2160, fx="default"))
    return out


def all_cases():
    return time_cases() + camera_cases() + effects_cases() + fullsize_cases()


def _ids(cases):
    return [pytest.param(c, id=c["id"]) for c in cases]


# ---- rendering ---------------------------------------------------------------------------------------------------------
def camera(ora, spec):
    """the rrt Camera of a case (checked against the oracle's where both build one)"""
    import relativisticraytracer_b200 as rrt
    if isinstance(spec, str):
        return rrt.camera_state_from(*CAMERAS[spec])
    if spec[0] == "path":
        cg, _ = rrt.path_state(spec[1], spec[2])
        co, _ = ora.path_state(spec[1], spec[2])
        assert bytes(cg) == bytes(co), spec
        return cg
    if spec[0] == "lens":
        aperture, focus, ss = LENS
        return rrt.lens_cameras(rrt.camera_state_from(*LENS_CAMS[spec[1]]), aperture, focus, ss)[spec[2]]
    pos, yaw, pitch = POSES[spec[1]]
    cg = rrt.camera_state_from(pos, yaw, pitch)
    assert bytes(cg) == bytes(ora.camera_from(pos, yaw, pitch)), spec
    return cg


def effects(fx):
    import relativisticraytracer_b200 as rrt
    if isinstance(fx, str):
        return fx
    e = rrt.effects_off()
    for k, v in fx.items():
        setattr(e, k, v)
    return e


def _frame_dicts(f, g):
    """oracle Frame and GPU dict -> two dicts of the same planes, rgba in the planes' row order"""
    fo = {k: getattr(f, k) for k in ("hdr", "dir", "emis", "pos", "vel", "cls", "steps", "counters")}
    fo["rgba"] = f.rgba[::-1]
    go = {k: g[k] for k in ("hdr", "dir", "emis", "pos", "vel", "cls", "steps", "counters")}
    go["rgba"] = g["rgba"][::-1]
    return fo, go


def sample_rows(h, cls_touched_per_row, n_even):
    """first, last and middle rows; both sides of the 16x4 split-pipeline tile-row boundary (kTile16H = 4) nearest the row
    with the most disk / dust pixels; n_even evenly spaced rows"""
    b = max(4, int(round(int(np.argmax(cls_touched_per_row)) / 4.0)) * 4)
    rows = {0, h - 1, h // 2, b - 1, b}
    rows |= {int(round(y)) for y in np.linspace(0, h - 1, n_even + 2)[1:-1]}
    return sorted(rows)


def oracle_rows(ora, po, co, fo, sky_np, time, w, h, rows):
    """the oracle's planes of the given rows of a w x h frame, one single-threaded render per row on every core"""
    def one(y):
        ora.set_num_threads(1)        # this worker thread's OpenMP team; the rows run side by side
        f = ora.render(po, co, fo, sky_np, time, w, h, y, y + 1)
        part = {k: getattr(f, k)[y].copy() for k in ("hdr", "dir", "emis", "pos", "vel", "cls", "steps")}
        part["rgba"] = f.rgba[h - 1 - y].copy()      # the stored frame is row-flipped
        return part, f.counters

    with ThreadPoolExecutor(max_workers=max(1, min(len(rows), os.cpu_count() or 1))) as ex:
        res = list(ex.map(one, rows))
    out = {k: np.stack([p[k] for p, _ in res]) for k in res[0][0]}
    out["counters"] = {k: sum(c[k] for _, c in res) for k in res[0][1]}
    return out


def _row_counters(d):
    cls = d["cls"]
    return {"rk4_steps": int(d["steps"].astype(np.int64).sum()), "n_captured": int(((cls & 3) == 0).sum()),
            "n_exhausted": int(((cls & 4) != 0).sum()), "n_touched": int(((cls & 8) != 0).sum())}


def render_rows(gpu, ora, sky_np, c):
    """GPU frame at full size with its planes, and the oracle on sampled rows; returns (oracle, gpu) dicts of those rows"""
    import relativisticraytracer_b200 as rrt
    import torch
    from oracle import Camera as OraCamera
    w, h, t = c["w"], c["h"], c["time"]
    pg = rrt.default_params(spin_a=0.99, flags=c["flags"], **c["prm"])
    po = ora.default_params(spin_a=0.99, flags=c["flags"], **c["prm"])
    cg = camera(ora, c["cam"])
    co = ora.camera_from(*CAMERAS[c["cam"]])
    assert bytes(cg) == bytes(co)
    sky = gpu.create_sky(sky_np)
    planes = gpu.alloc_planes(w, h)
    out = gpu.render(pg, cg, rrt.default_effects(), sky, t, w, h, planes=planes)
    torch.cuda.synchronize()
    touched_rows = ((planes["cls"] & rrt.CLSF_TOUCHED) != 0).sum(dim=1).cpu().numpy()
    rows = sample_rows(h, touched_rows, EVEN_ROWS)
    idx = torch.tensor(rows, device=gpu.device)
    g = {k: v.index_select(0, idx).cpu().numpy() for k, v in planes.items()}      # only the sampled rows reach the host
    g["rgba"] = out.index_select(0, (h - 1) - idx).cpu().numpy()
    del planes, out
    sky.close()
    f = oracle_rows(ora, po, co, ora.default_effects(), sky_np, t, w, h, rows)
    f["counters"] = {k: f["counters"][k] for k in ROW_COUNTERS + ("n_touched", "dense_samples")}
    g["counters"] = _row_counters(g)
    assert _row_counters(f)["rk4_steps"] == f["counters"]["rk4_steps"]
    f["rows"] = g["rows"] = rows
    return f, g


def run_case(gpu, ora, sky_np, c):
    """(oracle, gpu) dicts of the case's planes (all rows, or the sampled rows of a full-size frame)"""
    if c["section"] == 4:
        return render_rows(gpu, ora, sky_np, c)
    f, g = render_pair(gpu, ora, sky_np, None, 0.99, c["flags"], c["w"], c["h"], time=c["time"], fx=effects(c["fx"]),
                       cam=camera(ora, c["cam"]), **c["prm"])
    return _frame_dicts(f, g)


# ---- comparison --------------------------------------------------------------------------------------------------------
def _q(a):
    a = np.asarray(a, np.float64).ravel()
    if a.size == 0:
        return {"max": 0.0, "p999": 0.0, "p99": 0.0}
    return {"max": float(a.max()), "p999": float(np.quantile(a, 0.999)), "p99": float(np.quantile(a, 0.99))}


def _rel(g, f):
    a, b = f[..., :3].astype(np.float64), g[..., :3].astype(np.float64)
    return (np.abs(b - a) / np.maximum(np.abs(a), 1e-3)).max(axis=-1)


def compare(c, f, g):
    """The exact part (names of what differs: must be empty) and the census numbers of the toleranced part."""
    exact_bad = [k for k in ("steps", "pos", "vel", "dir") if not np.array_equal(f[k], g[k], equal_nan=True)]
    if not np.array_equal((f["cls"] & 3) == 0, (g["cls"] & 3) == 0):
        exact_bad.append("cls:CAPTURED")
    if not np.array_equal(f["cls"] & 4, g["cls"] & 4):
        exact_bad.append("cls:EXHAUSTED")
    if not np.array_equal(f["rgba"][..., 3], g["rgba"][..., 3]):
        exact_bad.append("rgba:alpha")
    for k in (ROW_COUNTERS if c["section"] == 4 else EXACT_COUNTERS):
        if f["counters"][k] != g["counters"][k]:
            exact_bad.append(f"counter:{k}")
    flip = ((f["cls"] ^ g["cls"]) & 8) != 0
    medium = ((f["cls"] & 8) != 0) | ((g["cls"] & 8) != 0) | ((f["cls"] & 3) == 0) | ((g["cls"] & 3) == 0)
    mask = medium if c["mask"] == "medium" else np.ones_like(flip)
    emis = np.maximum(np.abs(f["emis"][..., :3]), np.abs(g["emis"][..., :3])).max(axis=-1)
    d8 = np.abs(f["rgba"][..., :3].astype(int) - g["rgba"][..., :3].astype(int)).max(axis=-1)
    m = {"id": c["id"], "section": c["section"], "time": c["time"], "pixels": int(flip.size), "exact_bad": exact_bad,
         "emis_rel": _q(_rel(g["emis"], f["emis"])[~flip]), "hdr_rel": _q(_rel(g["hdr"], f["hdr"])[mask]),
         "rgba_diff": _q(d8[mask]), "touched_flips": int(flip.sum()), "flip_emis_max": float(emis[flip].max()) if flip.any() else 0.0,
         "dense_samples_diff": int(g["counters"]["dense_samples"]) - int(f["counters"]["dense_samples"])
         if "dense_samples" in g["counters"] else None,     # not in a row sample: the GPU counts the whole frame
         "n_touched_diff": int(g["counters"]["n_touched"] - f["counters"]["n_touched"])}
    if "rows" in f:
        m["rows"] = f["rows"]
    return m, d8, mask


def _within(pair, t):
    return pair[0] + pair[1] * abs(t)


def check(c, f, g, rgba_max=1, emis=EMIS_TOL):
    """`emis`: the emission bounds, EMIS_TOL unless a case has measured bounds of its own"""
    m, d8, mask = compare(c, f, g)
    t = c["time"]
    assert not m["exact_bad"], m
    for q in ("max", "p999", "p99"):
        assert m["emis_rel"][q] <= _within(emis[q], t), (q, m)
        assert m["hdr_rel"][q] <= _within(HDR_TOL[q], t), (q, m)
    # a TOUCHED flag that differs is a sample at the 0.001 density gate: same trajectory (the steps / pos / vel planes are
    # exact above, pixel by pixel), no emission to speak of
    assert m["touched_flips"] <= _within(TOUCHED_TOL, t), m
    assert m["flip_emis_max"] <= FLIP_EMIS_FLOOR, m
    if m["dense_samples_diff"] is not None:
        assert abs(m["dense_samples_diff"]) <= _within(DENSE_TOL, t), m
    assert abs(m["n_touched_diff"]) <= _within(TOUCHED_TOL, t), m
    if rgba_max is not None:
        assert m["rgba_diff"]["max"] <= rgba_max, m
    return m, d8, mask


# ---- 1. time ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("c", _ids(time_cases()))
def test_times(gpu, ora, sky_smooth, c):
    f, g = run_case(gpu, ora, sky_smooth, c)
    check(c, f, g)


@pytest.mark.parametrize("flags", CONTRACTS.values(), ids=CONTRACTS.keys())
@pytest.mark.parametrize("cam", ["C1", "C3"])
def test_trajectory_does_not_depend_on_time(gpu, sky_smooth, cam, flags):
    """on the GPU alone: the planes and counters no medium can change are the same at every time"""
    import relativisticraytracer_b200 as rrt
    import torch
    prm, cg, sky = rrt.default_params(spin_a=0.99, flags=flags), rrt.camera_state_from(*CAMERAS[cam]), gpu.create_sky(sky_smooth)
    ref = None
    for t in TIMES:
        planes = gpu.alloc_planes(160, 90, names=("pos", "vel", "dir", "cls", "steps"))
        gpu.read_counters(reset=True)
        gpu.render(prm, cg, rrt.effects_off(), sky, t, 160, 90, planes=planes)
        torch.cuda.synchronize()
        cnt = gpu.read_counters()
        cur = {k: v.cpu().numpy() for k, v in planes.items()}
        cur["cls"] = np.stack([(cur["cls"] & 3) == 0, (cur["cls"] & 4) != 0])    # CAPTURED, EXHAUSTED
        cur["counters"] = [cnt[k] for k in EXACT_COUNTERS]
        if ref is None:
            ref = cur
        for k in cur:
            assert np.array_equal(cur[k], ref[k]), (t, k)
    sky.close()


# ---- 2. cameras -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("c", _ids(camera_cases()))
def test_cameras(gpu, ora, sky_smooth, c):
    f, g = run_case(gpu, ora, sky_smooth, c)
    m, _, mask = check(c, f, g)
    if c["cam"][0] == "lens":
        cam = camera(ora, c["cam"])
        assert abs(float(np.linalg.norm(np.array(cam.forward, np.float64))) - 1.0) > 1e-3   # not an orthonormal basis
    if c["cam"][0] == "pose" and c["cam"][1] in ("in-disk-slab", "in-dust-layer"):
        assert g["counters"]["n_touched"] > 0.5 * m["pixels"]
    if c["cam"][0] == "pose" and c["cam"][1] == "near-horizon":
        assert 0 < g["counters"]["n_captured"] < m["pixels"]
    if c["mask"] == "medium":
        assert mask.sum() > 0.05 * m["pixels"]


# ---- 3. post effects --------------------------------------------------------------------------------------------------
LUMA = np.array([0.2126, 0.7152, 0.0722])


@pytest.mark.parametrize("c", _ids(effects_cases()))
def test_effects(gpu, ora, sky_smooth, c):
    f, g = run_case(gpu, ora, sky_smooth, c)
    fx = c["fx"] if isinstance(c["fx"], dict) else {}
    bloom = fx.get("use_bloom", 0)
    m, d8, _ = check(c, f, g, rgba_max=None if bloom else 1)
    if bloom:
        # a pixel on the other side of the bloom threshold than the oracle's may differ by more than a count; only where the
        # oracle's luminance lies within the hdr tolerance of the threshold
        lum = f["hdr"][..., :3].astype(np.float64) @ LUMA
        off = d8 > 1
        thr = fx["bloom_threshold"]
        assert np.all(np.abs(lum[off] - thr) <= _within(HDR_TOL["max"], c["time"]) * max(thr, 1e-3)), (lum[off], m)
        assert m["rgba_diff"]["p999"] <= 1, m
    if fx.get("use_ca"):
        # some escaped pixels' R or B tap crosses the texture seam at phi = +-pi, so the wrap is exercised
        d = f["dir"].astype(np.float64)
        phi = np.arctan2(d[..., 2], d[..., 0])
        esc = (f["cls"] & 3) == 2
        a = fx["ca_amount"]
        assert np.sum(esc & ((phi + a > np.pi) | (phi - a < -np.pi))) > 0
    if fx.get("use_lens") and fx.get("distortion_amount") == 0.6:
        tu = np.float32(0.0) - np.float32(0.5)      # corner pixel (0, 0): u = tu * (1 + 0.6 * 2 tu^2) + 0.5 < 0
        assert tu * (1 + 0.6 * 2 * tu * tu) + 0.5 < 0


# ---- 4. rows of full-size frames --------------------------------------------------------------------------------------
@pytest.mark.parametrize("c", _ids(fullsize_cases()))
def test_fullsize_rows(gpu, ora, sky_smooth, c):
    f, g = run_case(gpu, ora, sky_smooth, c)
    m, _, _ = check(c, f, g)
    assert len(f["rows"]) >= EVEN_ROWS + 3
