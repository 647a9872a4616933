"""rrt_render_pano / Renderer.render_pano / PathSequence(projection="equirect") / rrt_record --pano: 360-degree
equirectangular panoramas.

The contract every test here leans on: pixel (x, y) of the w x h panorama equals pixel (1, 1) of the 2 x 2 rrt_render with
camera {pos, d, right, up}, d = pano_directions(cam, w, h)[y, x] -- the pinhole ray there is unit3(d) -- in every plane,
and in its byte when the vignette (the one effect that reads the pixel's image-plane position) is off.  So most checks are
exact equality: against those 2 x 2 renders for every tracer, against the fused panorama for the split passes, against
rrt_resolve of the large panorama for ss > 1, and against whole-frame panoramas for bands, streams and sequences."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from test_gpu_dof import TRACERS, _cams, _hdr, _np, _renderer, _same, env  # noqa: F401  (env: the module's contexts)
from test_gpu_oracle_reach import check

pytestmark = pytest.mark.gpu

PLANES = ("hdr", "dir", "emis", "pos", "vel", "cls", "steps")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _setup(env, tracer, spin=0.99, **fx_over):
    """(renderer, prm, fx, sky) of a tracer; lens distortion (refused by render_pano) and vignette off unless overridden."""
    import relativisticraytracer_b200 as rrt
    ctxs, skies = env
    ctx, pipeline, flags = TRACERS[tracer]
    r = ctxs[ctx]
    r.set_pipeline(pipeline)
    fx = rrt.default_effects(**{"use_lens": 0, "use_vignette": 0, **fx_over})
    return r, rrt.default_params(spin_a=spin, flags=flags, exposure=0.8), fx, skies[ctx]["small"]


def _pano(r, prm, cam, fx, sky, w, h, time=1.0, **kw):
    """render_pano with every plane: dict of numpy planes plus "rgba" in the planes' row order (zenith last)."""
    pl = r.alloc_planes(w, h)
    out = r.render_pano(prm, cam, fx, sky, time, w, h, planes=pl, **kw)
    got = {k: v for k, v in zip(PLANES + ("rgba",), _np(*[pl[k] for k in PLANES], out))}
    got["rgba"] = got["rgba"][::-1]
    return got


def _pinhole_pixels(r, prm, cam, fx, sky, w, h, time=1.0):
    """Pixel (1, 1) of the 2 x 2 rrt_render with camera {pos, d, right, up} for every pixel of a w x h panorama, as (h, w)
    planes and "rgba" in the planes' row order."""
    import relativisticraytracer_b200 as rrt
    import torch
    n = w * h
    d = rrt.pano_directions(cam, w, h).reshape(n, 3)
    cams = (rrt.Camera * n)()
    arr = np.frombuffer(cams, np.float32).reshape(n, 12)
    arr[:, 0:3] = np.array(cam.pos, np.float32)
    arr[:, 3:6] = d
    arr[:, 6:9] = np.array(cam.right, np.float32)
    arr[:, 9:12] = np.array(cam.up, np.float32)
    planes = r.alloc_planes(2, 2 * n)                # frame k: rows 2k and 2k + 1
    out = torch.zeros((2 * n, 2, 4), dtype=torch.uint8, device=r.device)
    st = r._stream(None)
    for k in range(n):
        pl = rrt.Planes()
        for name in PLANES:
            t = planes[name]
            setattr(pl, name, t.data_ptr() + k * 4 * t.element_size() * (t.numel() // (4 * n)))
        r._check(r._lib.rrt_render(r._ctx, C.byref(prm), C.byref(cams[k]), C.byref(fx), C.c_uint64(sky.texture), float(time),
                                   2, 2, None, C.c_void_p(out.data_ptr() + 16 * k), rrt.OUT_FRAME, C.byref(pl), st))
    got = dict(zip(PLANES + ("rgba",), _np(*[planes[k] for k in PLANES], out)))
    res = {k: v.reshape((n, 2, 2) + v.shape[2:])[:, 1, 1].reshape((h, w) + v.shape[2:]) for k, v in got.items() if k != "rgba"}
    res["rgba"] = got["rgba"].reshape(n, 2, 2, 4)[:, 0, 1].reshape(h, w, 4)   # image row 1 is buffer row 0
    return res


def _equal(got, want, tag, rgba=True):
    for k in PLANES + (("rgba",) if rgba else ()):
        a, b = got[k], want[k]
        assert a.shape == b.shape and np.array_equal(a, b), f"{tag}: {k} differs at {int(np.sum(a != b))} elements"


@pytest.mark.parametrize("tracer", list(TRACERS))
@pytest.mark.parametrize("spin", [0.99, 0.0])
@pytest.mark.parametrize("cam", ["C0", "C1", "C2", "C3"])
def test_pinhole_equivalence_every_tracer(env, tracer, spin, cam):
    """Every pixel of a 48 x 24 and of an odd 37 x 19 panorama (a packed pair's parked half, the poles, the seam)."""
    r, prm, fx, sky = _setup(env, tracer, spin)
    c = _cams([cam])[0]
    for w, h in ((48, 24), (37, 19)):
        _equal(_pano(r, prm, c, fx, sky, w, h), _pinhole_pixels(r, prm, c, fx, sky, w, h), f"{tracer} a={spin} {cam} {w}x{h}")


@pytest.mark.parametrize("tracer", ["split_packed", "packed_fused"])
def test_pinhole_equivalence_with_effects(env, tracer):
    """Bloom, chromatic aberration, another exposure; with the vignette on every plane still agrees (the byte does not:
    the vignette darkens the panorama's own edges)."""
    import relativisticraytracer_b200 as rrt
    r, prm, fx, sky = _setup(env, tracer, use_bloom=1, bloom_threshold=0.3, use_ca=1, ca_amount=0.01)
    prm.exposure = 1.7
    c = _cams(["C1"])[0]
    _equal(_pano(r, prm, c, fx, sky, 40, 20, time=7.25), _pinhole_pixels(r, prm, c, fx, sky, 40, 20, time=7.25), tracer)
    fxv = rrt.default_effects(use_lens=0)
    _equal(_pano(r, prm, c, fxv, sky, 40, 20), _pinhole_pixels(r, prm, c, fxv, sky, 40, 20), f"{tracer} vignette", rgba=False)


def test_cpu_oracle(env, ora, sky_smooth):
    """A 64 x 32 disk + dust panorama against the CPU oracle port, pixel by pixel through the 2 x 2 equivalence (with
    right = up = 0 every ray of the oracle's 2 x 2 frame is the pixel's, so its counters are twice the pixel's).
    Trajectories, classes and counters exactly; emission, hdr and bytes within test_gpu_oracle_reach's bounds."""
    import relativisticraytracer_b200 as rrt
    from oracle import Camera as OraCamera, Effects as OraEffects
    r, _, _, _ = _setup(env, "split_packed")
    w, h, flags = 64, 32, 3
    prm, fx = rrt.default_params(spin_a=0.99, flags=flags), rrt.effects_off()
    sky = env[1]["auto"]["smooth"]   # the sky the bounds were measured on
    cam = _cams(["C0"])[0]
    r.read_counters(reset=True)
    g = _pano(r, prm, cam, fx, sky, w, h)
    g["counters"] = r.read_counters(reset=True)
    po, fo = ora.default_params(spin_a=0.99, flags=flags), OraEffects.from_buffer_copy(bytes(fx))
    d = rrt.pano_directions(cam, w, h)
    f = {k: np.zeros_like(g[k]) for k in PLANES + ("rgba",)}
    f["counters"] = {}
    for y in range(h):
        for x in range(w):
            c = OraCamera.from_buffer_copy(bytes(cam))
            c.forward[:] = [float(v) for v in d[y, x]]
            c.right[:] = [0.0, 0.0, 0.0]
            c.up[:] = [0.0, 0.0, 0.0]
            fr = ora.render(po, c, fo, sky_smooth, 1.0, 2, 2, y0=1, y1=2)
            for k in PLANES:
                f[k][y, x] = getattr(fr, k)[1, 1]
            f["rgba"][y, x] = fr.rgba[0, 1]
            for k, v in fr.counters.items():
                f["counters"][k] = f["counters"].get(k, 0) + v
    for k, v in f["counters"].items():
        assert v % 2 == 0, k
        f["counters"][k] = v // 2
    assert f["counters"]["disk_evals"] > 0 and f["counters"]["dust_evals"] > 0 and f["counters"]["n_captured"] > 0
    assert np.array_equal(f["cls"], g["cls"])
    check({"id": "pano", "section": 0, "time": 1.0, "mask": "all"}, f, g)


@pytest.mark.parametrize("trace", ["auto", "scalar"])
@pytest.mark.parametrize("max_passes", [32, 1])
def test_split_passes_redo_list_and_sweep(env, sky_small, trace, max_passes):
    """A 64 KiB sample pool: several passes, tiles handed to the next pass and to the closing fused sweep, every one of them
    re-creating its rays from the panorama's table.  Frames, planes and counters equal the fused panorama bit for bit."""
    import relativisticraytracer_b200 as rrt
    r0, _, fx, sky0 = _setup(env, "fused_media")
    prm = rrt.default_params(spin_a=0.99, flags=7)
    cam = _cams(["C3"])[0]
    w, h = 256, 128
    r0.read_counters(reset=True)
    want = _pano(r0, prm, cam, fx, sky0, w, h)
    want_cnt = r0.read_counters(reset=True)
    r = _renderer(trace)
    try:
        sky = r.create_sky(sky_small)
        r.set_pipeline("split")
        r.set_sample_pool(64 * 1024, max_passes)
        worked = swept = 0
        for rep in range(2):   # the pass count adapts from frame to frame
            r.read_counters(reset=True)
            _equal(_pano(r, prm, cam, fx, sky, w, h), want, f"{trace} {max_passes} passes, frame {rep}")
            assert r.read_counters(reset=True) == want_cnt
            st = r.split_stats()
            worked, swept = max(worked, st["passes_worked"]), max(swept, st["tiles_swept"])
        assert worked > 1 or swept > 0, "the small pool was expected to cut the frame into passes"
        if max_passes == 1:
            assert swept > 0, "one pass of a 64 KiB pool was expected to leave tiles to the closing sweep"
        sky.close()
    finally:
        r.close()


def _resolve_of_large(r, prm, cam, fx, sky, w, h, ss, **kw):
    """rrt_resolve(ss) of the hdr plane of the ss*w x ss*h panorama: (frame, hdr)."""
    hi = _hdr(r, ss * w, ss * h)
    r.render_pano(prm, cam, fx, sky, 1.0, ss * w, ss * h, planes={"hdr": hi})
    hdr = _hdr(r, w, h)
    out = r.resolve(prm, fx, hi, ss, w, h, hdr_out=hdr, **kw)
    return _np(out, hdr)


def _pano_ss(r, prm, cam, fx, sky, w, h, ss, **kw):
    hdr = _hdr(r, w, h)
    out = r.render_pano(prm, cam, fx, sky, 1.0, w, h, ss=ss, planes={"hdr": hdr}, **kw)
    return _np(out, hdr)


@pytest.mark.parametrize("tracer", ["split_packed", "packed_fused", "scalar_fused", "split_strict"])
@pytest.mark.parametrize("ss", [2, 3])
def test_supersampled_is_resolve_of_large_panorama(env, tracer, ss):
    r, prm, fx, sky = _setup(env, tracer, use_vignette=1)
    for cam in _cams(["C0", "C3"]):
        _same(_pano_ss(r, prm, cam, fx, sky, 37, 19, ss), _resolve_of_large(r, prm, cam, fx, sky, 37, 19, ss), f"{tracer} ss={ss}")
    # the frame alone (no hdr plane) is the same frame
    cam = _cams(["C1"])[0]
    want = _resolve_of_large(r, prm, cam, fx, sky, 24, 12, ss)[0]
    assert np.array_equal(_np(r.render_pano(prm, cam, fx, sky, 1.0, 24, 12, ss=ss))[0], want)


@pytest.mark.parametrize("layout", ["frame", "packed"])
@pytest.mark.parametrize("ss", [1, 2])
def test_bands(env, layout, ss):
    """Each band writes exactly its rows (the others keep a sentinel) and its hdr pixels only; the union of the bands is the
    full panorama."""
    import relativisticraytracer_b200 as rrt
    import torch
    from relativisticraytracer_b200.parallel import band_rows_of
    r, prm, fx, sky = _setup(env, "split_packed")
    w, h = 67, 41
    lay = rrt.OUT_FRAME if layout == "frame" else rrt.OUT_PACKED
    cam = _cams(["C0"])[0]
    full, full_hdr = _pano_ss(r, prm, cam, fx, sky, w, h, ss)
    for nranks in (2, 3):
        for group in (1, 8):
            union = np.full((h, w, 4), 77, np.uint8)
            for rank in range(nranks):
                band = rrt.Band(rank, nranks, group)
                rows = band_rows_of(rank, nranks, group, h)
                own = (h - 1 - rows) if lay == rrt.OUT_FRAME else np.arange(len(rows))
                out = torch.full((h, w, 4), 77, dtype=torch.uint8, device=r.device)
                hdr = _hdr(r, w, h, float("nan"))
                r.render_pano(prm, cam, fx, sky, 1.0, w, h, ss=ss, band=band, out=out, layout=lay, planes={"hdr": hdr})
                frame, hdr = _np(out, hdr)
                tag = f"{layout} ss={ss} band {rank}/{nranks}x{group}"
                assert (np.delete(frame, own, axis=0) == 77).all(), f"{tag}: rows outside the band were written"
                assert np.isnan(np.delete(hdr, rows, axis=0)).all(), f"{tag}: hdr outside the band was written"
                assert np.array_equal(hdr[rows], full_hdr[rows]), tag
                union[h - 1 - rows] = frame[own]
            assert np.array_equal(union, full), f"{layout} ss={ss} {nranks}x{group}: union of the bands"


@pytest.mark.parametrize("tracer", ["split_packed", "packed_fused", "fused_media", "split_scalar"])
@pytest.mark.parametrize("ss", [1, 2])
def test_counters_and_launches(env, tracer, ss):
    """rk4_steps and the class counts are the sums over the traced panorama's planes; launches are rrt_render's (the split
    pipeline's from its bookkeeping: 3 per pass + 1), + 1 for the resolve when ss > 1."""
    import relativisticraytracer_b200 as rrt
    r, prm, fx, sky = _setup(env, tracer)
    w, h = 61, 37
    cam = _cams(["C2"])[0]
    pl = r.alloc_planes(ss * w, ss * h, ("steps", "cls"))
    r.render_pano(prm, cam, fx, sky, 1.0, ss * w, ss * h, planes=pl)
    steps, cls = _np(pl["steps"], pl["cls"])
    r.read_counters(reset=True)
    l0 = r.kernel_launches()
    if ss == 1:
        r.render_pano(prm, cam, fx, sky, 1.0, w, h, planes=r.alloc_planes(w, h, ("steps", "cls")))
    else:
        _pano_ss(r, prm, cam, fx, sky, w, h, ss)
    launches = r.kernel_launches() - l0
    got = r.read_counters(reset=True)
    traced = 3 * r.split_stats()["passes_enqueued"] + 1 if tracer.startswith("split") else 1
    assert launches == traced + (ss > 1)
    assert got["rk4_steps"] == int(steps.astype(np.int64).sum()) > 0
    captured = (cls & rrt.CLS_MASK) == rrt.CLS_CAPTURED
    exhausted = (cls & rrt.CLSF_EXHAUSTED) != 0
    assert got["n_captured"] == captured.sum() > 0
    assert got["n_exhausted"] == exhausted.sum()
    assert got["n_escaped"] == (~captured & ~exhausted).sum() > 0
    assert got["n_touched"] == ((cls & rrt.CLSF_TOUCHED) != 0).sum()
    if not tracer.startswith("split"):   # rrt_render / rrt_render_ss of the pinhole frame launch as many kernels
        l0 = r.kernel_launches()
        if ss == 1:
            r.render(prm, cam, fx, sky, 1.0, w, h)
        else:
            r.render_ss(prm, cam, fx, sky, 1.0, w, h, ss)
        assert r.kernel_launches() - l0 == launches


def test_two_streams(env):
    import torch
    r, prm, fx, sky = _setup(env, "split_packed")
    w, h = 96, 48
    a, b = _cams(["C1", "C3"])
    want = [_pano_ss(r, prm, a, fx, sky, w, h, 1), _pano_ss(r, prm, b, fx, sky, w, h, 2)]
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    hdrs = [_hdr(r, w, h) for _ in range(4)]
    torch.cuda.synchronize()
    outs = []
    for k in range(4):   # interleaved: each call is enqueued while the other stream's may still run, on one scratch pool
        cam, ss, st = (a, 1, s1) if k % 2 == 0 else (b, 2, s2)
        with torch.cuda.stream(st):
            outs.append((r.render_pano(prm, cam, fx, sky, 1.0, w, h, ss=ss, planes={"hdr": hdrs[k]}, stream=st), hdrs[k]))
    torch.cuda.synchronize()
    for k, (out, hdr) in enumerate(outs):
        _same(_np(out, hdr), want[k % 2], f"stream call {k}")


@pytest.mark.parametrize("tracer", ["split_packed", "scalar_fused"])
def test_reshade(env, sky_smooth, tracer):
    """rrt_shade from a panorama's planes with another sky, exposure and effects is the panorama rendered with them."""
    import relativisticraytracer_b200 as rrt
    from relativisticraytracer_b200 import TRACE_PLANES
    r, prm, fx, sky = _setup(env, tracer)
    ctx = TRACERS[tracer][0]
    sky2 = env[1][ctx]["smooth"]
    w, h = 64, 32
    cam = _cams(["C0"])[0]
    traced = r.alloc_planes(w, h, TRACE_PLANES)
    r.render_pano(prm, cam, fx, sky, 1.0, w, h, planes=traced)
    prm2 = rrt.default_params(spin_a=0.99, flags=prm.flags, exposure=2.1)
    fx2 = rrt.default_effects(use_lens=0, use_vignette=1, vignette_intensity=0.9, use_ca=1, ca_amount=0.02, bloom_threshold=0.4)
    hdr = _hdr(r, w, h)
    got = _np(r.shade(prm2, fx2, sky2, traced, w, h, hdr_out=hdr), hdr)
    hdr2 = _hdr(r, w, h)
    want = _np(r.render_pano(prm2, cam, fx2, sky2, 1.0, w, h, planes={"hdr": hdr2}), hdr2)
    _same(got, want, f"{tracer} re-shaded")


@pytest.mark.parametrize("flags", [0, 4])
def test_flat_space_direction(env, flags):
    """No hole, no medium: rays go straight, so the exit direction is the panorama's unit3(d) (this pins the projection's
    orientation against the sky map)."""
    import relativisticraytracer_b200 as rrt
    r = env[0]["auto"]
    r.set_pipeline("auto")
    sky = env[1]["auto"]["small"]
    prm = rrt.default_params(event_horizon=0.0, flags=flags)
    w, h = 48, 24
    for cam in _cams(["C0", "C2"]):
        pl = r.alloc_planes(w, h, ("dir", "cls"))
        r.render_pano(prm, cam, rrt.effects_off(), sky, 1.0, w, h, planes=pl)
        d, cls = _np(pl["dir"], pl["cls"])
        assert ((cls & rrt.CLS_MASK) == rrt.CLS_ESCAPED).all()
        want = rrt.pano_directions(cam, w, h).astype(np.float64)
        want /= np.linalg.norm(want, axis=-1, keepdims=True)
        assert np.abs(d[..., :3] - want).max() <= 1e-6


def test_errors(env):
    """RRT_ERR_BAD_ARG with nothing launched or counted: lens distortion, ss outside 1..8, a plane other than hdr at ss > 1,
    and what rrt_render / rrt_render_ss refuse."""
    import relativisticraytracer_b200 as rrt
    import torch
    r, prm, fx, sky = _setup(env, "split_packed")
    w, h = 32, 16
    frame = torch.empty((h, w, 4), dtype=torch.uint8, device=r.device)
    planes = r.alloc_planes(8 * w, 8 * h)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call(ss=1, w_=w, h_=h, band=None, d_out=C.c_void_p(frame.data_ptr()), layout=rrt.OUT_FRAME, p=prm, f=fx, pl=None,
             tex=sky.texture, cam=_cams(["C1"])[0]):
        pls = None
        if pl is not None:
            pls = rrt.Planes()
            for k in pl:
                setattr(pls, k, planes[k].data_ptr())
        return r._lib.rrt_render_pano(r._ctx, C.byref(p), C.byref(cam) if cam is not None else None, C.byref(f) if f is not None else None,
                                      C.c_uint64(tex), 1.0, w_, h_, ss, C.byref(band) if band is not None else None, d_out, layout,
                                      C.byref(pls) if pls is not None else None, st)

    r.read_counters(reset=True)
    l0 = r.kernel_launches()
    for bad in (dict(f=rrt.default_effects()), dict(f=rrt.default_effects(use_lens=1, distortion_amount=0.0)),
                dict(ss=0), dict(ss=9), dict(ss=-1), dict(ss=2, pl=("hdr", "dir")), dict(ss=2, pl=("cls",)), dict(ss=3, pl=("steps",)),
                dict(d_out=None), dict(d_out=None, ss=2), dict(w_=0), dict(h_=-3), dict(ss=8, w_=1 << 28),
                dict(w_=1 << 16, h_=1 << 15), dict(band=rrt.Band(3, 3, 8)), dict(ss=8, w_=1 << 16, h_=1 << 12, band=rrt.Band(0, 1, 1)),
                dict(layout=7), dict(p=rrt.default_params(max_steps=-1)), dict(tex=0), dict(cam=None), dict(f=None)):
        assert call(**bad) == rrt._capi.ERR_BAD_ARG, bad
    assert r.kernel_launches() == l0
    assert all(v == 0 for v in r.read_counters(reset=True).values())
    # the accepted edges: every plane at ss = 1, the hdr plane alone at ss > 1, planes without a frame
    assert call(pl=PLANES) == 0 and call(ss=2, pl=("hdr",)) == 0 and call(d_out=None, pl=("vel",)) == 0
    torch.cuda.synchronize()
    with pytest.raises(rrt.RrtError):
        r.render_pano(prm, _cams(["C0"])[0], rrt.default_effects(), sky, 1.0, w, h)


def test_path_sequence_and_recorder(env, sky_small, tmp_path):
    import relativisticraytracer_b200 as rrt
    from relativisticraytracer_b200.parallel import PathSequence
    r, prm, fx, sky = _setup(env, "split_packed")
    w, h, n, path = 96, 48, 4, 0
    p = str(tmp_path / "pano.rgba")
    seq = PathSequence(r, w, h, depth=2, ss=2, projection="equirect")
    with rrt.FrameSink(p, w, h) as sink:
        done, _ = seq.render(path, n, prm, fx, sky, fps=24.0, sink=sink)
    assert done == n
    raw = np.fromfile(p, np.uint8).reshape(n, h, w, 4)
    for k in range(1, n + 1):
        t = rrt.path_clock(k, 24.0)
        cam, _ = rrt.path_state(path, t)
        assert np.array_equal(raw[k - 1], _np(r.render_pano(prm, cam, fx, sky, t, w, h, ss=2))[0]), k
    # rrt_record --pano: the recorder's default parameters and effects, less lens distortion and vignette
    binary = os.path.join(ROOT, "relativisticraytracer_b200", "rrt_record")
    sky_file, out = str(tmp_path / "sky.rgba"), str(tmp_path / "rec.rgba")
    sky_small.tofile(sky_file)
    res = subprocess.run([binary, str(path), str(n), str(w), str(h), out, "--pano", "--spin", "0.99", "--sky-raw", sky_file,
                          str(sky_small.shape[1]), str(sky_small.shape[0])], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    rec = np.fromfile(out, np.uint8).reshape(n, h, w, 4)
    sky2 = r.create_sky(sky_small)
    prm2, fx2 = rrt.default_params(spin_a=0.99), rrt.default_effects(use_lens=0, use_vignette=0)
    for k in range(1, n + 1):
        t = rrt.path_clock(k, 24.0)
        cam, _ = rrt.path_state(path, t)
        assert np.array_equal(rec[k - 1], _np(r.render_pano(prm2, cam, fx2, sky2, t, w, h))[0]), k
    sky2.close()
