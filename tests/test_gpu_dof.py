"""rrt_render_dof / Renderer.render_dof / lens_cameras / PathSequence(aperture=): depth of field, each sub-sample of a pixel
traced from its own camera.

Sub-sample (i, j) of output pixel (x, y) is pixel (ss*x + i, ss*y + j) of the ss*w x ss*h rrt_render with cams[j*ss + i], and
the pixel is rrt_resolve's mean of its sub-samples.  So everything here is exact equality: the expected ss*w x ss*h hdr plane
is put together in torch from ss*ss whole renders, one per camera, and rrt_resolve of it must give render_dof's bytes and
hdr values -- for every tracer (fused scalar / packed / with media, split with either trace kernel, several passes, the
closing sweep), bands, sizes and streams."""
import ctypes as C
import os

import numpy as np
import pytest

from parity import CAMERAS

pytestmark = pytest.mark.gpu

VARIANTS = [   # (sky, exposure, effect fields changed from the defaults), as in test_gpu_supersample.py
    ("small", 0.8, {}),
    ("smooth", 1.7, dict(use_bloom=0, use_vignette=1, vignette_intensity=0.7, use_ca=1, ca_amount=0.01)),
    ("small", 0.5, dict(bloom_threshold=0.3)),
]
# (context, pipeline, flags): the tracer each launch goes through
TRACERS = {
    "packed_fused": ("auto", "auto", 4),     # FMAD, no medium: render_kernel_p
    "scalar_fused": ("auto", "auto", 0),     # strict, no medium: render_kernel
    "fused_media": ("auto", "fused", 7),     # render_kernel with the media inline
    "split_packed": ("auto", "auto", 7),     # trace_kernel_p + media + fold
    "split_scalar": ("scalar", "auto", 7),   # trace_kernel + media + fold (FMAD contract, scalar tracer)
    "split_strict": ("auto", "auto", 3),     # trace_kernel under the strict contract
}


def _renderer(trace):
    """RRT_TRACE (scalar | packed | auto) is read when a context is created."""
    import relativisticraytracer_b200 as rrt
    old = os.environ.get("RRT_TRACE")
    os.environ["RRT_TRACE"] = trace
    try:
        return rrt.Renderer(0)
    finally:
        if old is None:
            os.environ.pop("RRT_TRACE", None)
        else:
            os.environ["RRT_TRACE"] = old


@pytest.fixture(scope="module")
def env(built, sky_small, sky_smooth):
    """Contexts of their own (pipeline, counters and launch count are per context) and the two skies."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    ctxs = {"auto": _renderer("auto"), "scalar": _renderer("scalar")}
    skies = {k: {"small": r.create_sky(sky_small), "smooth": r.create_sky(sky_smooth)} for k, r in ctxs.items()}
    yield ctxs, skies
    for k, r in ctxs.items():
        for s in skies[k].values():
            s.close()
        r.close()


def _setup(env, tracer, spin=0.99, variant=VARIANTS[0], **fx_over):
    """(renderer, prm, fx, sky) of a tracer."""
    import relativisticraytracer_b200 as rrt
    ctxs, skies = env
    ctx, pipeline, flags = TRACERS[tracer]
    r = ctxs[ctx]
    r.set_pipeline(pipeline)
    sky, exposure, over = variant
    return r, rrt.default_params(spin_a=spin, flags=flags, exposure=exposure), rrt.default_effects(**{**fx_over, **over}), skies[ctx][sky]


def _cams(names):
    import relativisticraytracer_b200 as rrt
    return [rrt.camera_state_from(*CAMERAS[n]) for n in names]


def _mix9():
    """Nine different cameras: the four BASELINE cameras and lens cameras of two of them."""
    import relativisticraytracer_b200 as rrt
    c0, c1, c2, c3 = _cams(["C0", "C1", "C2", "C3"])
    return [c0, c1, c2, c3] + rrt.lens_cameras(c1, 0.8, 20.0, 2)[:3] + rrt.lens_cameras(c0, 1.5, 45.0, 3)[7:9]


def _hdr(r, w, h, fill=0.0):
    import torch
    return torch.full((h, w, 4), fill, dtype=torch.float32, device=r.device)


def _np(*ts):
    import torch
    torch.cuda.synchronize()
    return tuple(t.cpu().numpy() for t in ts)


def _expected_hi(r, prm, cams, fx, sky, w, h, ss, time=1.0, planes=()):
    """The ss*w x ss*h hdr plane render_dof traces, put together from ss*ss renders: sub-sample (i, j) from the render with
    cams[j*ss + i].  With `planes`, also those planes of the renders (dict name -> list per camera)."""
    hi = _hdr(r, ss * w, ss * h)
    extra = {n: [] for n in planes}
    for k, cam in enumerate(cams):
        i, j = k % ss, k // ss
        pl = r.alloc_planes(ss * w, ss * h, ("hdr",) + tuple(planes))
        r.render(prm, cam, fx, sky, time, ss * w, ss * h, planes=pl)
        hi[j::ss, i::ss] = pl["hdr"][j::ss, i::ss]
        for n in planes:
            extra[n].append(pl[n])
    return (hi, extra) if planes else hi


def _resolve(r, prm, fx, hi, ss, w, h, **kw):
    hdr = _hdr(r, w, h)
    out = r.resolve(prm, fx, hi, ss, w, h, hdr_out=hdr, **kw)
    return _np(out, hdr)


def _dof(r, prm, cams, fx, sky, w, h, ss, time=1.0, **kw):
    hdr = _hdr(r, w, h)
    out = r.render_dof(prm, cams, fx, sky, time, w, h, ss, hdr_out=hdr, **kw)
    return _np(out, hdr)


def _same(got, want, tag):
    for name, a, b in zip(("frame", "hdr"), got, want):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), f"{tag}: {name} differs on {np.sum(a != b)} elements"


def _check(r, prm, cams, fx, sky, w, h, ss, tag, **kw):
    want = _resolve(r, prm, fx, _expected_hi(r, prm, cams, fx, sky, w, h, ss), ss, w, h)
    _same(_dof(r, prm, cams, fx, sky, w, h, ss, **kw), want, tag)
    return want


@pytest.mark.parametrize("tracer", list(TRACERS))
@pytest.mark.parametrize("spin", [0.99, 0.0])
def test_different_cameras_every_tracer(env, tracer, spin):
    """Four BASELINE cameras at ss = 2 and a nine-camera mix at ss = 3: an indexing slip shows at once."""
    r, prm, fx, sky = _setup(env, tracer, spin)
    _check(r, prm, _cams(["C0", "C1", "C2", "C3"]), fx, sky, 61, 37, 2, f"{tracer} a={spin} ss=2")
    _check(r, prm, _mix9(), fx, sky, 43, 29, 3, f"{tracer} a={spin} ss=3")


@pytest.mark.parametrize("cam", ["C0", "C1"])
@pytest.mark.parametrize("ss", [2, 4])
@pytest.mark.parametrize("tracer", ["split_packed", "packed_fused", "fused_media"])
def test_thin_lens(env, cam, ss, tracer):
    import relativisticraytracer_b200 as rrt
    r, prm, fx, sky = _setup(env, tracer)
    cams = rrt.lens_cameras(_cams([cam])[0], 0.5, 60.0, ss)
    _check(r, prm, cams, fx, sky, 96, 54, ss, f"{cam} ss={ss} {tracer}")


@pytest.mark.parametrize("tracer", list(TRACERS))
def test_equal_cameras_is_render_ss_and_ss1_is_render(env, tracer):
    r, prm, fx, sky = _setup(env, tracer)
    cam = _cams(["C1"])[0]
    w, h = 67, 41
    for ss in (2, 3):
        hdr = _hdr(r, w, h)
        want = _np(r.render_ss(prm, cam, fx, sky, 1.0, w, h, ss, hdr_out=hdr), hdr)
        _same(_dof(r, prm, [cam] * (ss * ss), fx, sky, w, h, ss), want, f"{tracer} ss={ss} equal cameras")
    for c in _cams(["C0", "C3"]):
        hdr = _hdr(r, w, h)
        want = _np(r.render(prm, c, fx, sky, 1.0, w, h, planes={"hdr": hdr}), hdr)
        _same(_dof(r, prm, [c], fx, sky, w, h, 1), want, f"{tracer} ss=1")


@pytest.mark.parametrize("trace", ["auto", "scalar"])
@pytest.mark.parametrize("pool_kib,max_passes", [(4 * 1024, 32), (256, 3), (64, 1)])
def test_passes_redo_list_and_sweep(env, sky_small, trace, pool_kib, max_passes):
    """A sample pool small enough to cut the frame into passes, give tiles up to the next pass and leave some to the closing
    fused sweep: every one of them re-creates its rays from their own cameras."""
    import relativisticraytracer_b200 as rrt
    r0, prm, fx, sky0 = _setup(env, "split_packed")
    cams = rrt.lens_cameras(_cams(["C3"])[0], 0.3, 8.0, 2)
    w, h, ss = 128, 72, 2
    want = _resolve(r0, prm, fx, _expected_hi(r0, prm, cams, fx, sky0, w, h, ss), ss, w, h)
    r = _renderer(trace)
    try:
        sky = r.create_sky(sky_small)
        r.set_pipeline("split")
        r.set_sample_pool(pool_kib * 1024, max_passes)
        worked = swept = 0
        for rep in range(2):   # the pass count adapts from frame to frame
            _same(_dof(r, prm, cams, fx, sky, w, h, ss), want, f"{trace} pool {pool_kib} KiB, {max_passes} passes, frame {rep}")
            st = r.split_stats()
            worked, swept = max(worked, st["passes_worked"]), max(swept, st["tiles_swept"])
        assert worked > 1 or swept > 0, "the small pool was expected to cut the frame into passes"
        sky.close()
    finally:
        r.close()


@pytest.mark.parametrize("k", range(len(VARIANTS)))
@pytest.mark.parametrize("lens", [1, 0])
def test_shading_variants_and_lens_distortion(env, k, lens):
    import relativisticraytracer_b200 as rrt
    r, prm, fx, sky = _setup(env, "split_packed", variant=VARIANTS[k], use_lens=lens)
    _check(r, prm, rrt.lens_cameras(_cams(["C3"])[0], 0.5, 10.0, 2), fx, sky, 61, 37, 2, f"variant {k} lens={lens}")


@pytest.mark.parametrize("layout", ["frame", "packed"])
def test_bands(env, layout):
    """Each band writes exactly its rows (the others keep a sentinel) and its hdr pixels only; the union of the bands is the
    full frame."""
    import relativisticraytracer_b200 as rrt
    import torch
    from relativisticraytracer_b200.parallel import band_rows_of
    r, prm, fx, sky = _setup(env, "split_packed")
    w, h, ss = 67, 41, 2
    lay = rrt.OUT_FRAME if layout == "frame" else rrt.OUT_PACKED
    cams = _cams(["C0", "C1", "C2", "C3"])
    full, full_hdr = _check(r, prm, cams, fx, sky, w, h, ss, "full frame")
    for nranks in (2, 3):
        for group in (1, 8):
            union = np.full((h, w, 4), 77, np.uint8)
            for rank in range(nranks):
                band = rrt.Band(rank, nranks, group)
                rows = band_rows_of(rank, nranks, group, h)
                own = (h - 1 - rows) if lay == rrt.OUT_FRAME else np.arange(len(rows))
                out = torch.full((h, w, 4), 77, dtype=torch.uint8, device=r.device)
                hdr = _hdr(r, w, h, float("nan"))
                r.render_dof(prm, cams, fx, sky, 1.0, w, h, ss, band=band, out=out, layout=lay, hdr_out=hdr)
                frame, hdr = _np(out, hdr)
                tag = f"{layout} band {rank}/{nranks}x{group}"
                assert (np.delete(frame, own, axis=0) == 77).all(), f"{tag}: rows outside the band were written"
                assert np.isnan(np.delete(hdr, rows, axis=0)).all(), f"{tag}: hdr outside the band was written"
                assert np.array_equal(hdr[rows], full_hdr[rows]), tag
                union[h - 1 - rows] = frame[own]
            assert np.array_equal(union, full), f"{layout} {nranks}x{group}: union of the bands"


@pytest.mark.parametrize("w,h", [(1, 1), (7, 5)])
def test_tiny_sizes(env, w, h):
    r, prm, fx, sky = _setup(env, "split_packed")
    _check(r, prm, _mix9(), fx, sky, w, h, 3, f"{w}x{h}")


def test_1080p(env):
    import relativisticraytracer_b200 as rrt
    r, prm, fx, sky = _setup(env, "split_packed")
    _check(r, prm, rrt.lens_cameras(_cams(["C0"])[0], 0.5, 60.0, 2), fx, sky, 1920, 1080, 2, "1080p ss=2")


def test_two_streams_and_path_sequence(env, tmp_path):
    import relativisticraytracer_b200 as rrt
    import torch
    from relativisticraytracer_b200.parallel import PathSequence
    r, prm, fx, sky = _setup(env, "split_packed")
    w, h = 96, 54
    a = rrt.lens_cameras(_cams(["C1"])[0], 0.5, 30.0, 2)
    b = _mix9()
    want = [_check(r, prm, a, fx, sky, w, h, 2, "stream case a"), _check(r, prm, b, fx, sky, w, h, 3, "stream case b")]
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    hdrs = [_hdr(r, w, h) for _ in range(4)]
    torch.cuda.synchronize()
    outs = []
    for k in range(4):   # interleaved: each call is enqueued while the other stream's may still run, on one scratch pool
        cams, ss, st = (a, 2, s1) if k % 2 == 0 else (b, 3, s2)
        with torch.cuda.stream(st):
            outs.append((r.render_dof(prm, cams, fx, sky, 1.0, w, h, ss, hdr_out=hdrs[k], stream=st), hdrs[k]))
    torch.cuda.synchronize()
    for k, (out, hdr) in enumerate(outs):
        _same(_np(out, hdr), want[k % 2], f"stream call {k}")

    n, path, p = 4, 0, str(tmp_path / "path.rgba")
    seq = PathSequence(r, w, h, depth=2, ss=2, aperture=0.5, focus=40.0)
    with rrt.FrameSink(p, w, h) as sink:
        done, _ = seq.render(path, n, prm, fx, sky, fps=24.0, sink=sink)
    assert done == n
    raw = np.fromfile(p, np.uint8).reshape(n, h, w, 4)
    for k in range(1, n + 1):
        t = rrt.path_clock(k, 24.0)
        cam, _ = rrt.path_state(path, t)
        out = r.render_dof(prm, rrt.lens_cameras(cam, 0.5, 40.0, 2), fx, sky, t, w, h, 2)
        assert np.array_equal(raw[k - 1], _np(out)[0]), k
    with pytest.raises(ValueError):
        PathSequence(r, w, h, ss=2, aperture=0.5, focus=40.0, samples=4, shutter=0.5)


@pytest.mark.parametrize("tracer", ["split_packed", "packed_fused", "fused_media"])
def test_counters_and_launches(env, tracer):
    """rk4_steps and the class counts are those of the ss*ss renders at the pixels each one contributes; launches are the
    large trace's + 1 (the split pipeline's from its bookkeeping: 3 per pass + 1)."""
    import relativisticraytracer_b200 as rrt
    r, prm, fx, sky = _setup(env, tracer)
    w, h, ss = 61, 37, 2
    cams = _cams(["C0", "C1", "C2", "C3"])
    _, pl = _expected_hi(r, prm, cams, fx, sky, w, h, ss, planes=("steps", "cls"))
    steps, cls = 0, []
    for k in range(ss * ss):   # the pixels camera k contributes: sub-sample (i, j) of every output pixel
        i, j = k % ss, k // ss
        s, c = _np(pl["steps"][k][j::ss, i::ss], pl["cls"][k][j::ss, i::ss])
        steps += int(s.astype(np.int64).sum())
        cls.append(c.ravel())
    cls = np.concatenate(cls)
    r.read_counters(reset=True)
    l0 = r.kernel_launches()
    _dof(r, prm, cams, fx, sky, w, h, ss)
    launches = r.kernel_launches() - l0
    got = r.read_counters(reset=True)
    traced = 3 * r.split_stats()["passes_enqueued"] + 1 if tracer == "split_packed" else 1
    assert launches == traced + 1
    assert got["rk4_steps"] == steps > 0
    captured = (cls & rrt.CLS_MASK) == rrt.CLS_CAPTURED
    exhausted = (cls & rrt.CLSF_EXHAUSTED) != 0
    assert got["n_captured"] == captured.sum()
    assert got["n_exhausted"] == exhausted.sum()
    assert got["n_escaped"] == (~captured & ~exhausted).sum()
    assert got["n_touched"] == ((cls & rrt.CLSF_TOUCHED) != 0).sum()


def test_errors(env):
    """RRT_ERR_BAD_ARG with nothing launched: a NULL table, a non-finite camera field, and what rrt_render_ss refuses."""
    import relativisticraytracer_b200 as rrt
    import torch
    r, prm, fx, sky = _setup(env, "split_packed")
    w, h = 32, 16
    frame = torch.empty((h, w, 4), dtype=torch.uint8, device=r.device)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    good = rrt.lens_cameras(_cams(["C1"])[0], 0.5, 30.0, 8)

    def call(ss=2, w_=w, h_=h, band=None, d_out=C.c_void_p(frame.data_ptr()), cams=good, layout=rrt.OUT_FRAME, p=prm):
        arr = (rrt.Camera * 64)(*cams) if cams is not None else None
        return r._lib.rrt_render_dof(r._ctx, C.byref(p), arr, C.byref(fx), C.c_uint64(sky.texture), 1.0, w_, h_, ss,
                                     C.byref(band) if band is not None else None, d_out, layout, None, st)

    def bad_cam(field, comp, value):
        cams = [rrt.Camera.from_buffer_copy(bytes(c)) for c in good]
        getattr(cams[3], field)[comp] = value
        return cams

    big = rrt.Band(0, 1, 1)
    l0 = r.kernel_launches()
    for bad in (dict(cams=None), dict(cams=bad_cam("pos", 0, float("nan"))), dict(cams=bad_cam("forward", 2, float("inf"))),
                dict(cams=bad_cam("right", 1, float("-inf"))), dict(cams=bad_cam("up", 0, float("nan"))),
                dict(ss=0), dict(ss=9), dict(ss=-1), dict(d_out=None), dict(w_=0), dict(h_=-3), dict(ss=8, w_=1 << 28),
                dict(band=rrt.Band(3, 3, 8)), dict(ss=8, w_=1 << 16, h_=1 << 12, band=big), dict(layout=7),
                dict(p=rrt.default_params(max_steps=-1))):
        assert call(**bad) == rrt._capi.ERR_BAD_ARG, bad
    assert r.kernel_launches() == l0
    # only the ss*ss cameras the call uses are read: a non-finite camera 3 does not matter at ss = 1
    assert call(ss=1, cams=bad_cam("pos", 0, float("nan"))) == 0
    with pytest.raises(ValueError):
        r.render_dof(prm, good[:3], fx, sky, 1.0, w, h, 2)
    # the host table may be reused as soon as the call returns
    arr = (rrt.Camera * 4)(*_cams(["C0", "C1", "C2", "C3"]))
    hdr = _hdr(r, w, h)
    r._check(r._lib.rrt_render_dof(r._ctx, C.byref(prm), arr, C.byref(fx), C.c_uint64(sky.texture), 1.0, w, h, 2, None,
                                   C.c_void_p(frame.data_ptr()), rrt.OUT_FRAME, C.c_void_p(hdr.data_ptr()), st))
    C.memset(arr, 0xff, C.sizeof(arr))   # NaN everywhere
    got = _np(frame, hdr)
    want = _resolve(r, prm, fx, _expected_hi(r, prm, _cams(["C0", "C1", "C2", "C3"]), fx, sky, w, h, 2), 2, w, h)
    _same(got, want, "table overwritten after the call")
