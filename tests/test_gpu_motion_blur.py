"""rrt_render_mb / rrt_capture_render_mb / rrt_resolve_time / Renderer.render_mb / Capture.render_mb: motion-blurred frames.

Sub-frame i of a blurred frame is rrt_render with camera cams[i] at time times[i] into an hdr plane, and the pixel's hdr
value is the mean of the n planes in a fixed order (plane 0 to n-1, round-to-nearest float32, divided by n), followed by
the render's own post step.  So everything here is exact equality: against rrt_render itself (n = 1), against n renders
followed by rrt_resolve_time, against a numpy float32 reduction in the same order, and between captures, bands, streams
and sequences."""
import ctypes as C

import numpy as np
import pytest

from parity import CAMERAS

pytestmark = pytest.mark.gpu

# (sky, exposure, effect fields changed from the defaults), as in test_gpu_supersample.py
VARIANTS = [
    ("small", 0.8, {}),
    ("smooth", 1.7, dict(use_bloom=0, use_vignette=1, vignette_intensity=0.7, use_ca=1, ca_amount=0.01)),
    ("small", 0.5, dict(bloom_threshold=0.3)),
]
TIMES = (1.0, 0.0, 123.5, 7.25, 3.5, -2.0, 50.0, 0.5)   # not monotonic; n sub-frames take the first n


@pytest.fixture(scope="module")
def env(built, sky_small, sky_smooth):
    """A context of its own (counters, launch count and pipeline are per context) and the two skies."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    import relativisticraytracer_b200 as rrt
    r = rrt.Renderer(0)
    skies = {"small": r.create_sky(sky_small), "smooth": r.create_sky(sky_smooth)}
    yield r, skies
    for s in skies.values():
        s.close()
    r.close()


def _args(skies, cam, spin, flags, variant=VARIANTS[0], **fx_over):
    import relativisticraytracer_b200 as rrt
    sky, exposure, over = variant
    return (rrt.default_params(spin_a=spin, flags=flags, exposure=exposure), rrt.camera_state_from(*CAMERAS[cam]),
            rrt.default_effects(**{**fx_over, **over}), skies[sky])


def _path_cams(n, path=0, t0=2.0):
    """n distinct cameras of a built-in path."""
    import relativisticraytracer_b200 as rrt
    return [rrt.path_state(path, t0 + 0.37 * i)[0] for i in range(n)]


def _hdr(r, w, h, fill=0.0):
    import torch
    return torch.full((h, w, 4), fill, dtype=torch.float32, device=r.device)


def _np(*ts):
    import torch
    torch.cuda.synchronize()
    return tuple(t.cpu().numpy() for t in ts)


def _render(r, prm, cam, fx, sky, t, w, h, **kw):
    """(frame, hdr plane) of rrt_render."""
    hdr = _hdr(r, w, h)
    out = r.render(prm, cam, fx, sky, t, w, h, planes={"hdr": hdr}, **kw)
    return _np(out, hdr)


def _render_mb(r, prm, cams, fx, sky, times, w, h, **kw):
    """(frame, mean hdr) of rrt_render_mb."""
    hdr = _hdr(r, w, h)
    out = r.render_mb(prm, cams, fx, sky, times, w, h, hdr_out=hdr, **kw)
    return _np(out, hdr)


def _stack(r, prm, cams, fx, sky, times, w, h):
    """The (n, h, w, 4) hdr planes of the n sub-frame renders (a device tensor)."""
    import relativisticraytracer_b200 as rrt
    import torch
    n = len(times)
    cams = [cams] * n if isinstance(cams, rrt.Camera) else cams
    st = torch.zeros((n, h, w, 4), dtype=torch.float32, device=r.device)
    for i in range(n):
        r.render(prm, cams[i], fx, sky, times[i], w, h, planes={"hdr": st[i]})
    return st


def _resolve_time(r, prm, fx, stack, w, h, **kw):
    hdr = _hdr(r, w, h)
    out = r.resolve_time(prm, fx, stack, w, h, hdr_out=hdr, **kw)
    return _np(out, hdr)


def _mean(stack):
    """numpy float32 reduction in the order rrt_resolve_time specifies: plane 0, then 1 .. n-1, / n."""
    s = stack[0].copy()
    for i in range(1, stack.shape[0]):
        s = s + stack[i]
    return s / np.float32(stack.shape[0])


def _same(got, want, tag):
    for name, a, b in zip(("frame", "hdr"), got, want):
        assert np.array_equal(a, b, equal_nan=True), f"{tag}: {name} differs on {np.sum(a != b)} elements"


@pytest.mark.parametrize("cam", ["C0", "C1", "C2", "C3"])
@pytest.mark.parametrize("spin,flags", [(0.99, 7), (0.0, 7), (0.99, 5), (0.99, 4), (0.99, 3), (0.0, 1)])
def test_n1_is_the_render(env, cam, spin, flags):
    """render_mb(n=1) writes rrt_render's bytes and hdr values: split pipeline (flags 7, 5, 3, 1), packed fused kernel
    (4), strict contract (3, 1); lens on (the default effects) and off."""
    r, skies = env
    for lens in (1, 0):
        prm, c, fx, sky = _args(skies, cam, spin, flags, use_lens=lens)
        _same(_render_mb(r, prm, c, fx, sky, [123.5], 203, 117), _render(r, prm, c, fx, sky, 123.5, 203, 117),
              f"{cam} a={spin} flags={flags} lens={lens}")


@pytest.mark.parametrize("lens", [1, 0])
@pytest.mark.parametrize("variant", range(len(VARIANTS)))
def test_n1_shading_variants(env, variant, lens):
    r, skies = env
    prm, c, fx, sky = _args(skies, "C3", 0.99, 7, VARIANTS[variant], use_lens=lens)
    _same(_render_mb(r, prm, c, fx, sky, [7.25], 203, 117), _render(r, prm, c, fx, sky, 7.25, 203, 117),
          f"variant {variant} lens={lens}")


@pytest.mark.parametrize("cams", ["still", "path"])
@pytest.mark.parametrize("flags", [7, 4, 3, 0])
@pytest.mark.parametrize("n", [2, 3, 8])
def test_render_mb_is_renders_then_resolve_time(env, n, flags, cams):
    """Both contracts, with and without media, non-monotonic times, one camera or n distinct path cameras.  The resolved
    hdr is also the numpy mean of the sub-frame planes."""
    r, skies = env
    w, h = 61, 37
    prm, c, fx, sky = _args(skies, "C1", 0.99, flags, VARIANTS[1])
    cam = c if cams == "still" else _path_cams(n)
    times = TIMES[:n]
    stack = _stack(r, prm, cam, fx, sky, times, w, h)
    want = _resolve_time(r, prm, fx, stack, w, h)
    _same(_render_mb(r, prm, cam, fx, sky, times, w, h), want, f"n={n} flags={flags} {cams}")
    assert np.array_equal(want[1].view(np.uint32), _mean(stack.cpu().numpy()).view(np.uint32))
    if flags & 3:   # the disk moves: the sub-frames differ, so the mean is not any one of them
        planes = stack.cpu().numpy()
        assert not np.array_equal(planes[0], planes[1])


@pytest.mark.parametrize("n", [1, 2, 5, 64])
def test_resolve_time_mean_of_a_random_stack(env, n):
    """Bit-equal to the numpy float32 reduction on magnitudes from 1e-6 to 1e4, where the order of the sum matters."""
    import relativisticraytracer_b200 as rrt
    import torch
    r, _ = env
    w, h = 37, 23
    rng = np.random.default_rng(2000 + n)
    st_np = (10.0 ** rng.uniform(-6, 4, size=(n, h, w, 4))).astype(np.float32)
    _, hdr = _resolve_time(r, rrt.default_params(), rrt.default_effects(), torch.from_numpy(st_np).to(r.device), w, h)
    assert np.array_equal(hdr.view(np.uint32), _mean(st_np).view(np.uint32))


@pytest.mark.parametrize("n", [2, 8])
def test_post_step_is_the_renders(env, n):
    """The bytes of resolve_time(n) equal those of resolve_time(1) of its own mean: the mean goes through the same post
    step (which test_n1_is_the_render ties to the render's), for changed exposure, bloom, vignette and lens."""
    import relativisticraytracer_b200 as rrt
    import torch
    r, skies = env
    w, h = 61, 37
    prm, c, fx, sky = _args(skies, "C3", 0.99, 7)
    stack = _stack(r, prm, c, fx, sky, TIMES[:n], w, h)
    overs = [(0.8, {}), (1.7, dict(use_bloom=0, use_vignette=1, vignette_intensity=0.7)), (0.5, dict(bloom_threshold=0.3)),
             (2.5, dict(use_vignette=0, bloom_intensity=1.5)), (0.8, dict(use_lens=0))]
    for exposure, over in overs:
        p2, f2 = rrt.default_params(exposure=exposure), rrt.default_effects(**over)
        frame, mean = _resolve_time(r, p2, f2, stack, w, h)
        again, _ = _resolve_time(r, p2, f2, torch.from_numpy(mean).to(r.device)[None], w, h)
        assert np.array_equal(frame, again), f"n={n} exposure={exposure} {over}"


def _capture(r, skies, cam, spin, flags, w, h, **kw):
    """A capture with exposure 0.8, the default effects and the small sky, as in test_gpu_retime.py."""
    import relativisticraytracer_b200 as rrt
    return r.capture(rrt.default_params(spin_a=spin, flags=flags, exposure=0.8), rrt.camera_state_from(*CAMERAS[cam]),
                     rrt.default_effects(), skies["small"], w, h, **kw)


def _capture_mb(r, cap, prm, fx, sky, times, **kw):
    hdr = _hdr(r, cap.w, cap.h)
    out = cap.render_mb(prm, fx, sky, times, hdr_out=hdr, **kw)
    return _np(out, hdr)


def _left_over_captures(r, skies, cam, spin, flags, w, h):
    """(capture holding part of the frame, capture holding none of it)."""
    none = _capture(r, skies, cam, spin, flags, w, h, max_bytes=1 << 20)
    info = none.info()
    assert info["tiles_left"] == info["tiles"] > 0 and info["groups_queued"] == 0, info
    for mib in (128, 384, 1024):
        part = _capture(r, skies, cam, spin, flags, w, h, max_bytes=mib << 20)
        info = part.info()
        if 0 < info["tiles_left"] < info["tiles"]:
            return part, none
        part.close()
    pytest.fail(f"no pool size left part of the frame: {info}")


@pytest.mark.parametrize("spin,flags", [(0.99, 7), (0.0, 3)])
def test_capture_render_mb_is_render_mb(env, spin, flags):
    """A capture that holds the whole frame, one that holds part of it and one that holds none: render_mb with the
    capture's camera for every sub-frame; at n = 1 the capture's own render."""
    r, skies = env
    w, h, cam = 203, 117, "C1"
    whole = _capture(r, skies, cam, spin, flags, w, h)
    assert whole.info()["tiles_left"] == 0
    part, none = _left_over_captures(r, skies, cam, spin, flags, w, h)
    prm, c, fx, sky = _args(skies, cam, spin, flags, VARIANTS[1])
    for cap in (whole, part, none):
        tag = str(cap.info())
        for n in (1, 4):
            times = TIMES[:n]
            got = _capture_mb(r, cap, prm, fx, sky, times)
            _same(got, _render_mb(r, prm, c, fx, sky, times, w, h), f"{tag} n={n}")
            if n == 1:
                hdr = _hdr(r, w, h)
                _same(got, _np(cap.render(prm, fx, sky, times[0], hdr_out=hdr), hdr), f"{tag}: Capture.render")
        cap.close()


@pytest.mark.parametrize("layout", ["frame", "packed"])
def test_bands(env, layout):
    """render_mb and Capture.render_mb write exactly the band's rows (the others keep a sentinel) and its hdr pixels only,
    equal to those of the full frame."""
    import relativisticraytracer_b200 as rrt
    import torch
    from relativisticraytracer_b200.parallel import band_rows_of
    r, skies = env
    w, h, n = 67, 41, 3
    lay = rrt.OUT_FRAME if layout == "frame" else rrt.OUT_PACKED
    prm, c, fx, sky = _args(skies, "C1", 0.99, 7)
    times = TIMES[:n]
    full, full_hdr = _render_mb(r, prm, c, fx, sky, times, w, h)
    for band in (rrt.Band(0, 3, 8), rrt.Band(2, 3, 8), rrt.Band(1, 2, 1)):
        rows = band_rows_of(band.rank, band.nranks, band.group, h)
        own = (h - 1 - rows) if lay == rrt.OUT_FRAME else np.arange(len(rows))   # buffer rows the band writes
        cap = _capture(r, skies, "C1", 0.99, 7, w, h, band=band)
        for how in ("render_mb", "capture"):
            out = torch.full((h, w, 4), 77, dtype=torch.uint8, device=r.device)      # h rows for either layout
            hdr = _hdr(r, w, h, float("nan"))
            if how == "render_mb":
                r.render_mb(prm, c, fx, sky, times, w, h, band=band, out=out, layout=lay, hdr_out=hdr)
            else:
                cap.render_mb(prm, fx, sky, times, out=out, layout=lay, hdr_out=hdr)
            frame, hdr = _np(out, hdr)
            tag = f"{how} {layout} band {band.rank}/{band.nranks}x{band.group}"
            assert (np.delete(frame, own, axis=0) == 77).all(), f"{tag}: rows outside the band were written"
            assert np.isnan(np.delete(hdr, rows, axis=0)).all(), f"{tag}: hdr outside the band was written"
            assert np.array_equal(hdr[rows], full_hdr[rows]), tag
            assert np.array_equal(frame[own], full[h - 1 - rows]), tag
        cap.close()


@pytest.mark.parametrize("w,h,cam,n", [(1, 1, "C3", 3), (7, 5, "C1", 5), (1920, 1080, "C0", 4)])
def test_sizes(env, w, h, cam, n):
    r, skies = env
    prm, c, fx, sky = _args(skies, cam, 0.99, 7, VARIANTS[1])
    times = TIMES[:n]
    stack = _stack(r, prm, c, fx, sky, times, w, h)
    want = _resolve_time(r, prm, fx, stack, w, h)
    _same(_render_mb(r, prm, c, fx, sky, times, w, h), want, f"{w}x{h}")
    assert np.array_equal(want[1].view(np.uint32), _mean(stack.cpu().numpy()).view(np.uint32))


def test_supersampled_composition(env):
    """resolve_time at 2w x 2h into an hdr plane, then resolve(2): the hdr is the two-stage numpy reduction (time, then
    each pixel's 2 x 2 block), the frame is resolve(2) of that plane."""
    r, skies = env
    w, h, ss, n = 61, 37, 2, 3
    prm, c, fx, sky = _args(skies, "C3", 0.99, 7)
    stack = _stack(r, prm, c, fx, sky, TIMES[:n], ss * w, ss * h)
    hi = _hdr(r, ss * w, ss * h)
    r.resolve_time(prm, fx, stack, ss * w, ss * h, hdr_out=hi)
    hdr = _hdr(r, w, h)
    frame, hdr = _np(r.resolve(prm, fx, hi, ss, w, h, hdr_out=hdr), hdr)
    t_mean = _mean(stack.cpu().numpy())
    H = t_mean.reshape(h, ss, w, ss, 4)
    s = H[:, 0, :, 0].copy()
    for j in range(ss):
        for i in range(ss):
            if i or j:
                s = s + H[:, j, :, i]
    assert np.array_equal(hdr.view(np.uint32), (s / np.float32(ss * ss)).view(np.uint32))
    assert np.array_equal(_np(hi)[0].view(np.uint32), t_mean.view(np.uint32))
    assert (frame != 0).any()


def test_path_sequence(env, tmp_path):
    """PathSequence(shutter=0.5, samples=4): frame k is render_mb at shutter_times(path_clock(k)) with the path's camera at
    each sub-frame's time."""
    import relativisticraytracer_b200 as rrt
    from relativisticraytracer_b200.parallel import PathSequence
    r, skies = env
    w, h, fps, samples = 96, 54, 24.0, 4
    prm, _, fx, sky = _args(skies, "C1", 0.99, 7)
    n, path, p = 4, 0, str(tmp_path / "path.rgba")
    seq = PathSequence(r, w, h, depth=2, shutter=0.5, samples=samples)
    with rrt.FrameSink(p, w, h) as sink:
        done, _ = seq.render(path, n, prm, fx, sky, fps=fps, sink=sink)
    assert done == n
    raw = np.fromfile(p, np.uint8).reshape(n, h, w, 4)
    for k in range(1, n + 1):
        times = rrt.shutter_times(rrt.path_clock(k, fps), 0.5, fps, samples)
        cams = [rrt.path_state(path, t)[0] for t in times]
        out = r.render_mb(prm, cams, fx, sky, times, w, h)
        assert np.array_equal(raw[k - 1], _np(out)[0]), k
    with pytest.raises(ValueError):
        PathSequence(r, w, h, ss=2, samples=2)
    for bad in (dict(samples=0), dict(samples=65), dict(samples=2, shutter=1.5)):
        with pytest.raises(ValueError):
            PathSequence(r, w, h, **bad)


@pytest.mark.parametrize("flags", [7, 4])
def test_counters_and_launches(env, flags):
    """render_mb counts what its n renders count and launches their kernels + 1."""
    r, skies = env
    w, h, n = 61, 37, 3
    prm, c, fx, sky = _args(skies, "C1", 0.99, flags)
    cams = _path_cams(n)
    times = TIMES[:n]
    r.read_counters(reset=True)
    l0 = r.kernel_launches()
    _stack(r, prm, cams, fx, sky, times, w, h)
    want_launches = r.kernel_launches() - l0
    want = r.read_counters(reset=True)
    l0 = r.kernel_launches()
    _render_mb(r, prm, cams, fx, sky, times, w, h)
    assert r.kernel_launches() - l0 == want_launches + 1
    assert r.read_counters(reset=True) == want and want["rk4_steps"] > 0


@pytest.mark.parametrize("left_over", [False, True])
def test_capture_counters_and_launches(env, left_over):
    """Capture.render_mb counts what its n capture renders count; launches n * (3 or 4) + 1."""
    r, skies = env
    w, h, cam, n = 203, 117, "C1", 4
    if left_over:
        cap, none = _left_over_captures(r, skies, cam, 0.99, 7, w, h)
        none.close()
    else:
        cap = _capture(r, skies, cam, 0.99, 7, w, h)
    prm, _, fx, sky = _args(skies, cam, 0.99, 7)
    times = TIMES[:n]
    r.read_counters(reset=True)
    for t in times:
        cap.render(prm, fx, sky, t, hdr_out=_hdr(r, w, h))
    want = r.read_counters(reset=True)
    l0 = r.kernel_launches()
    _capture_mb(r, cap, prm, fx, sky, times)
    assert r.kernel_launches() - l0 == n * (4 if left_over else 3) + 1
    assert r.read_counters(reset=True) == want and want["dense_samples"] > 0
    cap.close()


def test_two_streams_and_pool_reuse(env):
    """render_mb and Capture.render_mb interleaved on two streams without host synchronisation, each call taking its stack
    from the pool the previous calls returned blocks to."""
    import torch
    r, skies = env
    w, h = 96, 54
    a = _args(skies, "C1", 0.99, 7)
    b = _args(skies, "C3", 0.0, 3, VARIANTS[1])
    cap = _capture(r, skies, "C3", 0.0, 3, w, h)
    ta, tb = TIMES[:4], TIMES[2:5]
    want = [_render_mb(r, a[0], _path_cams(4), a[2], a[3], ta, w, h), _render_mb(r, b[0], b[1], b[2], b[3], tb, w, h)]
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    hdrs = [_hdr(r, w, h) for _ in range(6)]
    torch.cuda.synchronize()
    outs = []
    for k in range(6):
        st = s1 if k % 2 == 0 else s2
        with torch.cuda.stream(st):
            if k % 2 == 0:
                outs.append((r.render_mb(a[0], _path_cams(4), a[2], a[3], ta, w, h, hdr_out=hdrs[k], stream=st), hdrs[k]))
            else:
                outs.append((cap.render_mb(b[0], b[2], b[3], tb, hdr_out=hdrs[k], stream=st), hdrs[k]))
    torch.cuda.synchronize()
    for k, (out, hdr) in enumerate(outs):
        _same(_np(out, hdr), want[k % 2], f"stream call {k}")
    cap.close()


def test_errors(env):
    """RRT_ERR_BAD_ARG with nothing launched."""
    import relativisticraytracer_b200 as rrt
    import torch
    r, skies = env
    w, h = 32, 16
    bad_arg = rrt._capi.ERR_BAD_ARG
    prm, cam, fx, sky = _args(skies, "C1", 0.99, 7)
    frame = torch.empty((h, w, 4), dtype=torch.uint8, device=r.device)
    hdr = _hdr(r, w, h)
    stack = torch.zeros((4, h, w, 4), dtype=torch.float32, device=r.device)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    cams = (rrt.Camera * 65)(*([cam] * 65))
    times = (C.c_float * 65)(*([1.0] * 65))
    cap = _capture(r, skies, "C1", 0.99, 7, w, h)

    def render_mb(n=2, cams_=cams, times_=times, d_out=C.c_void_p(frame.data_ptr()), hdr_out=None, band=None):
        return r._lib.rrt_render_mb(r._ctx, C.byref(prm), cams_, C.byref(fx), C.c_uint64(sky.texture), times_, n, w, h,
                                    C.byref(band) if band is not None else None, d_out, rrt.OUT_FRAME, hdr_out, st)

    def resolve_time(n=4, stack_=C.c_void_p(stack.data_ptr()), d_out=C.c_void_p(frame.data_ptr()), hdr_out=None, band=None):
        return r._lib.rrt_resolve_time(r._ctx, C.byref(prm), C.byref(fx), n, w, h, C.byref(band) if band is not None else None,
                                       stack_, d_out, rrt.OUT_FRAME, hdr_out, st)

    def capture_mb(n=2, prm_=prm, fx_=fx, times_=times, d_out=C.c_void_p(frame.data_ptr()), hdr_out=None, handle=cap._h):
        return r._lib.rrt_capture_render_mb(handle, C.byref(prm_), C.byref(fx_), C.c_uint64(sky.texture), times_, n, d_out,
                                            rrt.OUT_FRAME, hdr_out, st)

    l0 = r.kernel_launches()
    for fn in (render_mb, resolve_time, capture_mb):
        for bad in (dict(n=0), dict(n=65), dict(n=-1), dict(d_out=None)):
            assert fn(**bad) == bad_arg, (fn.__name__, bad)
    for bad in (dict(cams_=None), dict(times_=None), dict(band=rrt.Band(3, 3, 8))):
        assert render_mb(**bad) == bad_arg, bad
    assert resolve_time(stack_=None) == bad_arg
    assert resolve_time(band=rrt.Band(0, 2, 0)) == bad_arg
    for bad in (dict(times_=None), dict(handle=None), dict(prm_=rrt.default_params(spin_a=0.99, flags=3)),
                dict(fx_=rrt.default_effects(use_lens=0)), dict(fx_=rrt.default_effects(distortion_amount=0.2))):
        assert capture_mb(**bad) == bad_arg, bad
    base = stack.data_ptr()
    for off in (0, 16 * (4 * w * h - 1), -16 * (w * h - 1)):   # hdr_out sharing a float4 with the stack, at either end
        assert resolve_time(hdr_out=C.c_void_p(base + off)) == bad_arg, off
    assert r.kernel_launches() == l0
    # a separate plane is fine, and so are hdr-only calls and planes that touch the stack without sharing a byte
    assert resolve_time(hdr_out=C.c_void_p(hdr.data_ptr())) == 0
    assert render_mb(d_out=None, hdr_out=C.c_void_p(hdr.data_ptr())) == 0
    assert capture_mb(d_out=None, hdr_out=C.c_void_p(hdr.data_ptr())) == 0
    assert render_mb(n=64) == 0 and capture_mb(n=64) == 0
    buf = _hdr(r, w, 6 * h, float("nan"))   # [hdr_out | 4 planes | hdr_out] in one allocation
    lo, mid, up = buf[:h], buf[h:5 * h], buf[5 * h:]
    mid.copy_(stack.view(4 * h, w, 4))
    for out_plane in (lo, up):
        assert resolve_time(stack_=C.c_void_p(mid.data_ptr()), hdr_out=C.c_void_p(out_plane.data_ptr())) == 0
    torch.cuda.synchronize()
    cap.close()
