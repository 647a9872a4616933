"""rrt_render_ss / rrt_resolve / Renderer.render_ss / Renderer.resolve: anti-aliased frames with ss x ss rays per pixel.

Sub-sample (i, j) of output pixel (x, y) is pixel (ss*x + i, ss*y + j) of the ss*w x ss*h render, and the pixel's hdr value
is the mean of its sub-samples in a fixed order (row-major, round-to-nearest float32), followed by the render's own post
step.  So everything here is exact equality: against rrt_render itself (ss = 1, and the large render + rrt_resolve),
against a numpy float32 reduction in the same order, and between bands, streams and sequences."""
import ctypes as C

import numpy as np
import pytest

from parity import CAMERAS

pytestmark = pytest.mark.gpu

# (sky, exposure, effect fields changed from the defaults), as in test_gpu_shade.py
VARIANTS = [
    ("small", 0.8, {}),
    ("smooth", 1.7, dict(use_bloom=0, use_vignette=1, vignette_intensity=0.7, use_ca=1, ca_amount=0.01)),
    ("small", 0.5, dict(bloom_threshold=0.3)),
]


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


def _hdr(r, w, h, fill=0.0):
    import torch
    return torch.full((h, w, 4), fill, dtype=torch.float32, device=r.device)


def _np(*ts):
    import torch
    torch.cuda.synchronize()
    return tuple(t.cpu().numpy() for t in ts)


def _render(r, args, w, h, **kw):
    """(frame, hdr plane) of rrt_render."""
    hdr = _hdr(r, w, h)
    out = r.render(*args, 1.0, w, h, planes={"hdr": hdr}, **kw)
    return _np(out, hdr)


def _render_ss(r, args, w, h, ss, **kw):
    """(frame, averaged hdr) of rrt_render_ss."""
    hdr = _hdr(r, w, h)
    out = r.render_ss(*args, 1.0, w, h, ss, hdr_out=hdr, **kw)
    return _np(out, hdr)


def _trace_hi(r, args, w, h, ss):
    """The hdr plane of the ss*w x ss*h render (a device tensor)."""
    hi = _hdr(r, ss * w, ss * h)
    r.render(*args, 1.0, ss * w, ss * h, planes={"hdr": hi})
    return hi


def _resolve(r, args, hi, ss, w, h, **kw):
    prm, _, fx, _ = args
    hdr = _hdr(r, w, h)
    out = r.resolve(prm, fx, hi, ss, w, h, hdr_out=hdr, **kw)
    return _np(out, hdr)


def _mean(hi, ss):
    """numpy float32 reduction in the order rrt_resolve specifies: (0,0), then row-major (j outer, i inner), / ss*ss."""
    hh, ww = hi.shape[0] // ss, hi.shape[1] // ss
    H = hi.reshape(hh, ss, ww, ss, 4)
    s = H[:, 0, :, 0].copy()
    for j in range(ss):
        for i in range(ss):
            if i or j:
                s = s + H[:, j, :, i]
    return s / np.float32(ss * ss)


def _same(got, want, tag):
    for name, a, b in zip(("frame", "hdr"), got, want):
        assert np.array_equal(a, b, equal_nan=True), f"{tag}: {name} differs on {np.sum(a != b)} elements"


@pytest.mark.parametrize("cam", ["C0", "C1", "C2", "C3"])
@pytest.mark.parametrize("spin,flags", [(0.99, 7), (0.0, 7), (0.99, 5), (0.99, 4), (0.99, 3), (0.0, 1)])
def test_ss1_is_the_render(env, cam, spin, flags):
    """render_ss(ss=1) writes rrt_render's bytes and hdr values: split pipeline (flags 7, 5, 3, 1), packed fused kernel
    (4), strict contract (3, 1); lens on (the default effects) and off."""
    r, skies = env
    for lens in (1, 0):
        args = _args(skies, cam, spin, flags, use_lens=lens)
        _same(_render_ss(r, args, 203, 117, 1), _render(r, args, 203, 117), f"{cam} a={spin} flags={flags} lens={lens}")


@pytest.mark.parametrize("flags", [7, 4, 3, 0])
@pytest.mark.parametrize("ss", [2, 3, 4])
def test_render_ss_is_large_render_then_resolve(env, ss, flags):
    """Both contracts, with and without media.  The resolved hdr is also the numpy mean of the traced plane."""
    r, skies = env
    w, h = 61, 37
    args = _args(skies, "C1", 0.99, flags)
    hi = _trace_hi(r, args, w, h, ss)
    want = _resolve(r, args, hi, ss, w, h)
    _same(_render_ss(r, args, w, h, ss), want, f"ss={ss} flags={flags}")
    assert np.array_equal(want[1].view(np.uint32), _mean(hi.cpu().numpy(), ss).view(np.uint32))


@pytest.mark.parametrize("ss", [1, 2, 3, 5, 8])
def test_resolve_mean_of_a_random_plane(env, ss):
    """Bit-equal to the numpy float32 reduction on magnitudes from 1e-6 to 1e4, where the order of the sum matters."""
    import relativisticraytracer_b200 as rrt
    import torch
    r, _ = env
    w, h = 37, 23
    rng = np.random.default_rng(1000 + ss)
    hi_np = (10.0 ** rng.uniform(-6, 4, size=(ss * h, ss * w, 4))).astype(np.float32)
    hi = torch.from_numpy(hi_np).to(r.device)
    _, hdr = _resolve(r, (rrt.default_params(), None, rrt.default_effects(), None), hi, ss, w, h)
    assert np.array_equal(hdr.view(np.uint32), _mean(hi_np, ss).view(np.uint32))


@pytest.mark.parametrize("ss", [2, 4])
def test_post_step_is_the_renders(env, ss):
    """The bytes of resolve(ss, H) equal those of resolve(1, mean): the averaged value goes through the same post step
    (which test_ss1_is_the_render ties to the render's), for changed exposure, bloom and vignette."""
    import relativisticraytracer_b200 as rrt
    import torch
    r, skies = env
    w, h = 61, 37
    hi = _trace_hi(r, _args(skies, "C3", 0.99, 7), w, h, ss)
    overs = [(0.8, {}), (1.7, dict(use_bloom=0, use_vignette=1, vignette_intensity=0.7)), (0.5, dict(bloom_threshold=0.3)),
             (2.5, dict(use_vignette=0, bloom_intensity=1.5)), (0.8, dict(use_lens=0))]
    for exposure, over in overs:
        args = (rrt.default_params(exposure=exposure), None, rrt.default_effects(**over), None)
        frame, mean = _resolve(r, args, hi, ss, w, h)
        again, _ = _resolve(r, args, torch.from_numpy(mean).to(r.device), 1, w, h)
        assert np.array_equal(frame, again), f"ss={ss} exposure={exposure} {over}"


@pytest.mark.parametrize("layout", ["frame", "packed"])
def test_bands(env, layout):
    """Each band writes exactly its rows (the others keep a sentinel) and its hdr pixels only; the union of the bands is
    the full frame."""
    import relativisticraytracer_b200 as rrt
    import torch
    from relativisticraytracer_b200.parallel import band_rows_of
    r, skies = env
    w, h, ss = 67, 41, 2
    lay = rrt.OUT_FRAME if layout == "frame" else rrt.OUT_PACKED
    args = _args(skies, "C1", 0.99, 7)
    full, full_hdr = _render_ss(r, args, w, h, ss)
    for nranks in (2, 3):
        for group in (1, 8):
            union = np.full((h, w, 4), 77, np.uint8)
            for rank in range(nranks):
                band = rrt.Band(rank, nranks, group)
                rows = band_rows_of(rank, nranks, group, h)
                own = (h - 1 - rows) if lay == rrt.OUT_FRAME else np.arange(len(rows))   # buffer rows the band writes
                out = torch.full((h, w, 4), 77, dtype=torch.uint8, device=r.device)      # h rows for either layout
                hdr = _hdr(r, w, h, float("nan"))
                r.render_ss(*args, 1.0, w, h, ss, band=band, out=out, layout=lay, hdr_out=hdr)
                frame, hdr = _np(out, hdr)
                tag = f"{layout} band {rank}/{nranks}x{group}"
                assert (np.delete(frame, own, axis=0) == 77).all(), f"{tag}: rows outside the band were written"
                assert np.isnan(np.delete(hdr, rows, axis=0)).all(), f"{tag}: hdr outside the band was written"
                assert np.array_equal(hdr[rows], full_hdr[rows]), tag
                union[h - 1 - rows] = frame[own]
            assert np.array_equal(union, full), f"{layout} {nranks}x{group}: union of the bands"


@pytest.mark.parametrize("w,h", [(1, 1), (7, 5)])
def test_tiny_sizes(env, w, h):
    r, skies = env
    args = _args(skies, "C3", 0.99, 7)
    hi = _trace_hi(r, args, w, h, 3)
    want = _resolve(r, args, hi, 3, w, h)
    _same(_render_ss(r, args, w, h, 3), want, f"{w}x{h}")
    assert np.array_equal(want[1].view(np.uint32), _mean(hi.cpu().numpy(), 3).view(np.uint32))


def test_1080p_ss2_is_the_4k_render(env):
    """The 2x2-supersampled 1080p frame traces the 3840x2160 frame's rays: its resolve of that render's hdr plane."""
    r, skies = env
    args = _args(skies, "C0", 0.99, 7)
    want = _resolve(r, args, _trace_hi(r, args, 1920, 1080, 2), 2, 1920, 1080)
    _same(_render_ss(r, args, 1920, 1080, 2), want, "1080p ss=2")


@pytest.mark.parametrize("ss", [2, 3])
def test_reshade_a_supersampled_frame(env, ss):
    """shade at ss*w x ss*h into a large hdr plane, then resolve, is render_ss with the new sky, exposure and effects."""
    import relativisticraytracer_b200 as rrt
    r, skies = env
    w, h, cam = 61, 37, "C3"
    traced = r.alloc_planes(ss * w, ss * h, rrt.TRACE_PLANES)
    r.render(*_args(skies, cam, 0.99, 7), 1.0, ss * w, ss * h, planes=traced)
    for k, v in enumerate(VARIANTS):
        args = _args(skies, cam, 0.99, 7, v)
        prm, _, fx, sky = args
        hi = _hdr(r, ss * w, ss * h)
        r.shade(prm, fx, sky, traced, ss * w, ss * h, hdr_out=hi)
        _same(_resolve(r, args, hi, ss, w, h), _render_ss(r, args, w, h, ss), f"ss={ss} variant {k}")


@pytest.mark.parametrize("flags", [7, 4])
def test_counters_and_launches(env, flags):
    """render_ss(k) counts the sub-rays of render(k*w, k*h) and launches that render's kernels + 1 (the split pipeline's
    launches come from its bookkeeping: 3 per pass + 1)."""
    r, skies = env
    w, h, ss = 61, 37, 3
    args = _args(skies, "C1", 0.99, flags)
    for how in ("render", "render_ss"):
        r.read_counters(reset=True)
        l0 = r.kernel_launches()
        if how == "render":
            _trace_hi(r, args, w, h, ss)
        else:
            _render_ss(r, args, w, h, ss)
        launches = r.kernel_launches() - l0
        counters = r.read_counters(reset=True)
        traced = 3 * r.split_stats()["passes_enqueued"] + 1 if flags == 7 else 1
        assert launches == traced + (how == "render_ss"), how
        if how == "render":
            want = counters
    assert counters == want and counters["rk4_steps"] > 0


def test_two_streams_and_path_sequence(env, tmp_path):
    import relativisticraytracer_b200 as rrt
    import torch
    from relativisticraytracer_b200.parallel import PathSequence
    r, skies = env
    w, h = 96, 54
    a = _args(skies, "C1", 0.99, 7)
    b = _args(skies, "C3", 0.0, 4, VARIANTS[1])
    want = [_render_ss(r, a, w, h, 2), _render_ss(r, b, w, h, 3)]
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    hdrs = [_hdr(r, w, h) for _ in range(4)]
    torch.cuda.synchronize()
    outs = []
    for k in range(4):   # interleaved: each call is enqueued while the other stream's may still run
        args, ss, st = (a, 2, s1) if k % 2 == 0 else (b, 3, s2)
        with torch.cuda.stream(st):
            outs.append((r.render_ss(*args, 1.0, w, h, ss, hdr_out=hdrs[k], stream=st), hdrs[k]))
    torch.cuda.synchronize()
    for k, (out, hdr) in enumerate(outs):
        _same(_np(out, hdr), want[k % 2], f"stream call {k}")

    prm, _, fx, sky = a
    n, path, p = 5, 0, str(tmp_path / "path.rgba")
    seq = PathSequence(r, w, h, depth=2, ss=2)
    with rrt.FrameSink(p, w, h) as sink:
        done, _ = seq.render(path, n, prm, fx, sky, fps=24.0, sink=sink)
    assert done == n
    raw = np.fromfile(p, np.uint8).reshape(n, h, w, 4)
    for k in range(1, n + 1):
        t = rrt.path_clock(k, 24.0)
        cam, _ = rrt.path_state(path, t)
        out = r.render_ss(prm, cam, fx, sky, t, w, h, 2)
        assert np.array_equal(raw[k - 1], _np(out)[0]), k


def test_errors(env):
    """RRT_ERR_BAD_ARG with nothing launched."""
    import relativisticraytracer_b200 as rrt
    import torch
    r, skies = env
    w, h = 32, 16
    prm, cam, fx, sky = _args(skies, "C1", 0.99, 7)
    frame = torch.empty((h, w, 4), dtype=torch.uint8, device=r.device)
    hdr = _hdr(r, w, h)
    hi = _hdr(r, 2 * w, 2 * h)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def render_ss(ss=2, w_=w, h_=h, band=None, d_out=C.c_void_p(frame.data_ptr()), hdr_out=None):
        return r._lib.rrt_render_ss(r._ctx, C.byref(prm), C.byref(cam), C.byref(fx), C.c_uint64(sky.texture), 1.0, w_, h_,
                                    ss, C.byref(band) if band is not None else None, d_out, rrt.OUT_FRAME, hdr_out, st)

    def resolve(ss=2, w_=w, h_=h, band=None, hdr_hi=C.c_void_p(hi.data_ptr()), d_out=C.c_void_p(frame.data_ptr()),
                hdr_out=None):
        return r._lib.rrt_resolve(r._ctx, C.byref(prm), C.byref(fx), ss, w_, h_, C.byref(band) if band is not None else None,
                                  hdr_hi, d_out, rrt.OUT_FRAME, hdr_out, st)

    big = rrt.Band(0, 1, 1)
    l0 = r.kernel_launches()
    for fn in (render_ss, resolve):
        for bad in (dict(ss=0), dict(ss=9), dict(ss=-1), dict(d_out=None), dict(w_=0), dict(ss=8, w_=1 << 28),
                    dict(band=rrt.Band(3, 3, 8)), dict(ss=8, w_=1 << 16, h_=1 << 12, band=big)):
            assert fn(**bad) == rrt._capi.ERR_BAD_ARG, (fn.__name__, bad)
    assert resolve(hdr_hi=None) == rrt._capi.ERR_BAD_ARG
    hi_base = hi.data_ptr()
    for off in (0, 16 * (4 * w * h - 1), -16 * (w * h - 1)):   # hdr_out sharing a float4 with hdr_hi, at either end
        assert resolve(hdr_out=C.c_void_p(hi_base + off)) == rrt._capi.ERR_BAD_ARG, off
    assert r.kernel_launches() == l0
    # a separate plane is fine, and so is an hdr-only call
    assert resolve(hdr_out=C.c_void_p(hdr.data_ptr())) == 0
    assert render_ss(d_out=None, hdr_out=C.c_void_p(hdr.data_ptr())) == 0
    # planes that touch hdr_hi without sharing a byte are accepted, at either end: one allocation holds
    # [hdr_out | hdr_hi | hdr_out], so every write stays inside it
    buf = _hdr(r, w, 6 * h, float("nan"))   # w*h + 4*w*h + w*h float4
    lo, mid, up = buf[:h], buf[h:5 * h].view(2 * h, 2 * w, 4), buf[5 * h:]
    mid.copy_(hi)
    for out_plane in (lo, up):
        assert resolve(hdr_hi=C.c_void_p(mid.data_ptr()), hdr_out=C.c_void_p(out_plane.data_ptr())) == 0
    _, want = _resolve(r, (prm, None, fx, None), hi, 2, w, h)
    got_lo, got_up, got_mid, hi_np = _np(lo, up, mid, hi)
    assert np.array_equal(got_lo, want) and np.array_equal(got_up, want) and np.array_equal(got_mid, hi_np)
