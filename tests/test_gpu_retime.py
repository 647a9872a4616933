"""rrt_capture_* / Renderer.capture / Capture.render: one trace, renders at other times.

The trace does not read the time (only the disk and dust densities do), so a capture keeps the trace's media samples and the
state of the rays it finished, and each render evaluates the media at its own time, folds, shades and stores.  Every byte
and hdr value it writes must be the one a fresh rrt_render writes at that time: exact equality throughout, in both rounding
contracts, through the packed and scalar tracers, for bands, sizes, left-over tiles, supersampling and streams."""
import ctypes as C

import numpy as np
import pytest

from parity import CAMERAS

pytestmark = pytest.mark.gpu

# (sky, exposure, effect fields changed from the capture's), as in test_gpu_shade.py
VARIANTS = [
    ("small", 0.8, {}),
    ("smooth", 1.7, dict(use_bloom=0, use_vignette=1, vignette_intensity=0.7, use_ca=1, ca_amount=0.01)),
    ("small", 0.5, dict(bloom_threshold=0.3)),
]
TIMES = (1.0, 0.0, 123.5, 7.25)   # not monotonic; 1.0 is the time the other GPU tests trace at


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


def _prm(spin, flags, exposure=0.8):
    import relativisticraytracer_b200 as rrt
    return rrt.default_params(spin_a=spin, flags=flags, exposure=exposure)


def _capture(r, skies, cam, spin, flags, w, h, **kw):
    """A capture with exposure 0.8, the default effects (overridden by fx_over) and the small sky."""
    import relativisticraytracer_b200 as rrt
    fx_over = kw.pop("fx_over", {})
    return r.capture(_prm(spin, flags), rrt.camera_state_from(*CAMERAS[cam]), rrt.default_effects(**fx_over), skies["small"], w, h,
                     **kw)


def _variant(skies, spin, flags, variant, fx_over=None):
    import relativisticraytracer_b200 as rrt
    sky, exposure, over = variant
    return _prm(spin, flags, exposure), rrt.default_effects(**{**(fx_over or {}), **over}), skies[sky]


def _np(*ts):
    import torch
    torch.cuda.synchronize()
    return tuple(t.cpu().numpy() for t in ts)


def _hdr(r, w, h, fill=0.0):
    import torch
    return torch.full((h, w, 4), fill, dtype=torch.float32, device=r.device)


def _retimed(r, cap, args, t, **kw):
    """(frame, hdr plane) of Capture.render."""
    hdr = _hdr(r, cap.w, cap.h)
    out = cap.render(*args, t, hdr_out=hdr, **kw)
    return _np(out, hdr)


def _fresh(r, cam, args, t, w, h, **kw):
    """(frame, hdr plane) of a new rrt_render with the same parameters."""
    import relativisticraytracer_b200 as rrt
    prm, fx, sky = args
    hdr = _hdr(r, w, h)
    out = r.render(prm, rrt.camera_state_from(*CAMERAS[cam]), fx, sky, t, w, h, planes={"hdr": hdr}, **kw)
    return _np(out, hdr)


def _same(got, want, tag):
    for name, a, b in zip(("frame", "hdr"), got, want):
        assert np.array_equal(a, b, equal_nan=True), f"{tag}: {name} differs on {np.sum(a != b)} elements"


@pytest.mark.parametrize("cam", ["C0", "C1", "C2", "C3"])
@pytest.mark.parametrize("spin,flags", [(0.99, 7), (0.0, 7), (0.99, 5), (0.99, 3), (0.0, 1)])
def test_capture_renders_are_renders(env, cam, spin, flags):
    """FMAD through the packed tracer (7, 5), strict through the scalar one (3, 1); one capture, four times."""
    r, skies = env
    w, h = 203, 117
    cap = _capture(r, skies, cam, spin, flags, w, h)
    info = cap.info()
    assert info["packed"] == bool(flags & 4) and info["tiles_left"] == 0 and info["samples"] > 0
    args = _variant(skies, spin, flags, VARIANTS[0])
    for t in TIMES:
        _same(_retimed(r, cap, args, t), _fresh(r, cam, args, t, w, h), f"{cam} a={spin} flags={flags} t={t}")
    cap.close()


@pytest.mark.parametrize("lens", [1, 0])
def test_shading_variants(env, lens):
    r, skies = env
    w, h, cam, spin, flags = 203, 117, "C3", 0.99, 7
    cap = _capture(r, skies, cam, spin, flags, w, h, fx_over=dict(use_lens=lens))
    for k, v in enumerate(VARIANTS):
        args = _variant(skies, spin, flags, v, dict(use_lens=lens))
        for t in (123.5, 1.0):
            _same(_retimed(r, cap, args, t), _fresh(r, cam, args, t, w, h), f"lens={lens} variant {k} t={t}")
    cap.close()


def _left_over_captures(r, skies, cam, spin, flags, w, h):
    """(capture holding part of the frame, capture holding none of it): the first pool size that leaves some tiles."""
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
def test_left_over_tiles(env, spin, flags):
    """Tiles whose samples do not fit the capture's pool are rendered by the fused sweep at every render."""
    r, skies = env
    w, h, cam = 203, 117, "C1"
    for cap in _left_over_captures(r, skies, cam, spin, flags, w, h):
        for t in (123.5, 1.0):
            args = _variant(skies, spin, flags, VARIANTS[1])
            _same(_retimed(r, cap, args, t), _fresh(r, cam, args, t, w, h), f"{cap.info()} t={t}")
        cap.close()


@pytest.mark.parametrize("layout", ["frame", "packed"])
def test_bands(env, layout):
    """Only the band's rows are written (the others keep a sentinel) and they equal rrt_render's for that band."""
    import relativisticraytracer_b200 as rrt
    import torch
    from relativisticraytracer_b200.parallel import band_rows_of
    r, skies = env
    w, h, cam, spin, flags = 160, 90, "C1", 0.99, 7
    lay = rrt.OUT_FRAME if layout == "frame" else rrt.OUT_PACKED
    for band in (rrt.Band(0, 3, 8), rrt.Band(2, 3, 8), rrt.Band(1, 2, 1)):
        rows = band_rows_of(band.rank, band.nranks, band.group, h)
        own = (h - 1 - rows) if lay == rrt.OUT_FRAME else np.arange(len(rows))   # buffer rows the band writes
        others = np.setdiff1d(np.arange(h), own)
        cap = _capture(r, skies, cam, spin, flags, w, h, band=band)
        for k, v in enumerate(VARIANTS[:2]):
            args = _variant(skies, spin, flags, v)
            res = []
            for how in ("capture", "render"):
                out = torch.full((h, w, 4), 77, dtype=torch.uint8, device=r.device)   # h rows for either layout
                hdr = _hdr(r, w, h, float("nan"))
                if how == "capture":
                    cap.render(*args, 7.25, out=out, layout=lay, hdr_out=hdr)
                else:
                    prm, fx, sky = args
                    r.render(prm, rrt.camera_state_from(*CAMERAS[cam]), fx, sky, 7.25, w, h, band=band, out=out, layout=lay,
                             planes={"hdr": hdr})
                res.append(_np(out, hdr))
            tag = f"{layout} band {band.rank}/{band.nranks}x{band.group} variant {k}"
            _same(res[0], res[1], tag)
            frame, hdr = res[0]
            assert (frame[others] == 77).all(), f"{tag}: rows outside the band were written"
            assert (frame[own] != 77).any(), tag
            assert np.isnan(np.delete(hdr, rows, axis=0)).all(), f"{tag}: hdr outside the band was written"
        cap.close()


@pytest.mark.parametrize("w,h,cam", [(1, 1, "C3"), (7, 5, "C1"), (1920, 1080, "C0"), (1920, 1080, "C3"), (3840, 2160, "C0")])
def test_sizes(env, w, h, cam):
    r, skies = env
    cap = _capture(r, skies, cam, 0.99, 7, w, h)
    for t in (123.5, 1.0):
        args = _variant(skies, 0.99, 7, VARIANTS[1])
        _same(_retimed(r, cap, args, t), _fresh(r, cam, args, t, w, h), f"{w}x{h} {cam} t={t}")
    cap.close()


def test_supersampled(env):
    """A capture at 2w x 2h rendered into an hdr plane and resolved is render_ss(ss=2) at that time."""
    import relativisticraytracer_b200 as rrt
    r, skies = env
    w, h, cam, ss = 61, 37, "C3", 2
    cap = _capture(r, skies, cam, 0.99, 7, ss * w, ss * h)
    for t in (123.5, 7.25):
        prm, fx, sky = _variant(skies, 0.99, 7, VARIANTS[1])
        hi = _hdr(r, ss * w, ss * h)
        cap.render(prm, fx, sky, t, hdr_out=hi)
        got = _np(r.resolve(prm, fx, hi, ss, w, h, hdr_out=(hd := _hdr(r, w, h))), hd)
        hd2 = _hdr(r, w, h)
        want = _np(r.render_ss(prm, rrt.camera_state_from(*CAMERAS[cam]), fx, sky, t, w, h, ss, hdr_out=hd2), hd2)
        _same(got, want, f"ss={ss} t={t}")
    cap.close()


@pytest.mark.parametrize("left_over", [False, True])
def test_counters_and_launches(env, left_over):
    """capture + one render counts what one rrt_render counts; 1 launch per capture, 3 per render (4 with a sweep)."""
    r, skies = env
    w, h, cam, spin, flags = 203, 117, "C1", 0.99, 7
    args = _variant(skies, spin, flags, VARIANTS[0])
    max_bytes = 0
    if left_over:
        part, none = _left_over_captures(r, skies, cam, spin, flags, w, h)
        max_bytes = part.info()["pool_bytes"]
        part.close()
        none.close()
    r.read_counters(reset=True)
    _fresh(r, cam, args, 7.25, w, h)
    want = r.read_counters(reset=True)
    l0 = r.kernel_launches()
    cap = _capture(r, skies, cam, spin, flags, w, h, max_bytes=max_bytes)
    assert (cap.info()["tiles_left"] > 0) == left_over
    assert r.kernel_launches() - l0 == 1
    traced = r.read_counters(reset=True)
    assert traced["dense_samples"] == traced["n_touched"] == 0 and traced["rk4_steps"] > 0
    for t in (7.25, 123.5, 7.25):
        l0 = r.kernel_launches()
        _retimed(r, cap, args, t)
        assert r.kernel_launches() - l0 == (4 if left_over else 3)
        got = r.read_counters(reset=True)
        if t == 7.25:
            assert {k: traced[k] + got[k] for k in want} == want, (traced, got, want)
    assert want["dense_samples"] > 0
    cap.close()


def test_two_captures_and_two_streams(env):
    import torch
    r, skies = env
    w, h = 96, 54
    a = _capture(r, skies, "C1", 0.99, 7, w, h)
    b = _capture(r, skies, "C3", 0.0, 3, w, h)
    aa, ba = _variant(skies, 0.99, 7, VARIANTS[0]), _variant(skies, 0.0, 3, VARIANTS[1])
    want = {(k, t): _fresh(r, cam, args, t, w, h) for k, cam, args in (("a", "C1", aa), ("b", "C3", ba)) for t in (0.0, 123.5)}
    got = {}
    for t in (0.0, 123.5):   # interleaved renders of two live captures
        got[("a", t)] = _retimed(r, a, aa, t)
        got[("b", t)] = _retimed(r, b, ba, t)
    for k in want:
        _same(got[k], want[k], f"capture {k}")
    # one capture on two streams back to back, no host synchronisation in between
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    hdrs = [_hdr(r, w, h) for _ in range(4)]
    torch.cuda.synchronize()
    outs = []
    for k, t in enumerate((0.0, 123.5, 0.0, 123.5)):
        st = s1 if k % 2 == 0 else s2
        with torch.cuda.stream(st):
            outs.append((a.render(*aa, t, hdr_out=hdrs[k], stream=st), hdrs[k], t))
    torch.cuda.synchronize()
    for k, (out, hdr, t) in enumerate(outs):
        _same(_np(out, hdr), want[("a", t)], f"stream render {k}")
    a.close()
    b.close()


def test_errors(env):
    import relativisticraytracer_b200 as rrt
    import torch
    r, skies = env
    w, h, cam = 32, 16, "C1"
    ok = rrt._capi.ERR_BAD_ARG
    with pytest.raises(rrt.RrtError) as e:   # no medium: nothing depends on the time
        _capture(r, skies, cam, 0.99, 4, w, h)
    assert e.value.code == ok
    with pytest.raises(rrt.RrtError) as e:
        r.capture(rrt.default_params(max_steps=1 << 20), rrt.camera_state_from(*CAMERAS[cam]), rrt.default_effects(),
                  skies["small"], w, h)
    assert e.value.code == ok
    for band in (rrt.Band(3, 3, 8), rrt.Band(0, 2, 0)):
        with pytest.raises(rrt.RrtError) as e:
            _capture(r, skies, cam, 0.99, 7, w, h, band=band)
        assert e.value.code == ok
    cap = _capture(r, skies, cam, 0.99, 7, w, h)
    prm, fx, sky = _variant(skies, 0.99, 7, VARIANTS[0])
    frame = torch.empty((h, w, 4), dtype=torch.uint8, device=r.device)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def render(handle=cap._h, prm_=prm, fx_=fx, tex=sky.texture, d_out=C.c_void_p(frame.data_ptr()), layout=rrt.OUT_FRAME):
        return r._lib.rrt_capture_render(handle, C.byref(prm_), C.byref(fx_), C.c_uint64(tex), 1.0, d_out, layout, None, st)

    l0 = r.kernel_launches()
    for bad in (dict(prm_=_prm(0.99, 3)), dict(fx_=rrt.default_effects(use_lens=0)), dict(fx_=rrt.default_effects(distortion_amount=0.2)),
                dict(layout=2), dict(d_out=None), dict(tex=0), dict(handle=None)):
        assert render(**bad) == ok, bad
    assert r.kernel_launches() == l0
    info = (C.c_uint64 * 8)()
    assert r._lib.rrt_capture_info(None, info) == ok
    assert render() == 0 and render(prm_=_prm(0.0, 7, 2.0)) == 0   # other fields of prm are not the capture's to change
    torch.cuda.synchronize()
    cap.close()
    cap.close()
