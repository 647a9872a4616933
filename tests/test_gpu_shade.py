"""rrt_shade / Renderer.shade: the step after the ray loop (sky, final_hdr = I + bg*T, bloom, vignette, CA, tonemap,
row-flipped store) run again from the planes of an earlier render.  It calls the render kernels' own finish_ray_inl with
the exit state they stored, so every byte it writes must be the byte a fresh rrt_render writes with the new sky, exposure
and bloom / vignette / CA settings: exact equality for the uchar4 frame and the hdr plane, in both rounding contracts,
with and without media, through the packed and scalar tracers, for bands, tiny and full-size frames."""
import ctypes as C

import numpy as np
import pytest

from parity import CAMERAS

pytestmark = pytest.mark.gpu

# (sky, exposure, effect fields changed from the trace's) -- the first repeats the trace's own settings
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


def _trace(r, sky, cam, spin, flags, w, h, band=None, **fx_over):
    """Planes (TRACE_PLANES) of one render with the default effects, exposure 0.8 and `sky`."""
    import relativisticraytracer_b200 as rrt
    traced = r.alloc_planes(w, h, rrt.TRACE_PLANES)
    kw = dict(band=band, layout=rrt.OUT_PACKED) if band is not None else {}
    r.render(rrt.default_params(spin_a=spin, flags=flags, exposure=0.8), rrt.camera_state_from(*CAMERAS[cam]),
             rrt.default_effects(**fx_over), sky, 1.0, w, h, planes=traced, **kw)
    return traced


def _variant(skies, flags, variant, **fx_over):
    import relativisticraytracer_b200 as rrt
    sky, exposure, over = variant
    return (rrt.default_params(flags=flags, exposure=exposure), rrt.default_effects(**{**fx_over, **over}), skies[sky])


def _fresh(r, skies, cam, spin, flags, w, h, variant, **fx_over):
    """(frame, hdr plane) of a new render with the variant's sky, exposure and effects."""
    import relativisticraytracer_b200 as rrt
    import torch
    prm, fx, sky = _variant(skies, flags, variant, **fx_over)
    prm.spin_a = spin
    hdr = torch.empty((h, w, 4), dtype=torch.float32, device=r.device)
    out = r.render(prm, rrt.camera_state_from(*CAMERAS[cam]), fx, sky, 1.0, w, h, planes={"hdr": hdr})
    torch.cuda.synchronize()
    return out.cpu().numpy(), hdr.cpu().numpy()


def _shade(r, skies, traced, flags, w, h, variant, **fx_over):
    import torch
    prm, fx, sky = _variant(skies, flags, variant, **fx_over)
    hdr = torch.empty((h, w, 4), dtype=torch.float32, device=r.device)
    out = r.shade(prm, fx, sky, traced, w, h, hdr_out=hdr)
    torch.cuda.synchronize()
    return out.cpu().numpy(), hdr.cpu().numpy()


def _same(got, want, tag):
    for name, a, b in zip(("frame", "hdr"), got, want):
        assert np.array_equal(a, b, equal_nan=True), f"{tag}: {name} differs on {np.sum(a != b)} elements"


def _check_variants(r, skies, cam, spin, flags, w, h, tag, **fx_over):
    traced = _trace(r, skies["small"], cam, spin, flags, w, h, **fx_over)
    for k, v in enumerate(VARIANTS):
        _same(_shade(r, skies, traced, flags, w, h, v, **fx_over), _fresh(r, skies, cam, spin, flags, w, h, v, **fx_over),
              f"{tag} variant {k}")


@pytest.mark.parametrize("cam", ["C0", "C1", "C2", "C3"])
@pytest.mark.parametrize("spin,flags", [(0.99, 7), (0.0, 7), (0.99, 5), (0.99, 4), (0.99, 3), (0.0, 1)])
def test_shade_reproduces_render(env, cam, spin, flags):
    """FMAD with media (split pipeline, packed tracer), FMAD without media (packed fused kernel), strict with media
    (split pipeline, scalar tracer)."""
    r, skies = env
    _check_variants(r, skies, cam, spin, flags, 203, 117, f"{cam} a={spin} flags={flags}")


def test_shade_with_lens_off(env):
    r, skies = env
    _check_variants(r, skies, "C1", 0.99, 7, 203, 117, "lens off", use_lens=0)


@pytest.mark.parametrize("layout", ["frame", "packed"])
def test_shade_bands(env, layout):
    """Only the band's rows are written (the others keep a sentinel) and they equal rrt_render's for that band."""
    import relativisticraytracer_b200 as rrt
    import torch
    from relativisticraytracer_b200.parallel import band_rows_of
    r, skies = env
    w, h, cam = 160, 90, "C1"
    lay = rrt.OUT_FRAME if layout == "frame" else rrt.OUT_PACKED
    for band in (rrt.Band(0, 3, 8), rrt.Band(2, 3, 8), rrt.Band(1, 2, 1)):
        rows = band_rows_of(band.rank, band.nranks, band.group, h)
        own = (h - 1 - rows) if lay == rrt.OUT_FRAME else np.arange(len(rows))   # buffer rows the band writes
        others = np.setdiff1d(np.arange(h), own)
        assert len(others) > 0
        traced = _trace(r, skies["small"], cam, 0.99, 7, w, h, band=band)
        for k, v in enumerate(VARIANTS):
            res = []
            for how in ("shade", "render"):
                prm, fx, sky = _variant(skies, 7, v)
                out = torch.full((h, w, 4), 77, dtype=torch.uint8, device=r.device)   # h rows for either layout
                hdr = torch.full((h, w, 4), float("nan"), dtype=torch.float32, device=r.device)
                if how == "shade":
                    r.shade(prm, fx, sky, traced, w, h, band=band, out=out, layout=lay, hdr_out=hdr)
                else:
                    prm.spin_a = 0.99
                    r.render(prm, rrt.camera_state_from(*CAMERAS[cam]), fx, sky, 1.0, w, h, band=band, out=out, layout=lay,
                             planes={"hdr": hdr})
                torch.cuda.synchronize()
                res.append((out.cpu().numpy(), hdr.cpu().numpy()))
            tag = f"{layout} band {band.rank}/{band.nranks}x{band.group} variant {k}"
            _same(res[0], res[1], tag)
            frame, hdr = res[0]
            assert (frame[others] == 77).all(), f"{tag}: rows outside the band were written"
            assert (frame[own] != 77).any(), tag
            assert np.isnan(np.delete(hdr, rows, axis=0)).all(), f"{tag}: hdr outside the band was written"


@pytest.mark.parametrize("w,h,cam", [(1, 1, "C3"), (3, 5, "C1"), (1920, 1080, "C0"), (1920, 1080, "C3"), (3840, 2160, "C0")])
def test_shade_sizes(env, w, h, cam):
    r, skies = env
    _check_variants(r, skies, cam, 0.99, 7, w, h, f"{w}x{h} {cam}")


def test_shade_hdr_in_place_and_without_frame(env):
    """hdr_out may be traced["hdr"] itself (T in .w survives, so the planes can be shaded again); through the C ABI a
    shade may write hdr_out alone."""
    import relativisticraytracer_b200 as rrt
    import torch
    r, skies = env
    w, h, cam, spin, flags = 203, 117, "C3", 0.99, 7
    traced = _trace(r, skies["small"], cam, spin, flags, w, h)
    for v in (VARIANTS[1], VARIANTS[0], VARIANTS[2]):
        prm, fx, sky = _variant(skies, flags, v)
        out = r.shade(prm, fx, sky, traced, w, h, hdr_out=traced["hdr"])
        torch.cuda.synchronize()
        _same((out.cpu().numpy(), traced["hdr"].cpu().numpy()), _fresh(r, skies, cam, spin, flags, w, h, v), "in place")

    traced = _trace(r, skies["small"], cam, spin, flags, w, h)
    prm, fx, sky = _variant(skies, flags, VARIANTS[1])
    hdr = torch.empty((h, w, 4), dtype=torch.float32, device=r.device)
    pl = rrt.Planes(**{n: t.data_ptr() for n, t in traced.items()})
    r._check(r._lib.rrt_shade(r._ctx, C.byref(prm), C.byref(fx), C.c_uint64(sky.texture), w, h, None, C.byref(pl), None,
                              rrt.OUT_FRAME, C.c_void_p(hdr.data_ptr()), C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    assert np.array_equal(hdr.cpu().numpy(), _fresh(r, skies, cam, spin, flags, w, h, VARIANTS[1])[1], equal_nan=True)


def test_shade_fused_and_split_traces_agree(env, sky_small, sky_smooth):
    """Planes traced by the fused kernel and by the split pipeline shade to the same bytes."""
    import relativisticraytracer_b200 as rrt
    r, skies = env
    w, h, flags = 203, 117, 7
    fused = rrt.Renderer(0)
    try:
        fused.set_pipeline("fused")
        fsky = {"small": fused.create_sky(sky_small), "smooth": fused.create_sky(sky_smooth)}
        for cam in ("C1", "C3"):
            a = _trace(fused, fsky["small"], cam, 0.99, flags, w, h)
            b = _trace(r, skies["small"], cam, 0.99, flags, w, h)
            for v in VARIANTS:
                _same(_shade(fused, fsky, a, flags, w, h, v), _shade(r, skies, b, flags, w, h, v), f"{cam} fused vs split trace")
        for s in fsky.values():
            s.close()
    finally:
        fused.close()


_PEER_RANK = """
import sys
import numpy as np
import torch
import relativisticraytracer_b200 as rrt
from test_gpu_shade import VARIANTS, _trace, _variant
handle, sky_dir, w, h, cam, rank, nranks, group = sys.argv[1:]
w, h, band = int(w), int(h), rrt.Band(int(rank), int(nranks), int(group))
r = rrt.Renderer(0)
skies = {n: r.create_sky(np.load(f"{sky_dir}/{n}.npy")) for n in ("small", "smooth")}
try:
    peer = rrt.PeerFrame(r, h, w, handle=bytes.fromhex(handle))
except rrt.RrtError as e:
    print(e)
    sys.exit(77)
traced = _trace(r, skies["small"], cam, 0.99, 7, w, h, band=band)
r.shade(*_variant(skies, 7, VARIANTS[1]), traced, w, h, band=band, out=peer)
torch.cuda.synchronize()
peer.close()
"""


def test_shade_into_a_peer_frame(env, sky_small, sky_smooth, tmp_path):
    """Each rank of a band-parallel frame re-shades its own band straight into rank 0's frame.  Rank 1 is a second process
    on the same GPU that maps rank 0's frame (a CUDA IPC handle cannot be opened by the process that created it)."""
    import os
    import subprocess
    import sys
    import relativisticraytracer_b200 as rrt
    import torch
    r, skies = env
    w, h, cam, group = 160, 90, "C1", 8
    np.save(tmp_path / "small.npy", sky_small)
    np.save(tmp_path / "smooth.npy", sky_smooth)
    peer = rrt.PeerFrame(r, h, w)
    try:
        band = rrt.Band(0, 2, group)
        traced = _trace(r, skies["small"], cam, 0.99, 7, w, h, band=band)
        r.shade(*_variant(skies, 7, VARIANTS[1]), traced, w, h, band=band, out=peer)
        torch.cuda.synchronize()
        tests = os.path.dirname(os.path.abspath(__file__))
        env_vars = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.dirname(tests), tests, os.environ.get("PYTHONPATH", "")]))
        res = subprocess.run([sys.executable, "-c", _PEER_RANK, peer.handle.hex(), str(tmp_path), str(w), str(h), cam, "1", "2",
                              str(group)], env=env_vars, capture_output=True, text=True, timeout=600)
        if res.returncode == 77:
            pytest.skip(f"CUDA IPC mapping unavailable: {res.stdout.strip()}")
        assert res.returncode == 0, res.stderr[-3000:]
        got = torch.empty((h, w, 4), dtype=torch.uint8, device=r.device)
        peer.read_into(got)
        torch.cuda.synchronize()
        assert np.array_equal(got.cpu().numpy(), _fresh(r, skies, cam, 0.99, 7, w, h, VARIANTS[1])[0])
    finally:
        peer.close()


def test_shade_on_a_side_stream_counters_and_launches(env):
    import torch
    r, skies = env
    w, h, cam, spin, flags = 203, 117, "C1", 0.99, 7
    traced = _trace(r, skies["small"], cam, spin, flags, w, h)
    torch.cuda.synchronize()
    r.read_counters(reset=True)
    want = _shade(r, skies, traced, flags, w, h, VARIANTS[1])
    prm, fx, sky = _variant(skies, flags, VARIANTS[1])
    side = torch.cuda.Stream()
    hdr = torch.empty((h, w, 4), dtype=torch.float32, device=r.device)
    l0 = r.kernel_launches()
    with torch.cuda.stream(side):
        out = r.shade(prm, fx, sky, traced, w, h, hdr_out=hdr, stream=side)
    side.synchronize()
    _same((out.cpu().numpy(), hdr.cpu().numpy()), want, "side stream")
    for k in range(5):
        r.shade(*_variant(skies, flags, VARIANTS[k % 3]), traced, w, h)
    assert r.kernel_launches() - l0 == 6
    assert all(v == 0 for v in r.read_counters().values())


def test_shade_errors(env):
    import relativisticraytracer_b200 as rrt
    import torch
    r, skies = env
    w, h, flags = 32, 16, 7
    traced = _trace(r, skies["small"], "C1", 0.99, flags, w, h)
    prm, fx, sky = _variant(skies, flags, VARIANTS[0])
    for missing in rrt.TRACE_PLANES:
        part = {n: t for n, t in traced.items() if n != missing}
        with pytest.raises(rrt.RrtError) as e:
            r.shade(prm, fx, sky, part, w, h)
        assert e.value.code == rrt._capi.ERR_BAD_ARG, missing
    for band in (rrt.Band(3, 3, 8), rrt.Band(0, 0, 8), rrt.Band(0, 2, 0)):
        with pytest.raises(rrt.RrtError) as e:
            r.shade(prm, fx, sky, traced, w, h, band=band)
        assert e.value.code == rrt._capi.ERR_BAD_ARG
    with pytest.raises(rrt.RrtError) as e:
        r.shade(prm, fx, 0, traced, w, h)
    assert e.value.code == rrt._capi.ERR_BAD_ARG

    pl = rrt.Planes(**{n: t.data_ptr() for n, t in traced.items()})
    frame = torch.empty((h, w, 4), dtype=torch.uint8, device=r.device)
    hdr = torch.empty((h, w, 4), dtype=torch.float32, device=r.device)

    def shade(w_=w, h_=h, planes=C.byref(pl), d_out=C.c_void_p(frame.data_ptr()), hdr_out=None, layout=rrt.OUT_FRAME):
        r._check(r._lib.rrt_shade(r._ctx, C.byref(prm), C.byref(fx), C.c_uint64(sky.texture), w_, h_, None, planes,
                                  d_out, layout, hdr_out, None))

    for bad in (dict(d_out=None), dict(w_=0), dict(w_=-3), dict(h_=0), dict(layout=2), dict(planes=None)):
        with pytest.raises(rrt.RrtError) as e:
            shade(**bad)
        assert e.value.code == rrt._capi.ERR_BAD_ARG, bad
    shade()
    shade(d_out=None, hdr_out=C.c_void_p(hdr.data_ptr()))
    torch.cuda.synchronize()
