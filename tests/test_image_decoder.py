"""The native skybox decoder (C ABI rrt_image_load / rrt_image_decode, csrc/rrt_image.cpp) against stb_image itself.

The reference decodes its skybox with stbi_load(path, &w, &h, &c, 4) (src/main.cpp:240; stb_image v2.30 is vendored in
the reference tree).  Checker: oracle/_ref/libref_stb.so = that header compiled where it lies (oracle/ref_stb.c).  The
product's bytes must equal stb_image's byte for byte -- on the two assets the reference ships, and on files generated
here with PIL that walk the decoder's subset: JPEG 4:4:4 / 4:2:2 / 4:2:0 / 4:4:0 / 4:1:1, grey, odd sizes, restart
intervals, high and low quality; PNG grey / grey+alpha / RGB / RGBA / palette (1, 2, 4, 8 bit, with tRNS), all five
row filters.  Files outside the subset must be refused, not decoded differently.  Where stb_image is not built, the PNG
files are checked against PIL's decoder instead (see png_ref).  CPU only."""
import ctypes as C
import hashlib
import io
import json
import os

import numpy as np
import pytest

# the reference's skybox assets, where a copy of its tree is named by RRT_REFERENCE_TREE
REF_ASSETS = os.path.join(os.environ["RRT_REFERENCE_TREE"], "assets", "skyboxes") if "RRT_REFERENCE_TREE" in os.environ else None
# sha256 of the RGBA8 bytes stb_image v2.30 returns for the reference's assets (the pin when the tree is absent is
# the synthetic-file test below; these two make sure the shipped files themselves keep decoding to the same bytes)
GOLDEN_SHA256 = {
    "skybox2.jpg": (4096, 2048, "5447bcf9da311a4e958fd0e6f491b0d68d13edea71a401239100e9e049fc5174"),
    "skybox.png": (1024, 1024, "0e2c39dadbbc7c3f6cffaf57467ac21992b99933e8fbc502c7c26afb430d261f"),
}


STB_LIB = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref", "libref_stb.so")
# The JPEG files the JPEG tests decode, as PIL wrote them from _gradient (write_jpeg), and the sha256 of the RGBA8 bytes
# stb_image returns for each (tests/tools/make_golden_jpeg.py): the check where libref_stb.so is not built.
JPEG_GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "jpeg")


@pytest.fixture(scope="module")
def stb(built):
    if not os.path.exists(STB_LIB):
        pytest.skip("oracle/_ref/libref_stb.so not built (reference tree absent at build time)")
    return _stb_loader(STB_LIB)


@pytest.fixture(scope="module")
def stb_if_built(built):
    return _stb_loader(STB_LIB) if os.path.exists(STB_LIB) else None


@pytest.fixture(scope="module")
def png_ref(built):
    """Checker for PNG files: stb_image where oracle/_ref/libref_stb.so is built, else PIL.  PNG is lossless, so its RGBA8
    bytes are fixed by the file and every conforming decoder returns the same ones (not so for JPEG, whose IDCT and chroma
    upsampling differ from decoder to decoder: the JPEG tests check stb_image's own bytes, see JPEG_GOLD)."""
    if os.path.exists(STB_LIB):
        return _stb_loader(STB_LIB)
    from PIL import Image
    return lambda path: np.asarray(Image.open(path).convert("RGBA"))


def _stb_loader(path):
    lib = C.CDLL(path)
    lib.refstb_load.restype = C.POINTER(C.c_uint8)
    lib.refstb_load.argtypes = [C.c_char_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.refstb_free.argtypes = [C.POINTER(C.c_uint8)]

    def load(path):
        w, h, c = C.c_int(), C.c_int(), C.c_int()
        p = lib.refstb_load(path.encode(), C.byref(w), C.byref(h), C.byref(c))
        if not p:
            return None
        a = np.ctypeslib.as_array(p, shape=(h.value, w.value, 4)).copy()
        lib.refstb_free(p)
        return a
    return load


def _gradient(w, h, seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    y, x = np.mgrid[0:h, 0:w]
    img = np.stack([(x * 255 // max(w - 1, 1)), (y * 255 // max(h - 1, 1)), ((x + y) * 7) % 256], axis=-1).astype(np.float64)
    img += rng.normal(scale=25.0, size=img.shape)            # texture, so that every AC band and Huffman path is used
    img[h // 3: h // 3 + 5, :, :] = 255                      # hard edges: clamping in the IDCT and in the colour conversion
    img[:, w // 2: w // 2 + 3, :] = 0
    return np.clip(img, 0, 255).astype(np.uint8)


def test_reference_assets_decode_to_stb_bytes(built, stb):
    import relativisticraytracer_b200 as rrt
    if REF_ASSETS is None or not os.path.isdir(REF_ASSETS):
        pytest.skip("reference assets not present")
    for name, (w, h, sha) in GOLDEN_SHA256.items():
        path = os.path.join(REF_ASSETS, name)
        ours = rrt.decode_image(path)
        assert ours.shape == (h, w, 4)
        assert np.array_equal(ours, stb(path)), name
        assert hashlib.sha256(ours.tobytes()).hexdigest() == sha, name
        assert np.array_equal(rrt.load_skybox(path), ours)


JPEG_CASES = [
    # (w, h, PIL mode, subsampling, quality, extra save options)
    (64, 48, "RGB", "4:4:4", 90, {}),
    (67, 45, "RGB", "4:4:4", 75, {}),
    (160, 120, "RGB", "4:2:0", 85, {}),
    (161, 119, "RGB", "4:2:0", 60, {}),
    (33, 17, "RGB", "4:2:0", 95, {}),
    (1, 1, "RGB", "4:2:0", 90, {}),
    (2, 3, "RGB", "4:2:2", 90, {}),
    (130, 70, "RGB", "4:2:2", 80, {}),
    (131, 71, "RGB", "4:2:2", 30, {}),
    (96, 64, "L", None, 90, {}),
    (97, 65, "L", None, 50, {}),
    (200, 150, "RGB", "4:2:0", 100, {}),
    (200, 150, "RGB", "4:4:4", 5, {}),
    (256, 128, "RGB", "4:4:4", 92, {"restart_marker_blocks": 7}),
    (255, 127, "RGB", "4:2:0", 88, {"restart_marker_rows": 1}),
    (120, 90, "RGB", "4:2:0", 85, {"optimize": True}),
]


JPEG_411 = (150, 100, "RGB", "4:1:1", 85, {})   # seed 7


def jpeg_name(case):
    w, h, mode, sub, q, extra = case
    return f"{w}x{h}-{mode.lower()}-{(sub or 'grey').replace(':', '')}-q{q}" + "".join(f"-{k}" for k in extra) + ".jpg"


def write_jpeg(case, path):
    from PIL import Image
    w, h, mode, sub, q, extra = case
    img = _gradient(w, h, seed=7 if case == JPEG_411 else w * 1000 + h)
    kw = dict(quality=q, **extra)
    if sub is not None:
        kw["subsampling"] = sub
    Image.fromarray(img if mode == "RGB" else img[..., 0]).save(path, "JPEG", **kw)


def _check_jpeg_against_stb(case, stb_if_built):
    import relativisticraytracer_b200 as rrt
    w, h = case[:2]
    path = os.path.join(JPEG_GOLD, jpeg_name(case))
    got = rrt.decode_image(path)
    assert got.shape == (h, w, 4)
    if stb_if_built is not None:
        want = stb_if_built(path)
        assert np.array_equal(got, want), f"{int((got != want).sum())} bytes differ, max {int(np.abs(got.astype(int) - want).max())}"
    with open(os.path.join(JPEG_GOLD, "stb_rgba_sha256.json")) as f:
        assert hashlib.sha256(got.tobytes()).hexdigest() == json.load(f)[jpeg_name(case)], "bytes differ from stb_image's"


@pytest.mark.parametrize("case", JPEG_CASES, ids=lambda c: f"{c[0]}x{c[1]}-{c[2]}-{c[3]}-q{c[4]}" + ("-rst" if c[5] else ""))
def test_generated_jpeg_equals_stb(built, stb_if_built, case):
    _check_jpeg_against_stb(case, stb_if_built)


def test_jpeg_4_1_1_sampling_equals_stb(built, stb_if_built):
    """4:1:1 (chroma 4x1): stb_image has no filter for that ratio and falls back to nearest neighbour -- so must we."""
    _check_jpeg_against_stb(JPEG_411, stb_if_built)


def test_progressive_and_cmyk_jpeg_are_refused(built, tmp_path):
    from PIL import Image
    import relativisticraytracer_b200 as rrt
    from relativisticraytracer_b200 import _capi
    img = _gradient(64, 64, seed=3)
    p1 = str(tmp_path / "prog.jpg")
    Image.fromarray(img, "RGB").save(p1, "JPEG", quality=85, progressive=True)
    with pytest.raises(rrt.RrtError) as e:
        rrt.decode_image(p1)
    assert e.value.code == _capi.ERR_UNSUPPORTED
    p2 = str(tmp_path / "cmyk.jpg")
    Image.fromarray(img, "RGB").convert("CMYK").save(p2, "JPEG", quality=85)
    with pytest.raises(rrt.RrtError) as e:
        rrt.decode_image(p2)
    assert e.value.code == _capi.ERR_UNSUPPORTED
    with pytest.raises(rrt.RrtError) as e:
        rrt.decode_image(str(tmp_path / "missing.jpg"))
    assert e.value.code == _capi.ERR_IO
    p3 = str(tmp_path / "trunc.jpg")
    Image.fromarray(img, "RGB").save(p3, "JPEG", quality=85)
    data = open(p3, "rb").read()
    open(p3, "wb").write(data[:200])
    with pytest.raises(rrt.RrtError):
        rrt.decode_image(p3)


PNG_CASES = ["L", "LA", "RGB", "RGBA", "P", "P-trns", "1", "P2", "P4", "L-trns", "RGB-trns"]


@pytest.mark.parametrize("kind", PNG_CASES)
@pytest.mark.parametrize("size", [(61, 37), (128, 64), (1, 1), (7, 300)])
def test_generated_png_equals_stb(built, png_ref, tmp_path, kind, size):
    from PIL import Image
    import relativisticraytracer_b200 as rrt
    w, h = size
    img = _gradient(w, h, seed=w + 31 * h)
    rng = np.random.Generator(np.random.PCG64(5))
    kw = {}
    if kind == "L":
        im = Image.fromarray(img[..., 0], "L")
    elif kind == "LA":
        im = Image.fromarray(np.stack([img[..., 0], img[..., 1]], -1), "LA")
    elif kind == "RGB":
        im = Image.fromarray(img, "RGB")
    elif kind == "RGBA":
        im = Image.fromarray(np.concatenate([img, img[..., :1] ^ 0x5a], -1), "RGBA")
    elif kind in ("P", "P-trns", "P2", "P4"):
        ncol = {"P": 200, "P-trns": 200, "P2": 4, "P4": 16}[kind]
        im = Image.fromarray((img[..., 0].astype(int) * ncol // 256).astype(np.uint8), "P")
        im.putpalette(rng.integers(0, 256, size=ncol * 3, dtype=np.uint8).tobytes())
        if kind == "P-trns":
            kw["transparency"] = bytes(rng.integers(0, 256, size=150, dtype=np.uint8))
        if kind in ("P2", "P4"):
            kw["bits"] = 2 if kind == "P2" else 4
    elif kind == "1":
        im = Image.fromarray(img[..., 0] > 127).convert("1")
    elif kind == "L-trns":
        im = Image.fromarray(img[..., 0], "L")
        kw["transparency"] = int(img[0, 0, 0])
    elif kind == "RGB-trns":
        im = Image.fromarray(img, "RGB")
        kw["transparency"] = tuple(int(x) for x in img[0, 0])
    path = str(tmp_path / "t.png")
    im.save(path, "PNG", **kw)
    want = png_ref(path)
    assert want is not None
    got = rrt.decode_image(path)
    assert got.shape == want.shape == (h, w, 4)
    assert np.array_equal(got, want), f"{kind}: {int((got != want).sum())} bytes differ"


def test_png_16bit_and_interlaced_are_refused(built, tmp_path):
    from PIL import Image
    import relativisticraytracer_b200 as rrt
    from relativisticraytracer_b200 import _capi
    img = _gradient(40, 30, seed=9)
    p1 = str(tmp_path / "i16.png")
    Image.fromarray((img[..., 0].astype(np.uint16) * 257), "I;16").save(p1, "PNG")
    with pytest.raises(rrt.RrtError) as e:
        rrt.decode_image(p1)
    assert e.value.code == _capi.ERR_UNSUPPORTED
    # Adam7: PIL cannot write interlaced PNGs; flip the interlace byte of a valid header (the CRC is not checked by
    # stb_image either) -- the decoder must refuse rather than read the rows as if they were progressive
    p2 = str(tmp_path / "adam7.png")
    Image.fromarray(img, "RGB").save(p2, "PNG")
    data = bytearray(open(p2, "rb").read())
    assert data[12:16] == b"IHDR"
    data[28] = 1
    open(p2, "wb").write(bytes(data))
    with pytest.raises(rrt.RrtError) as e:
        rrt.decode_image(p2)
    assert e.value.code == _capi.ERR_UNSUPPORTED


def test_decode_from_memory_and_stored_deflate_blocks(built, png_ref, tmp_path):
    """rrt_image_decode on a buffer, and a PNG whose zlib stream uses stored (uncompressed) blocks."""
    import struct
    import zlib
    import relativisticraytracer_b200 as rrt
    from relativisticraytracer_b200 import _capi
    w, h = 50, 20
    img = _gradient(w, h, seed=11)
    raw = b"".join(b"\x00" + img[y].tobytes() for y in range(h))
    comp = zlib.compressobj(level=0)
    z = comp.compress(raw) + comp.flush()

    def chunk(t, d):
        return struct.pack(">I", len(d)) + t + d + struct.pack(">I", zlib.crc32(t + d) & 0xffffffff)
    png = b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, 8, 2, 0, 0, 0)) + chunk(b"IDAT", z[:100]) + \
        chunk(b"IDAT", z[100:]) + chunk(b"IEND", b"")
    path = str(tmp_path / "stored.png")
    open(path, "wb").write(png)
    lib = _capi.load()
    px, ww, hh = C.POINTER(C.c_uint8)(), C.c_int(), C.c_int()
    buf = (C.c_uint8 * len(png)).from_buffer_copy(png)
    assert lib.rrt_image_decode(buf, len(png), C.byref(px), C.byref(ww), C.byref(hh)) == 0
    got = np.ctypeslib.as_array(px, shape=(hh.value, ww.value, 4)).copy()
    lib.rrt_image_free(px)
    assert np.array_equal(got[..., :3], img) and (got[..., 3] == 255).all()
    assert np.array_equal(got, png_ref(path))
    assert lib.rrt_image_decode(buf, 4, C.byref(px), C.byref(ww), C.byref(hh)) == _capi.ERR_UNSUPPORTED   # not an image
