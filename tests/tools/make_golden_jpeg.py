"""Writes tests/golden/jpeg/: the JPEG files tests/test_image_decoder.py decodes (written by PIL from the test's
synthetic images) and stb_rgba_sha256.json, the sha256 of the RGBA8 bytes stb_image returns for each.  Needs
oracle/_ref/libref_stb.so (stb_image as the reference vendors it); nothing is written unless our decoder returns
stb_image's bytes on every file:
    python tests/tools/make_golden_jpeg.py"""
import hashlib
import json
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import relativisticraytracer_b200 as rrt  # noqa: E402
import test_image_decoder as T  # noqa: E402

if not os.path.exists(T.STB_LIB):
    sys.exit(f"{T.STB_LIB} is needed: the digests are stb_image's")
stb = T._stb_loader(T.STB_LIB)
tmp = tempfile.mkdtemp()
sums = {}
for case in T.JPEG_CASES + [T.JPEG_411]:
    path = os.path.join(tmp, T.jpeg_name(case))
    T.write_jpeg(case, path)
    want = stb(path)
    if want is None or not np.array_equal(rrt.decode_image(path), want):
        sys.exit(f"{T.jpeg_name(case)}: our decoder does not return stb_image's bytes; nothing written")
    sums[T.jpeg_name(case)] = hashlib.sha256(want.tobytes()).hexdigest()
os.makedirs(T.JPEG_GOLD, exist_ok=True)
for name in sums:
    os.replace(os.path.join(tmp, name), os.path.join(T.JPEG_GOLD, name))
with open(os.path.join(T.JPEG_GOLD, "stb_rgba_sha256.json"), "w") as f:
    json.dump(sums, f, indent=1, sort_keys=True)
    f.write("\n")
print("wrote", len(sums), "files to", T.JPEG_GOLD)
