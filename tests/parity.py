"""Parity metrics of SURVEY.md 8d, shared by the CPU and GPU tests.

* class: exact integer equality per pixel
* escape direction: atan2(|d_ref x d_new|, d_ref . d_new) in float64 on the normalised exit velocity over
  pixels whose class agrees and is not captured; tolerance 1e-5 rad (north_star)
* linear RGB: |dc| / max(|c_ref|, 1e-3) per channel on final_hdr with effects off; tolerance 1e-3 (north_star)
"""
import hashlib
import json
import os

import numpy as np

DIR_TOL_RAD = 1e-5
RGB_TOL_REL = 1e-3

# cameras of SURVEY.md 8d: (pos, yaw_deg, pitch_deg)
CAMERAS = {
    "C0": ((0.0, 10.0, -60.0), 0.0, -10.0),      # reference default, src/main.cpp:128-130
    "C1": ((15.0, 3.0, -30.0), -26.6, -5.1),     # Gargantua key 2, camera_paths.cpp:38
    "C2": ((35.0, 0.8, 10.0), -106.0, -1.2),     # Gargantua key 3, camera_paths.cpp:39
    "C3": ((4.2, 0.6, 4.2), -90.0, -5.7),        # Skimmer key 3, camera_paths.cpp:66
}


def class_flips(cls_ref, cls_new):
    return int(np.sum((cls_ref & 3) != (cls_new & 3)))


def direction_error(dir_ref, dir_new, cls_ref, cls_new):
    """radians, float64, over non-captured pixels whose class agrees; returns array (possibly empty)."""
    ok = ((cls_ref & 3) == (cls_new & 3)) & ((cls_ref & 3) != 0)
    a = dir_ref[ok][:, :3].astype(np.float64)
    b = dir_new[ok][:, :3].astype(np.float64)
    cr = np.linalg.norm(np.cross(a, b), axis=1)
    dt = np.sum(a * b, axis=1)
    return np.arctan2(cr, dt)


def rgb_rel_error(hdr_ref, hdr_new):
    a = hdr_ref[..., :3].astype(np.float64)
    b = hdr_new[..., :3].astype(np.float64)
    return np.abs(b - a) / np.maximum(np.abs(a), 1e-3)


def census(ref, new):
    """Summary dict comparing two frames that carry cls/dir/hdr planes (Frame or dict-like)."""
    def g(o, k):
        return o[k] if isinstance(o, dict) else getattr(o, k)
    cr, cn = g(ref, "cls"), g(new, "cls")
    ang = direction_error(g(ref, "dir"), g(new, "dir"), cr, cn)
    rel = rgb_rel_error(g(ref, "hdr"), g(new, "hdr"))
    pix = rel.max(axis=-1)
    return {
        "pixels": int(cr.size),
        "class_flips": class_flips(cr, cn),
        "flag_diffs": int(np.sum(cr != cn)),
        "dir_max_rad": float(ang.max()) if ang.size else 0.0,
        "dir_frac_over_tol": float(np.mean(ang > DIR_TOL_RAD)) if ang.size else 0.0,
        "rgb_max_rel": float(pix.max()),
        "rgb_p999_rel": float(np.quantile(pix, 0.999)),
        "rgb_frac_over_tol": float(np.mean(pix > RGB_TOL_REL)),
    }


# Where the reference's own CUDA builds (oracle/_ref) are absent, the GPU tests that compare with them check the exact
# part of that comparison: the arrays those tests require to be bit-identical to the reference's, against sha256 digests
# of the reference's arrays committed in tests/golden/reference_exact_digests.json (tests/tools/make_reference_digests.py
# writes them from the reference builds, after running the tests' own checks against those builds).  The parts compared
# within a tolerance (touched pixels, probe quantiles) are checked only where the reference builds are present.
REFERENCE_DIGESTS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_exact_digests.json")


def digests(arrays):
    """sha256 of the bytes (C order) of each array of a dict."""
    return {k: hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest() for k, a in arrays.items()}


def assert_reference_digests(key, parts):
    with open(REFERENCE_DIGESTS) as f:
        want = json.load(f)[key]
    got = digests(parts)
    assert sorted(got) == sorted(want), key
    assert got == want, f"{key}: {sorted(k for k in want if got[k] != want[k])} differ from the reference's"
