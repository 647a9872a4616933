"""render_kernel_p (csrc/rrt_packed.cuh: two rays per thread in packed f32x2 registers, FMAD contract, no medium) against
render_kernel.  Each half of a packed instruction is rounded like the scalar instruction it replaces, so frames, parity
planes and counters must be bit-identical whichever kernel traced them -- for every camera, for ragged sizes (odd widths
leave a thread with one ray), bands, and the step budget's edge.  RRT_KERNEL=auto|scalar is read when a context is
created; auto (the default) uses the packed kernel for launches without a medium, scalar always uses render_kernel.
Launches with a medium go through the split pipeline, which tests/test_gpu_split.py checks against render_kernel."""
import os

import numpy as np
import pytest

from parity import CAMERAS

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pair(built):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    import relativisticraytracer_b200 as rrt
    old = os.environ.get("RRT_KERNEL")
    made = {}
    try:
        os.environ["RRT_KERNEL"] = "scalar"
        made["scalar"] = rrt.Renderer(0)
        os.environ.pop("RRT_KERNEL")
        made["packed"] = rrt.Renderer(0)   # auto: the packed kernel for these launches
    finally:
        if old is None:
            os.environ.pop("RRT_KERNEL", None)
        else:
            os.environ["RRT_KERNEL"] = old
    yield made["scalar"], made["packed"]
    for r in made.values():
        r.close()


def _frame(r, sky_np, cam, spin, flags, w, h, fx="default", band=None, **over):
    import relativisticraytracer_b200 as rrt
    import torch
    sky = r.create_sky(sky_np)
    planes = r.alloc_planes(w, h) if band is None else None
    r.read_counters(reset=True)
    kw = dict(band=band, layout=rrt.OUT_PACKED) if band is not None else {}
    out = r.render(rrt.default_params(spin_a=spin, flags=flags, **over), rrt.camera_state_from(*CAMERAS[cam]),
                   rrt.default_effects() if fx == "default" else rrt.effects_off(), sky, 1.0, w, h, planes=planes, **kw)
    torch.cuda.synchronize()
    res = {k: v.cpu().numpy() for k, v in (planes or {}).items()}
    res["rgba"] = out.cpu().numpy()
    res["counters"] = r.read_counters()
    sky.close()
    return res


def _same(a, b, tag):
    assert a["counters"] == b["counters"], tag
    for k in a:
        if k != "counters":
            assert np.array_equal(a[k], b[k], equal_nan=True), f"{tag}: {k}"


@pytest.mark.parametrize("cam", ["C0", "C1", "C2", "C3"])
@pytest.mark.parametrize("spin,flags", [(0.99, 4), (0.0, 4)])
def test_packed_equals_scalar(pair, sky_small, cam, spin, flags):
    scalar, packed = pair
    w, h = 203, 117      # odd width: the last thread of a row owns a single ray
    _same(_frame(scalar, sky_small, cam, spin, flags, w, h), _frame(packed, sky_small, cam, spin, flags, w, h), f"{cam} a={spin} flags={flags}")


def test_packed_equals_scalar_bands_budget_and_one_pixel(pair, sky_small):
    import relativisticraytracer_b200 as rrt
    scalar, packed = pair
    for band in (rrt.Band(0, 3, 8), rrt.Band(2, 3, 8), rrt.Band(1, 2, 1)):
        _same(_frame(scalar, sky_small, "C1", 0.99, 4, 160, 90, band=band), _frame(packed, sky_small, "C1", 0.99, 4, 160, 90, band=band), "band")
    for steps in (0, 1, 7, 8, 9, 17, 333):    # around the burst length
        _same(_frame(scalar, sky_small, "C0", 0.99, 4, 64, 36, max_steps=steps), _frame(packed, sky_small, "C0", 0.99, 4, 64, 36, max_steps=steps), f"max_steps={steps}")
    _same(_frame(scalar, sky_small, "C0", 0.99, 4, 1, 1), _frame(packed, sky_small, "C0", 0.99, 4, 1, 1), "1x1")
    _same(_frame(scalar, sky_small, "C2", 0.99, 4, 2, 5, fx="off"), _frame(packed, sky_small, "C2", 0.99, 4, 2, 5, fx="off"), "2x5")


def test_auto_picks_packed_only_without_media(pair, sky_small, gpu):
    """The default context (RRT_KERNEL unset = auto) must give the same bytes either way; this pins the policy's outputs."""
    scalar, _ = pair
    for flags in (4, 7):
        _same(_frame(gpu, sky_small, "C1", 0.99, flags, 120, 67), _frame(scalar, sky_small, "C1", 0.99, flags, 120, 67), f"auto flags={flags}")
