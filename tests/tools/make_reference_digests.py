"""Writes tests/golden/reference_exact_digests.json (see tests/parity.py): sha256 digests of the REFERENCE's arrays that
tests/test_gpu_refcuda_planes.py and tests/test_gpu_fmad.py require our build to match bit for bit -- class, step count,
exit velocity and position of its instrumented CUDA build, its final_hdr and uchar4 frame on untouched pixels, the
zero pattern of its density probes and its disk temperature.  Needs the reference builds (oracle/_ref) and a B200; every
case first runs the test's own comparison against those builds, and nothing is written unless all of them pass:
    python tests/tools/make_reference_digests.py tests/golden/reference_exact_digests.json"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import relativisticraytracer_b200 as rrt  # noqa: E402
from oracle import RefCuda, RefCudaPlanes  # noqa: E402
import test_gpu_fmad as F  # noqa: E402
import test_gpu_refcuda_planes as P  # noqa: E402
from inputs import disk_points, phase_space  # noqa: E402
from parity import CAMERAS, digests  # noqa: E402

if not (RefCuda.available() and RefCudaPlanes.available()):
    sys.exit("oracle/_ref/libref_cuda.so and libref_cuda_planes.so are needed: the digests are the reference's")
gpu = rrt.Renderer(0)
refp, refcuda = RefCudaPlanes(), RefCuda()
pair = (refp, refcuda)
sky_small = rrt.procedural_sky(512, 256, seed=1234, stars=400)     # tests/conftest.py::sky_small
sky_big = rrt.procedural_sky(4096, 2048)                            # test_gpu_refcuda_planes.py::sky_big
out = {}


def reference_frames(sky_np, cam, spin, w, h, fx):
    cg = rrt.camera_state_from(*CAMERAS[cam])
    return refp.render(spin, cg, fx, sky_np, 1.0, w, h), refcuda.render(spin, cg, fx, sky_np, 1.0, w, h)[0]


for spin in (0.0, 0.99):
    for cam in ("C0", "C1", "C2", "C3"):
        P.test_fmad_planes_equal_reference_cuda_arithmetic(gpu, pair, sky_small, cam, spin)
        key, g = P.fmad_planes_case(gpu, sky_small, cam, spin)
        planes, plain = reference_frames(sky_small, cam, spin, 480, 270, rrt.effects_off())
        out[key] = digests(P.planes_exact(planes, plain, P.touched_of(g["cls"])))

        F.test_fmad_bytes_equal_reference_cuda_kernel(gpu, sky_small, cam, spin)
        key, g = F.fmad_bytes_case(gpu, sky_small, cam, spin, 320, 180)
        ref_rgba = refcuda.render(spin, rrt.camera_state_from(*CAMERAS[cam]), rrt.default_effects(), sky_small, 1.0, 320, 180)[0]
        out[key] = digests(F.fmad_bytes_exact(ref_rgba, (g["cls"] & rrt.CLSF_TOUCHED) == 0))

    P.test_fmad_media_probes_against_nvcc_compiled_reference_functions(gpu, pair, spin)
    key, _ = P.media_probes_case(gpu, spin)
    pts = disk_points(seed=31, n=1 << 15)
    r = np.linalg.norm(phase_space(seed=32, n=1 << 15)[0], axis=1).astype(np.float32)
    out[key] = digests(P.probes_exact(refp.probe("disk_density", spin, pts, None, 1.0), refp.probe("dust_density", spin, pts, None, 1.0),
                                      refp.probe("disk_temperature", spin, r)))

for w, h, cam in ((1920, 1080, "C0"), (1920, 1080, "C1"), (3840, 2160, "C0")):
    P.test_fmad_full_size_frames_equal_reference_cuda(gpu, pair, sky_big, w, h, cam)
    key, g = P.full_size_case(gpu, sky_big, w, h, cam)
    planes, plain = reference_frames(sky_big, cam, 0.99, w, h, rrt.effects_off())
    _, plain_d = reference_frames(sky_big, cam, 0.99, w, h, rrt.default_effects())
    out[key] = digests(P.full_size_exact(planes, plain, plain_d, P.touched_of(g["cls"]), P.touched_of(g["fxd_cls"])))

with open(sys.argv[1], "w") as f:
    json.dump(out, f, indent=1, sort_keys=True)
    f.write("\n")
print("wrote", sys.argv[1], len(out), "cases")
