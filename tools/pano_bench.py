"""Cost of a 360-degree panorama (rrt_render_pano) against pinhole frames of about the same ray count, on one B200.
Prints one JSON line (and one per case on stderr); with --out, appends it to that file.

    python tools/pano_bench.py [--renders 5] [--out profiles/pano_bench_b200.jsonl]

Per camera (C0, the reference default, and D0, a camera in the disk plane looking at the hole), a = 0.99, disk + dust, the
default (FMAD) contract, the default effects less lens distortion and vignette, a 4096x2048 procedural sky, these calls
are timed in alternation, --renders rounds, from CUDA events around the call with L2 flushed (a 256 MiB write) before it,
outside the events:
  * pinhole_3840x2160: rrt_render, 8.29 M rays;
  * pano_4096x2048: rrt_render_pano, 8.39 M rays;
  * pano_7680x3840: rrt_render_pano, 29.5 M rays;
  * render_ss_3840x2160_ss2: rrt_render_ss, 33.2 M rays;
  * pano_4096x2048_ss2: rrt_render_pano at ss = 2, 33.6 M rays.
Every timed frame is compared byte for byte with the first frame of its call (the renders are deterministic).  The GPU's
name, power limit and maximum SM clock are queried (nvidia-smi --query-gpu, read only) in the same run."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import relativisticraytracer_b200 as rrt  # noqa: E402

CAMS = {"C0": ((0.0, 10.0, -60.0), 0.0, -10.0),   # reference default camera, src/main.cpp:128-130
        "D0": ((0.0, 0.0, -40.0), 0.0, 0.0)}      # in the disk plane (y = 0), 40 units out, looking at the hole


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    try:
        line = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.TimeoutExpired) as e:
        line = f"unavailable: {e}"
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": {"query": q, "result": line}}


def median(xs):
    s = sorted(xs)
    return s[len(s) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--renders", type=int, default=5)
    ap.add_argument("--out", default="", help="append the JSON line to this file")
    a = ap.parse_args()
    if a.renders < 1:
        ap.error("--renders must be at least 1")
    torch.cuda.set_device(0)
    r = rrt.Renderer(0)
    sky = r.create_sky(rrt.procedural_sky(4096, 2048, seed=1234))
    prm = rrt.default_params(spin_a=0.99)
    fx = rrt.default_effects(use_lens=0, use_vignette=0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731

    out = {"tool": "tools/pano_bench.py", "gpu": gpu_info(), "spin_a": 0.99, "media": "disk+dust", "contract": "FMAD",
           "effects": "default less lens distortion and vignette (bloom on)", "sky": "procedural 4096x2048",
           "l2": "flushed (256 MiB write) before every timed call", "order": "the calls alternate, --renders rounds",
           "renders": a.renders, "cases": []}
    for name, spec in CAMS.items():
        cam = rrt.camera_state_from(*spec)
        frames = {}

        def call(key, w, h, fn):
            frames[key] = torch.empty((h, w, 4), dtype=torch.uint8, device="cuda")
            return key, (w * h, fn)

        calls = dict([
            call("pinhole_3840x2160", 3840, 2160, lambda f: r.render(prm, cam, fx, sky, 1.0, 3840, 2160, out=f)),
            call("pano_4096x2048", 4096, 2048, lambda f: r.render_pano(prm, cam, fx, sky, 1.0, 4096, 2048, out=f)),
            call("pano_7680x3840", 7680, 3840, lambda f: r.render_pano(prm, cam, fx, sky, 1.0, 7680, 3840, out=f)),
            call("render_ss_3840x2160_ss2", 3840, 2160, lambda f: r.render_ss(prm, cam, fx, sky, 1.0, 3840, 2160, 2, out=f)),
            call("pano_4096x2048_ss2", 4096, 2048, lambda f: r.render_pano(prm, cam, fx, sky, 1.0, 4096, 2048, ss=2, out=f)),
        ])
        rays = {"pinhole_3840x2160": 3840 * 2160, "pano_4096x2048": 4096 * 2048, "pano_7680x3840": 7680 * 3840,
                "render_ss_3840x2160_ss2": 4 * 3840 * 2160, "pano_4096x2048_ss2": 4 * 4096 * 2048}
        first = {}
        for k, (_, fn) in calls.items():   # warm-up: sample pools, scratch blocks; the reference bytes of each call
            fn(frames[k])
            torch.cuda.synchronize()
            first[k] = frames[k].clone()
        times = {k: [] for k in calls}
        same = {k: True for k in calls}
        for _ in range(a.renders):
            for k, (_, fn) in calls.items():
                frames[k].fill_(0)
                flush.fill_(1)
                e0, e1 = ev(), ev()
                e0.record()
                fn(frames[k])
                e1.record()
                torch.cuda.synchronize()
                times[k].append(e0.elapsed_time(e1))
                same[k] = same[k] and bool(torch.equal(frames[k], first[k]))
        case = {"camera": name, "pos_yaw_pitch": spec}
        for k in calls:
            case[k] = {"rays": rays[k], "ms": median(times[k]), "ms_all": times[k], "ns_per_ray": median(times[k]) * 1e6 / rays[k],
                       "frames_identical": same[k]}
        case["pano_4096x2048_over_pinhole_3840x2160"] = case["pano_4096x2048"]["ms"] / case["pinhole_3840x2160"]["ms"]
        case["pano_4096x2048_ss2_over_render_ss_3840x2160_ss2"] = (case["pano_4096x2048_ss2"]["ms"] /
                                                                   case["render_ss_3840x2160_ss2"]["ms"])
        out["cases"].append(case)
        print(json.dumps({k: (v["ms"] if isinstance(v, dict) and "ms" in v else v) for k, v in case.items()}), file=sys.stderr,
              flush=True)
        del frames, first
    line = json.dumps(out)
    print(line, flush=True)
    if a.out:
        with open(a.out, "a") as f:
            f.write(line + "\n")
    sky.close()
    r.close()


if __name__ == "__main__":
    main()
