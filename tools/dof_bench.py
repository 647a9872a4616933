"""Cost of a depth-of-field frame (rrt_render_dof) against the supersampled frame it is built on (rrt_render_ss), on one B200.
Prints one JSON line.

    python tools/dof_bench.py [--renders 5] [--skip 3840x2160x2]

Per case (1920x1080 and 3840x2160 at ss = 2; camera C0, a = 0.99, disk + dust, default effects, a 4096x2048 procedural
sky), three calls are timed in alternation, --renders times each, from CUDA events around the call with L2 flushed (a
256 MiB write) before it, outside the events:
  * render_ss_ms: rrt_render_ss(C0);
  * dof_pinhole_ms: rrt_render_dof with lens_cameras(C0, 0, 60, ss) -- ss*ss copies of C0, the same rays as render_ss;
  * dof_lens_ms: rrt_render_dof with lens_cameras(C0, 0.5, 60, ss) -- a thin lens of radius 0.5 focused 60 units out.
Every timed frame is compared byte for byte with its composition, built once outside the timing: rrt_resolve of the
ss*w x ss*h hdr plane put together from the ss*ss rrt_render calls with the table's cameras (one call for the pinhole).
The GPU's name, power limit and maximum SM clock are queried (nvidia-smi --query-gpu, read only) in the same run."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import relativisticraytracer_b200 as rrt  # noqa: E402

CAM_C0 = ((0.0, 10.0, -60.0), 0.0, -10.0)   # reference default camera, src/main.cpp:128-130
CASES = [(1920, 1080, 2), (3840, 2160, 2)]
APERTURE, FOCUS = 0.5, 60.0


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


def composed(r, prm, cams, fx, sky, w, h, ss):
    """The frame render_dof(cams) must write: rrt_resolve of the hdr plane taken, sub-sample (i, j) by sub-sample, from the
    ss*w x ss*h render with cams[j*ss + i] (one render when every camera is the same)."""
    hi = torch.empty((ss * h, ss * w, 4), dtype=torch.float32, device="cuda")
    same = all(bytes(c) == bytes(cams[0]) for c in cams)
    if same:
        r.render(prm, cams[0], fx, sky, 1.0, ss * w, ss * h, planes={"hdr": hi})
    else:
        plane = torch.empty_like(hi)
        for k, cam in enumerate(cams):
            i, j = k % ss, k // ss
            r.render(prm, cam, fx, sky, 1.0, ss * w, ss * h, planes={"hdr": plane})
            hi[j::ss, i::ss] = plane[j::ss, i::ss]
    out = r.resolve(prm, fx, hi, ss, w, h)
    torch.cuda.synchronize()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--renders", type=int, default=5)
    ap.add_argument("--skip", default="", help="cases to leave out, e.g. 3840x2160x2")
    a = ap.parse_args()
    if a.renders < 1:
        ap.error("--renders must be at least 1")
    skip = {s.strip() for s in a.skip.split(",") if s.strip()}
    torch.cuda.set_device(0)
    r = rrt.Renderer(0)
    sky = r.create_sky(rrt.procedural_sky(4096, 2048, seed=1234))
    prm = rrt.default_params(spin_a=0.99)   # disk + dust, the default (FMAD) contract
    cam, fx = rrt.camera_state_from(*CAM_C0), rrt.default_effects()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731

    out = {"tool": "tools/dof_bench.py", "gpu": gpu_info(), "camera": "C0", "spin_a": 0.99, "media": "disk+dust",
           "effects": "default (bloom, vignette, lens)", "lens": {"aperture": APERTURE, "focus": FOCUS},
           "l2": "flushed (256 MiB write) before every timed call", "order": "the three calls alternate, --renders rounds",
           "cases": []}
    for w, h, ss in CASES:
        if f"{w}x{h}x{ss}" in skip:
            continue
        pinhole = rrt.lens_cameras(cam, 0.0, FOCUS, ss)
        lens = rrt.lens_cameras(cam, APERTURE, FOCUS, ss)
        want_pin = composed(r, prm, pinhole, fx, sky, w, h, ss)
        want_lens = composed(r, prm, lens, fx, sky, w, h, ss)
        frame = torch.empty((h, w, 4), dtype=torch.uint8, device="cuda")
        calls = {
            "render_ss": (lambda: r.render_ss(prm, cam, fx, sky, 1.0, w, h, ss, out=frame), want_pin),
            "dof_pinhole": (lambda: r.render_dof(prm, pinhole, fx, sky, 1.0, w, h, ss, out=frame), want_pin),
            "dof_lens": (lambda: r.render_dof(prm, lens, fx, sky, 1.0, w, h, ss, out=frame), want_lens),
        }
        times = {k: [] for k in calls}
        equal = {k: True for k in calls}
        for fn, _ in calls.values():   # warm-up: sample pool, scratch block
            fn()
        torch.cuda.synchronize()
        for _ in range(a.renders):
            for k, (fn, want) in calls.items():
                frame.fill_(0)
                flush.fill_(1)
                e0, e1 = ev(), ev()
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                times[k].append(e0.elapsed_time(e1))
                equal[k] = equal[k] and bool(torch.equal(frame, want))
        case = {"width": w, "height": h, "ss": ss, "rays": ss * ss * w * h}
        for k in calls:
            case[f"{k}_ms"] = median(times[k])
            case[f"{k}_ms_all"] = times[k]
            case[f"{k}_equals_composition"] = equal[k]
        case["dof_pinhole_over_render_ss"] = case["dof_pinhole_ms"] / case["render_ss_ms"]
        case["dof_lens_over_render_ss"] = case["dof_lens_ms"] / case["render_ss_ms"]
        out["cases"].append(case)
        print(json.dumps(case), file=sys.stderr, flush=True)
        del frame, want_pin, want_lens
    print(json.dumps(out), flush=True)
    sky.close()
    r.close()


if __name__ == "__main__":
    main()
