"""Cost of re-timing a traced frame (rrt_capture_create / rrt_capture_render) against a new trace (rrt_render), on one
B200.  Prints one JSON line.

    python tools/retime_bench.py [--renders 5] [--retimes 20] [--c3-max-gib 64] [--skip 3840x2160xC3]

Per case (cameras C0 and C3 at 1920x1080 and 3840x2160; a = 0.99, disk + dust, default effects, a 4096x2048 procedural
sky), every time from CUDA events around the call with L2 flushed (a 256 MiB write) before it, outside the events:
  * render_ms: median of --renders rrt_render frames at t = 1;
  * capture_ms: one rrt_capture_create (host clock from a synchronised device to its return; it synchronises);
  * retime_ms: median of --retimes rrt_capture_render frames at times 0, 0.5, 1, ... (each a new time);
  * the capture's rrt_capture_info (bytes held, samples, tiles left to the fused sweep);
  * retime_equals_render: the capture's frame at t = 1 is rrt_render's byte for byte.
The capture's pool follows the context's sizing rule (max_bytes = 0, at most 16 GiB); C3 is measured again with a pool of
--c3-max-gib GiB (0: skip), which holds the whole media-heavy frame.  --skip drops cases (WxHxCAM[xGiB], comma-separated).
The GPU's name, power limit and maximum SM clock are queried (nvidia-smi --query-gpu, read only) in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import relativisticraytracer_b200 as rrt  # noqa: E402

CAMS = {"C0": ((0.0, 10.0, -60.0), 0.0, -10.0), "C3": ((4.2, 0.6, 4.2), -90.0, -5.7)}   # as tests/parity.py CAMERAS
SIZES = [(1920, 1080), (3840, 2160)]


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
    ap.add_argument("--retimes", type=int, default=20)
    ap.add_argument("--c3-max-gib", type=int, default=64)
    ap.add_argument("--skip", default="", help="cases to leave out, e.g. 3840x2160xC3x64")
    a = ap.parse_args()
    if a.renders < 1 or a.retimes < 1:
        ap.error("--renders and --retimes must be at least 1")
    skip = {s.strip() for s in a.skip.split(",") if s.strip()}
    torch.cuda.set_device(0)
    r = rrt.Renderer(0)
    sky = r.create_sky(rrt.procedural_sky(4096, 2048, seed=1234))
    prm = rrt.default_params(spin_a=0.99)   # disk + dust, the default (FMAD) contract
    fx = rrt.default_effects()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731

    def timed(fn, args):
        """CUDA-event times of fn(x) for x in args, L2 flushed before each, in ms."""
        ts = []
        for x in args:
            flush.fill_(1)
            e0, e1 = ev(), ev()
            e0.record()
            fn(x)
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return ts

    out = {"tool": "tools/retime_bench.py", "gpu": gpu_info(), "spin_a": 0.99, "media": "disk+dust",
           "effects": "default (bloom, vignette, lens)", "l2": "flushed (256 MiB write) before every timed call", "cases": []}
    cases = [(w, h, cam, 0) for w, h in SIZES for cam in CAMS]
    if a.c3_max_gib:
        cases += [(w, h, "C3", a.c3_max_gib) for w, h in SIZES]
    for w, h, cam_name, gib in cases:
        tag = f"{w}x{h}x{cam_name}" + (f"x{gib}" if gib else "")
        if tag in skip:
            continue
        cam = rrt.camera_state_from(*CAMS[cam_name])
        frame = torch.empty((h, w, 4), dtype=torch.uint8, device="cuda")
        r.render(prm, cam, fx, sky, 1.0, w, h, out=frame)   # warm-up (sample pool)
        render_ms = timed(lambda _: r.render(prm, cam, fx, sky, 1.0, w, h, out=frame), range(a.renders))
        want = frame.clone()
        torch.cuda.synchronize()
        flush.fill_(1)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        cap = r.capture(prm, cam, fx, sky, w, h, max_bytes=gib << 30)
        capture_ms = (time.perf_counter() - t0) * 1e3
        info = cap.info()
        cap.render(prm, fx, sky, 3.0, out=frame)   # warm-up (launch configuration of the new kernels)
        retime_ms = timed(lambda t: cap.render(prm, fx, sky, t, out=frame), [0.5 * k for k in range(a.retimes)])
        cap.render(prm, fx, sky, 1.0, out=frame)
        equal = bool(torch.equal(frame, want))
        cap.close()
        res = {"width": w, "height": h, "camera": cam_name, "max_bytes": gib << 30,
               "render_ms": median(render_ms), "render_ms_all": render_ms, "capture_ms": capture_ms,
               "retime_ms": median(retime_ms), "retime_ms_min": min(retime_ms), "retime_ms_max": max(retime_ms),
               "retimes": a.retimes, "render_over_retime": median(render_ms) / median(retime_ms),
               "capture_bytes": info["bytes"], "capture_gb": info["bytes"] / 1e9, "info": info,
               "retime_equals_render": equal}
        out["cases"].append(res)
        print(json.dumps(res), file=sys.stderr, flush=True)
        del frame, want
    print(json.dumps(out), flush=True)
    sky.close()
    r.close()


if __name__ == "__main__":
    main()
