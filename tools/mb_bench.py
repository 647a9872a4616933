"""Cost of a motion-blurred frame (rrt_render_mb, rrt_capture_render_mb) and of its resolve pass (rrt_resolve_time), on one
B200.  Prints one JSON line.

    python tools/mb_bench.py [--renders 3] [--launches 100] [--skip 3840x2160x8]

Per case (1920x1080 and 3840x2160, n = 4 and 8 sub-frames at shutter_times(1, 0.5, 24, n); camera C0 held still, a = 0.99,
disk + dust, default effects, a 4096x2048 procedural sky), every time from CUDA events around the call with L2 flushed (a
256 MiB write) before it, outside the events:
  * frame1_ms: median of --renders rrt_render frames at t = 1;
  * renders_ms: median of --renders sequences of the n sub-frame renders (rrt_render into the planes of a stack): what
    render_mb runs before its resolve;
  * render_mb_ms: median of --renders rrt_render_mb frames, against renders_ms and n x frame1_ms;
  * capture_renders_ms: median of --renders sequences of n rrt_capture_render calls at the sub-frame times (the capture is
    made once per size, outside the timed calls, with the context's pool sizing rule);
  * capture_mb_ms: median of --renders rrt_capture_render_mb frames, against capture_renders_ms and render_mb_ms;
  * resolve_time_us: median of --launches rrt_resolve_time launches of the stack into the uchar4 frame (no hdr_out);
    bytes from shapes, 16*n B read and 4 B written per pixel, and that over resolve_time_us as GB/s and as a fraction of
    7.7 TB/s (the HBM3e bandwidth of one B200 on NVIDIA's data sheet, for a 1000 W card).
Every timed frame is compared byte for byte with its reference composition: render_mb's and capture_mb's with the
resolve_time of the n renders' stack, and each resolve_time launch's with the first.  The GPU's name, power limit and
maximum SM clock are queried (nvidia-smi --query-gpu, read only) in the same run.  --skip drops cases (WxHxN,
comma-separated)."""
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
SIZES = [(1920, 1080), (3840, 2160)]
SAMPLES = [4, 8]
T, SHUTTER, FPS = 1.0, 0.5, 24.0
HBM_BYTES_PER_S = 7.7e12


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
    ap.add_argument("--renders", type=int, default=3)
    ap.add_argument("--launches", type=int, default=100)
    ap.add_argument("--skip", default="", help="cases to leave out, e.g. 3840x2160x8")
    a = ap.parse_args()
    if a.launches < 1 or a.renders < 1:
        ap.error("--launches and --renders must be at least 1")
    skip = {s.strip() for s in a.skip.split(",") if s.strip()}
    torch.cuda.set_device(0)
    r = rrt.Renderer(0)
    sky = r.create_sky(rrt.procedural_sky(4096, 2048, seed=1234))
    prm = rrt.default_params(spin_a=0.99)   # disk + dust, the default (FMAD) contract
    cam, fx = rrt.camera_state_from(*CAM_C0), rrt.default_effects()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    mismatches = []

    def timed(fn, n, check=None):
        """CUDA-event times of n calls of fn, L2 flushed before each, in ms; check() after each, outside the events."""
        ts = []
        for _ in range(n):
            flush.fill_(1)
            e0, e1 = ev(), ev()
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
            if check is not None:
                check()
        return ts

    out = {"tool": "tools/mb_bench.py", "gpu": gpu_info(), "camera": "C0 (still)", "spin_a": 0.99, "media": "disk+dust",
           "effects": "default (bloom, vignette, lens)", "times": f"shutter_times({T}, {SHUTTER}, {FPS}, n)",
           "l2": "flushed (256 MiB write) before every timed call", "cases": []}
    for w, h in SIZES:
        frame = torch.empty((h, w, 4), dtype=torch.uint8, device="cuda")
        r.render(prm, cam, fx, sky, T, w, h, out=frame)   # warm-up (sample pool)
        frame1 = timed(lambda: r.render(prm, cam, fx, sky, T, w, h, out=frame), a.renders)
        cap = r.capture(prm, cam, fx, sky, w, h)
        info = cap.info()
        for n in SAMPLES:
            tag = f"{w}x{h}x{n}"
            if tag in skip:
                continue
            times = rrt.shutter_times(T, SHUTTER, FPS, n)
            stack = torch.empty((n, h, w, 4), dtype=torch.float32, device="cuda")

            def renders():   # the sub-frames render_mb traces (its stack comes from the context's pool instead)
                for i in range(n):
                    r.render(prm, cam, fx, sky, times[i], w, h, planes={"hdr": stack[i]})

            def capture_renders():
                for i in range(n):
                    cap.render(prm, fx, sky, times[i], hdr_out=stack[i])

            resolve = lambda: r.resolve_time(prm, fx, stack, w, h, out=frame)  # noqa: E731
            render_mb = lambda: r.render_mb(prm, cam, fx, sky, times, w, h, out=frame)  # noqa: E731
            capture_mb = lambda: cap.render_mb(prm, fx, sky, times, out=frame)  # noqa: E731

            def same(name):
                def check():
                    if not torch.equal(frame, want):
                        mismatches.append(f"{tag} {name}")
                return check

            renders()
            renders_ms = timed(renders, a.renders)
            resolve()
            torch.cuda.synchronize()
            want = frame.clone()   # the reference composition: resolve_time of the n renders' stack
            resolve_ms = timed(resolve, a.launches, same("resolve_time"))
            render_mb()   # warm-up (stack from the context's pool)
            render_mb_ms = timed(render_mb, a.renders, same("render_mb"))
            capture_renders()
            capture_renders_ms = timed(capture_renders, a.renders)
            resolve()
            torch.cuda.synchronize()
            capture_equal = bool(torch.equal(frame, want))   # the capture's sub-frames are the renders' planes
            capture_mb()
            capture_mb_ms = timed(capture_mb, a.renders, same("capture_mb"))
            t_us = median(resolve_ms) * 1e3
            nbytes = w * h * (16 * n + 4)
            out["cases"].append({
                "width": w, "height": h, "n": n, "times": times,
                "frame1_ms": median(frame1), "renders_ms": median(renders_ms), "renders_ms_all": renders_ms,
                "render_mb_ms": median(render_mb_ms), "render_mb_ms_all": render_mb_ms,
                "render_mb_over_n_frame1": median(render_mb_ms) / (n * median(frame1)),
                "render_mb_minus_renders_ms": median(render_mb_ms) - median(renders_ms),
                "capture_renders_ms": median(capture_renders_ms), "capture_mb_ms": median(capture_mb_ms),
                "capture_mb_ms_all": capture_mb_ms, "capture_mb_minus_capture_renders_ms": median(capture_mb_ms) - median(capture_renders_ms),
                "render_mb_over_capture_mb": median(render_mb_ms) / median(capture_mb_ms),
                "resolve_time_us": t_us, "resolve_time_us_min": min(resolve_ms) * 1e3, "resolve_time_us_max": max(resolve_ms) * 1e3,
                "resolve_time_launches": a.launches, "resolve_time_bytes": nbytes,
                "resolve_time_GBps": nbytes / (t_us * 1e-6) / 1e9,
                "resolve_time_frac_of_hbm_7p7TBps": nbytes / (t_us * 1e-6) / HBM_BYTES_PER_S,
                "resolve_share_of_render_mb": t_us * 1e-3 / median(render_mb_ms),
                "resolve_share_of_capture_mb": t_us * 1e-3 / median(capture_mb_ms),
                "stack_bytes": 16 * n * w * h, "capture_bytes": info["bytes"], "capture_tiles_left": info["tiles_left"],
                "capture_renders_equal_renders": capture_equal,
            })
            print(json.dumps(out["cases"][-1]), file=sys.stderr, flush=True)
            del stack
        cap.close()
        del frame
    out["timed_frames_equal_reference"] = not mismatches and all(c["capture_renders_equal_renders"] for c in out["cases"])
    out["mismatches"] = mismatches
    print(json.dumps(out), flush=True)
    sky.close()
    r.close()


if __name__ == "__main__":
    main()
