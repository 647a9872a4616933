"""Cost of a supersampled frame (rrt_render_ss) and of its resolve pass (rrt_resolve), on one B200.  Prints one JSON line.

    python tools/ss_bench.py [--renders 3] [--launches 100] [--skip 3840x2160x4]

Per case (1920x1080 and 3840x2160, ss = 1, 2, 3, 4; camera C0, a = 0.99, disk + dust, default effects, a 4096x2048
procedural sky), every time from CUDA events around the call with L2 flushed (a 256 MiB write) before it, outside the
events:
  * frame1_ms: median of --renders 1-sample rrt_render frames at w x h;
  * trace_ms: median of --renders rrt_render calls at ss*w x ss*h with d_out = NULL and only the hdr plane: the trace
    render_ss runs;
  * resolve_us: median of --launches rrt_resolve launches of that plane into the uchar4 frame (no hdr_out);
  * resolve bytes from shapes: 16*ss*ss B read and 4 B written per output pixel, and that over resolve_us as GB/s and
    as a fraction of 7.7 TB/s (the HBM3e bandwidth of one B200 on NVIDIA's data sheet, for a 1000 W card);
  * render_ss_ms: median of --renders rrt_render_ss frames, against ss*ss x frame1_ms, and the share of it the resolve
    takes;
  * render_ss_equals_resolve: render_ss's frame is the resolve of the traced plane, byte for byte.
--skip drops cases (WxHxSS, comma-separated).  The GPU's name, power limit and maximum SM clock are queried
(nvidia-smi --query-gpu, read only) in the same run."""
import argparse
import ctypes as C
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
FACTORS = [1, 2, 3, 4]
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
    ap.add_argument("--skip", default="", help="cases to leave out, e.g. 3840x2160x4")
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

    def timed(fn, n):
        """CUDA-event times of n calls of fn, L2 flushed before each, in ms."""
        ts = []
        for _ in range(n):
            flush.fill_(1)
            e0, e1 = ev(), ev()
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return ts

    out = {"tool": "tools/ss_bench.py", "gpu": gpu_info(), "camera": "C0", "spin_a": 0.99, "media": "disk+dust",
           "effects": "default (bloom, vignette, lens)", "l2": "flushed (256 MiB write) before every timed call", "cases": []}
    for w, h in SIZES:
        frame = torch.empty((h, w, 4), dtype=torch.uint8, device="cuda")
        r.render(prm, cam, fx, sky, 1.0, w, h, out=frame)   # warm-up (sample pool)
        frame1 = timed(lambda: r.render(prm, cam, fx, sky, 1.0, w, h, out=frame), a.renders)
        for ss in FACTORS:
            if f"{w}x{h}x{ss}" in skip:
                continue
            hi = torch.empty((ss * h, ss * w, 4), dtype=torch.float32, device="cuda")
            pl = rrt.Planes(hdr=hi.data_ptr())

            def trace():   # what render_ss traces: the hdr plane only, no uchar4 frame (d_out = NULL)
                r._check(r._lib.rrt_render(r._ctx, C.byref(prm), C.byref(cam), C.byref(fx), C.c_uint64(sky.texture), 1.0,
                                           ss * w, ss * h, None, None, rrt.OUT_FRAME, C.byref(pl),
                                           C.c_void_p(torch.cuda.current_stream().cuda_stream)))
            resolve = lambda: r.resolve(prm, fx, hi, ss, w, h, out=frame)  # noqa: E731
            render_ss = lambda: r.render_ss(prm, cam, fx, sky, 1.0, w, h, ss, out=frame)  # noqa: E731
            trace()
            trace_ms = timed(trace, a.renders)
            resolve()
            resolve_ms = timed(resolve, a.launches)
            resolved = frame.clone()
            render_ss()   # warm-up (scratch plane from the context's pool)
            render_ss_ms = timed(render_ss, a.renders)
            equal = bool(torch.equal(frame, resolved))
            t_us = median(resolve_ms) * 1e3
            nbytes = w * h * (16 * ss * ss + 4)
            out["cases"].append({
                "width": w, "height": h, "ss": ss, "rays": ss * ss * w * h,
                "frame1_ms": median(frame1), "trace_ms": median(trace_ms), "trace_ms_all": trace_ms,
                "resolve_us": t_us, "resolve_us_min": min(resolve_ms) * 1e3, "resolve_us_max": max(resolve_ms) * 1e3,
                "resolve_launches": a.launches, "resolve_bytes": nbytes,
                "resolve_GBps": nbytes / (t_us * 1e-6) / 1e9, "resolve_frac_of_hbm_7p7TBps": nbytes / (t_us * 1e-6) / HBM_BYTES_PER_S,
                "render_ss_ms": median(render_ss_ms), "render_ss_ms_all": render_ss_ms,
                "render_ss_over_ss2_frame1": median(render_ss_ms) / (ss * ss * median(frame1)),
                "resolve_share_of_render_ss": t_us * 1e-3 / median(render_ss_ms),
                "render_ss_equals_resolve": equal,
            })
            print(json.dumps(out["cases"][-1]), file=sys.stderr, flush=True)
            del hi
        del frame
    print(json.dumps(out), flush=True)
    sky.close()
    r.close()


if __name__ == "__main__":
    main()
