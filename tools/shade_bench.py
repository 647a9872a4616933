"""Cost of re-shading a traced frame (rrt_shade) against tracing it (rrt_render), on one B200.  Prints one JSON line.

    python tools/shade_bench.py [--launches 200] [--renders 5]

Per size (1920x1080 and 3840x2160; camera C0, a = 0.99, disk + dust, default effects, 4096x2048 procedural skies):
  * render_ms: median of --renders rrt_render launches that also write the four planes Renderer.shade needs
    (TRACE_PLANES), CUDA events around each launch;
  * shade_us: median of --launches rrt_shade launches into the uchar4 frame (no hdr_out), CUDA events around each launch.
    Consecutive launches alternate two skies and two exposures, so no launch repeats the one before it.  L2 is flushed
    (a 256 MiB write) before every timed launch, outside the events: the 1080p planes (102 MB) would otherwise stay in
    the 126 MB L2 from one launch to the next;
  * shade_back_to_back_us: the same launches enqueued back to back without the flush (a viewer re-shading a frame again
    and again), mean per launch;
  * bytes per launch from shapes: 16 B vel + 16 B emis + 16 B hdr + 1 B cls read and 4 B written per pixel (sky texels,
    read through the texture cache, not counted), and that over shade_us as GB/s and as a fraction of 7.7 TB/s (the
    HBM3e bandwidth of one B200 on NVIDIA's data sheet, for a 1000 W card);
  * shade_equals_render: the shade with the trace's own settings reproduces the traced frame byte for byte.
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
SIZES = [(1920, 1080), (3840, 2160)]
READ_BYTES_PER_PIXEL, WRITE_BYTES_PER_PIXEL = 16 + 16 + 16 + 1, 4
HBM_BYTES_PER_S = 7.7e12
L2_BYTES = 126e6


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
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--renders", type=int, default=5)
    a = ap.parse_args()
    if a.launches < 2 or a.renders < 1:
        ap.error("--launches must be at least 2 and --renders at least 1")
    torch.cuda.set_device(0)
    r = rrt.Renderer(0)
    skies = [r.create_sky(rrt.procedural_sky(4096, 2048, seed=s)) for s in (1234, 99)]
    exposures = [0.8, 1.3]
    prm = rrt.default_params(spin_a=0.99)   # disk + dust, the default (FMAD) contract
    cam, fx = rrt.camera_state_from(*CAM_C0), rrt.default_effects()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    out = {"tool": "tools/shade_bench.py", "gpu": gpu_info(), "camera": "C0", "spin_a": 0.99, "media": "disk+dust",
           "effects": "default (bloom, vignette, lens)", "sizes": []}
    for w, h in SIZES:
        traced = r.alloc_planes(w, h, rrt.TRACE_PLANES)
        frame = torch.empty((h, w, 4), dtype=torch.uint8, device="cuda")
        shaded = torch.empty_like(frame)
        r.render(prm, cam, fx, skies[0], 1.0, w, h, out=frame, planes=traced)   # warm-up (pool allocation)
        render_ms = []
        for _ in range(a.renders):
            flush.fill_(1)
            e0, e1 = ev(), ev()
            e0.record()
            r.render(prm, cam, fx, skies[0], 1.0, w, h, out=frame, planes=traced)
            e1.record()
            torch.cuda.synchronize()
            render_ms.append(e0.elapsed_time(e1))

        r.shade(prm, fx, skies[0], traced, w, h, out=shaded)
        torch.cuda.synchronize()
        equal = bool(torch.equal(shaded, frame))

        def launch(k):
            p = rrt.default_params(spin_a=0.99, exposure=exposures[(k // 2) % 2])   # (sky, exposure) cycles through 4 pairs
            r.shade(p, fx, skies[k % 2], traced, w, h, out=shaded)

        for k in range(8):
            launch(k)
        shade_us = []
        for k in range(a.launches):
            flush.fill_(1)
            e0, e1 = ev(), ev()
            e0.record()
            launch(k)
            e1.record()
            torch.cuda.synchronize()
            shade_us.append(e0.elapsed_time(e1) * 1e3)
        torch.cuda.synchronize()
        e0, e1 = ev(), ev()
        e0.record()
        for k in range(a.launches):
            launch(k)
        e1.record()
        torch.cuda.synchronize()
        b2b_us = e0.elapsed_time(e1) * 1e3 / a.launches

        px = w * h
        bytes_launch = px * (READ_BYTES_PER_PIXEL + WRITE_BYTES_PER_PIXEL)
        t = median(shade_us)
        out["sizes"].append({
            "width": w, "height": h,
            "render_ms": median(render_ms), "render_ms_all": render_ms,
            "shade_us": t, "shade_us_min": min(shade_us), "shade_us_max": max(shade_us), "shade_launches": a.launches,
            "shade_l2": "flushed (256 MiB write) before every timed launch",
            "shade_back_to_back_us": b2b_us, "shade_back_to_back_l2": "not flushed",
            "render_over_shade": median(render_ms) * 1e3 / t,
            "bytes_per_launch": bytes_launch, "plane_bytes": px * READ_BYTES_PER_PIXEL,
            "planes_fit_l2": px * READ_BYTES_PER_PIXEL < L2_BYTES,
            "achieved_GBps": bytes_launch / (t * 1e-6) / 1e9,
            "frac_of_hbm_7p7TBps": bytes_launch / (t * 1e-6) / HBM_BYTES_PER_S,
            "shade_equals_render": equal,
        })
        del traced, frame, shaded
    print(json.dumps(out), flush=True)
    for s in skies:
        s.close()
    r.close()


if __name__ == "__main__":
    main()
