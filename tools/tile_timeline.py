"""What does the tail of one render launch consist of?  Renders the bench frame once with the per-tile log switched on
(rrt_debug_tile_log) and prints: launch span, how the number of busy warp slots decays at the end, and the tiles that
finish last (position, duration, steps of their longest ray, SM).
Needs the profiling build: make -C relativisticraytracer_b200/csrc timeline, then
Usage: RRT_B200_LIB=$PWD/build/timeline/librrt_b200_timeline.so python tools/tile_timeline.py [--width W --height H --camera C0
       --flags 3 --band RANK NRANKS]   (GPU box)"""
import argparse
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import relativisticraytracer_b200 as rrt  # noqa: E402

CAMS = {"C0": ((0.0, 10.0, -60.0), 0.0, -10.0), "C1": ((15.0, 3.0, -30.0), -26.6, -5.1),
        "C2": ((35.0, 0.8, 10.0), -106.0, -1.2), "C3": ((4.2, 0.6, 4.2), -90.0, -5.7)}
ap = argparse.ArgumentParser()
ap.add_argument("--width", type=int, default=3840)
ap.add_argument("--height", type=int, default=2160)
ap.add_argument("--camera", default="C0")
ap.add_argument("--flags", type=int, default=3)
ap.add_argument("--band", type=int, nargs=2, default=None, help="rank nranks: trace one cyclic 8-row band set only")
a = ap.parse_args()
r = rrt.Renderer(0)
sky = r.create_sky(rrt.procedural_sky(4096, 2048))
prm = rrt.default_params(spin_a=0.99, flags=a.flags | rrt.FLAG_FMAD)
cam, fx = rrt.camera_state_from(*CAMS[a.camera]), rrt.default_effects()
band = rrt.Band(a.band[0], a.band[1], 8) if a.band else None
rows = r.band_rows(band, a.height)
ntiles = ((a.width + 7) // 8) * ((rows + 3) // 4)
log = torch.zeros((ntiles, 4), dtype=torch.int64, device="cuda")
kw = dict(band=band, layout=rrt.OUT_PACKED) if band else {}
for _ in range(2):
    r.render(prm, cam, fx, sky, 1.0, a.width, a.height, **kw)
torch.cuda.synchronize()
r.tile_log(log)
r.render(prm, cam, fx, sky, 1.0, a.width, a.height, **kw)
torch.cuda.synchronize()
r.tile_log(None)
L = log.cpu().numpy()
L = L[L[:, 1] > 0]
t0 = L[:, 0].min()
beg, end = (L[:, 0] - t0) / 1e6, (L[:, 1] - t0) / 1e6       # ms
dur = end - beg
span = end.max()
print(f"{len(L)} tiles, launch span {span:.2f} ms, sum of tile durations {dur.sum() / 1e3:.2f} s = {dur.sum() / span:.0f} busy warp slots on average")
print(f"tile duration ms: median {np.median(dur):.3f}  p99 {np.quantile(dur, .99):.3f}  max {dur.max():.3f}")
for frac in (0.5, 0.8, 0.9, 0.95, 0.98, 0.99, 1.0):
    t = span * frac
    busy = int(((beg <= t) & (end > t - 1e-9)).sum())
    print(f"  at {frac * 100:5.1f} % of the span ({t:7.2f} ms): {busy:5d} tiles in flight")
last_start = beg.max()
print(f"last tile handed out at {last_start:.2f} ms ({last_start / span * 100:.1f} % of the span): after that the launch only drains")
order = np.argsort(-end)[:12]
print("tiles finishing last:  end ms   start ms  duration ms   row  col   sm  longest ray (steps)")
for i in order:
    print(f"                     {end[i]:8.2f} {beg[i]:9.2f} {dur[i]:11.2f} {L[i, 2] >> 32:5d} {L[i, 2] & 0xffffffff:4d} {L[i, 3] >> 32:4d} {L[i, 3] & 0xffffffff:8d}")
slow = np.argsort(-dur)[:8]
print("longest tiles:         end ms   start ms  duration ms   row  col   sm  longest ray (steps)")
for i in slow:
    print(f"                     {end[i]:8.2f} {beg[i]:9.2f} {dur[i]:11.2f} {L[i, 2] >> 32:5d} {L[i, 2] & 0xffffffff:4d} {L[i, 3] >> 32:4d} {L[i, 3] & 0xffffffff:8d}")
