#!/usr/bin/env python
"""bench.py -- RK4 geodesic steps/s and frames/s of the render path on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[3], the one the headline metric is quoted on): ONE 3840x2160 frame, Kerr-like
spin a=0.99, accretion disk + dust clouds with Doppler/redshift transfer, reference default camera
(0,10,-60) yaw 0 pitch -10 (src/main.cpp:128-130), time 1.0, reference default CameraEffects, procedural
4096x2048 RGBA8 skybox.  A "step" is one such frame.  At N>1 the frame is cut into cyclic 8-row bands, one
set per rank (no communication while tracing), gathered to rank 0 over NCCL/NVLink and assembled there:
total work is fixed, so scaling is "strong".

The one JSON line printed by rank 0 follows the driver contract; see DESIGN.md "Measurement" for how
`roofline`, `cpu_baseline`, `e2e` and `gpu_launches` are defined for this path.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W4K, H4K = 3840, 2160
CAM_POS, CAM_YAW, CAM_PITCH = (0.0, 10.0, -60.0), 0.0, -10.0
SPIN = 0.99
TIME = 1.0
BAND_GROUP = 8
FLOP_PER_STEP = 218.0          # SURVEY.md 8d: algorithmic FLOP of one RK4 geodesic step, a != 0
FP32_THEORETICAL_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12   # 74.4, at clocks.max.sm
CPU_SAMPLE = (1280, 720)       # bounded CPU sample of the same camera / parameters (~5 s on 16 host cores)
WORKLOAD = "3840x2160 Kerr a=0.99 volumetric (disk+dust) frame, camera C0, cyclic 8-row bands over N GPUs"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--width", type=int, default=W4K)
    ap.add_argument("--height", type=int, default=H4K)
    ap.add_argument("--flags", type=int, default=3, help="experiment only: media flags (3 = disk+dust = the headline workload)")
    ap.add_argument("--camera", default="C0", help="experiment only: C0 (headline) .. C3")
    ap.add_argument("--strict", action="store_true",
                    help="experiment only: clear RRT_FLAG_FMAD (unfused arithmetic, the twin of the reference headers on a host) "
                         "instead of the default contract, the arithmetic of the reference's own CUDA build")
    ap.add_argument("--depth", type=int, default=0,
                    help="frames in flight in the timed sequence (1..4); 0 (default) = pick the schedule at start-up")
    ap.add_argument("--share", type=int, default=-1,
                    help="with --depth: rrt_set_frames_in_flight value, each launch gets 1/share of the CTA slots (default 1)")
    ap.add_argument("--workload", default="frame", choices=["frame", "path"],
                    help="frame (default, the headline: one 4K frame cut into row bands) or path (BASELINE config 5: "
                         "the 300-frame 'Gargantua Fly-By' at 1080p, frame k on GPU k mod N, sustained frames/s)")
    ap.add_argument("--path-frames", type=int, default=300)
    ap.add_argument("--exchange", default="auto", choices=["auto", "peer", "nccl"],
                    help="N > 1: how the bands reach rank 0 -- peer: every rank's kernel stores straight into rank 0's frame over "
                         "NVLink (CUDA IPC mapping) + a 4-byte all-reduce; nccl: packed bands + NCCL gather + assemble kernel; "
                         "auto (default): peer when the mapping can be set up, else nccl")
    ap.add_argument("--no-path", action="store_true", help="N > 1: skip the frame-parallel camera-path sub-record")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-cuda", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the frame of the last timed step to DIR/frame.npy (see dump_frame), "
                         "so that two builds can be compared output for output on the same inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 0:
        ap.error("--warmup must not be negative")
    if args.dump_outputs and (args.impl, args.workload) != ("ours", "frame"):
        ap.error("--dump-outputs needs --impl ours --workload frame")
    return args


DUMP_MAX_PIXELS = 1 << 21      # 2 Mi pixels x 4 channels x float32 = 32 MiB


def dump_frame(directory: str, frame) -> None:
    """DIR/frame.npy: the RGBA8 bytes of `frame` ([h, w, 4] uint8) as float32 -- the whole frame, shape [h, w, 4], or for
    a frame of more than DUMP_MAX_PIXELS pixels (the 4K frame has 8.3 M) that many pixels drawn with a fixed seed, shape
    [n, 4], with their row-major indices y * w + x in DIR/frame_pixel_index.npy (float64, exact), the same on every run."""
    import numpy as np
    px = frame.cpu().numpy()
    os.makedirs(directory, exist_ok=True)
    if px.shape[0] * px.shape[1] > DUMP_MAX_PIXELS:
        idx = np.sort(np.random.Generator(np.random.PCG64(0)).choice(px.shape[0] * px.shape[1], DUMP_MAX_PIXELS, replace=False))
        px = px.reshape(-1, 4)[idx]
        np.save(os.path.join(directory, "frame_pixel_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(directory, "frame.npy"), px.astype(np.float32))


# ------------------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clock / throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index: int):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
                 "hw_power_brake": 0x80, "sync_boost": 0x10}
        while not self._stop.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for n, bit in names.items():
                    if r & bit:
                        self.reasons.add(n)
            except Exception:
                pass
            self._stop.wait(0.05)

    def __enter__(self):
        if self.nv is not None:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._t:
            self._t.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml unavailable"]}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ------------------------------------------------------------------------------------------------------
def host_threads() -> int:
    """Threads the CPU arm may use: every core this process is allowed on (launchers such as torchrun export
    OMP_NUM_THREADS=1, which says nothing about the box)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


_ORACLE = {}


def cpu_oracle():
    """The reference's own CPU implementation of the path behind the oracle ABI.  Preference: the reference headers built
    -O3 -mavx2 -mfma with contraction (the fastest honest CPU build, when the host has AVX2+FMA), else the same headers
    built -O2 -ffp-contract=off, else the plain-C port.  The OpenMP team is set explicitly to every host core."""
    if "ora" not in _ORACLE:
        from oracle import Oracle, available
        kind = "reference_fast" if available("reference_fast") else ("reference" if available("reference") else "port")
        ora = Oracle(kind, auto_build=(kind == "port"))
        ora.set_num_threads(host_threads())
        _ORACLE["ora"], _ORACLE["kind"] = ora, kind
    return _ORACLE["ora"], _ORACLE["kind"]


def cpu_reference_run(w, h, repeats=1):
    """One w x h sample frame of the bench camera/parameters on the host cores.  Returns (steps, best_seconds, meta)."""
    import relativisticraytracer_b200 as rrt
    ora, kind = cpu_oracle()
    prm = ora.default_params(spin_a=SPIN)
    cam = ora.camera_from(CAM_POS, CAM_YAW, CAM_PITCH)
    fx = ora.default_effects()
    if "sky" not in _ORACLE:
        _ORACLE["sky"] = rrt.procedural_sky(4096, 2048)
    sky = _ORACLE["sky"]
    best, steps = 1e30, 0
    for _ in range(repeats):
        t0 = time.perf_counter()
        f = ora.render(prm, cam, fx, sky, TIME, w, h)
        best = min(best, time.perf_counter() - t0)
        steps = f.counters["rk4_steps"]
    flags = {"reference_fast": "reference headers, g++ -O3 -mavx2 -mfma -ffp-contract=fast",
             "reference": "reference headers, g++ -O2 -ffp-contract=off", "port": "plain-C port, gcc -O2 -ffp-contract=off"}[kind]
    return steps, best, {"kind": "port" if kind == "port" else "reference", "cores": ora.num_threads(),
                         "sample": f"{w}x{h} frame of the bench camera/params (a=0.99 disk+dust), {flags}, OpenMP dynamic rows"}


REFERENCE_ARM_BUDGET_S = 100.0   # wall-time bound of the whole --impl reference run (warm-up + timed steps)


def run_reference_arm(args):
    """--impl reference: the reference's CPU path on the host cores; rank 0 only (the other ranks exit at once).
    Each step is one sample frame of the bench workload (same camera, parameters, media, effects and sky; steps/s is
    resolution-invariant to ~0.1 %, SURVEY.md 8d).  The sample resolution is chosen from a 0.1-s calibration frame so
    that the whole run stays under REFERENCE_ARM_BUDGET_S whatever --steps/--warmup and core count are."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t_start = time.perf_counter()
    cpu_reference_run(160, 90)                                   # page the library in, spin the team up
    steps_c, dt_c, _ = cpu_reference_run(320, 180, repeats=2)
    per_pixel = dt_c / (320 * 180)
    n_frames = max(args.steps, 1) + max(args.warmup, 0)
    w, h = CPU_SAMPLE
    for cand in [(1280, 720), (960, 540), (640, 360), (480, 270), (320, 180)]:
        w, h = cand
        if per_pixel * w * h * n_frames <= REFERENCE_ARM_BUDGET_S - 10.0:
            break
    for _ in range(args.warmup):
        cpu_reference_run(w, h)
    tot_t, steps = 0.0, 0
    for _ in range(max(args.steps, 1)):
        steps, dt, meta = cpu_reference_run(w, h)
        tot_t += dt
    per = tot_t / max(args.steps, 1)
    value = steps / per
    line = {
        "impl": "reference", "metric": "geodesic_rk4_steps_per_s", "value": value, "unit": "steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": per * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample": meta["sample"], "sample_width": w, "sample_height": h,
                   "sample_note": "each step traces a bounded sample frame of the same camera/params instead of the 4K frame; "
                                  "steps/s is resolution-invariant (SURVEY.md 8d), so the unit compares like for like",
                   "rk4_steps_per_sample": steps, "host_threads": meta["cores"], "wall_s": time.perf_counter() - t_start},
        "cpu_baseline": {"value": value, "unit": "steps/s", "cores": meta["cores"], "kind": meta["kind"],
                         "sample": meta["sample"]},
        "e2e": {"value": value, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "frames_per_s_4k_equiv": value / (steps / (w * h)) / (W4K * H4K),
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------
def run_path_workload(args, r, sky, prm, world, rank, dev):
    """BASELINE config 5: 300 frames of the reference's 'Gargantua Fly-By' path (src/camera_paths.cpp:33-43) under
    the recorder's 1/24 s clock at 1080p, frame k on GPU k mod N, frames gathered to rank 0 over NCCL and copied to
    pinned host memory there (where the encoder would read them).  One timed pass over the whole path per step."""
    import torch
    import torch.distributed as dist
    import relativisticraytracer_b200 as rrt
    from relativisticraytracer_b200.parallel import PathSequence
    w, h = (1920, 1080) if (args.width, args.height) == (W4K, H4K) else (args.width, args.height)
    fx = rrt.default_effects()
    seq = PathSequence(r, w, h, depth=max(1, min(args.depth, 4)) if args.depth > 0 else 2)
    n = args.path_frames

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    seq.render(0, min(n, 2 * world * seq.depth), prm, fx, sky)          # warm-up: a few rounds
    barrier()
    r.read_counters(reset=True)
    times, launches = [], 0
    with ClockSampler(dev) as clk:
        for _ in range(max(1, args.steps)):
            barrier()
            t0 = time.perf_counter()
            done, l = seq.render(0, n, prm, fx, sky)
            barrier()
            times.append(time.perf_counter() - t0)
            launches += l
    cnt = r.read_counters(reset=True)
    tot = torch.tensor([cnt["rk4_steps"]], dtype=torch.float64, device="cuda")
    tmax = torch.tensor([sum(times)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tot)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    if rank != 0:
        return
    secs = float(tmax.item()) / len(times)
    steps_per_pass = float(tot.item()) / len(times)
    line = {
        "metric": "geodesic_rk4_steps_per_s", "value": steps_per_pass / secs, "unit": "steps/s", "n_gpus": world,
        "steps": len(times), "warmup": 1, "ms_per_step": secs * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{n}-frame Catmull-Rom camera path ('Gargantua Fly-By') at {w}x{h}, Kerr a=0.99 disk+dust, "
                               f"frame-parallel across {world} GPU(s), frames gathered to rank 0 and copied to host",
                   "frames": n, "fps_clock": 24, "frames_in_flight": seq.depth, "parallelism": f"frames{world}",
                   "rk4_steps_per_pass": steps_per_pass},
        "frames_per_s": n / secs,
        "e2e": {"value": steps_per_pass / secs, "unit": "steps/s", "frames_per_s": n / secs,
                "h2d_bytes_per_step": 164 * n, "d2h_bytes_per_step": w * h * 4 * n,
                "timing": "host wall clock around the whole path incl. gathers, device->host copies and final synchronize"},
        "gpu_launches": launches, "clocks": clk.summary(),
    }
    print(json.dumps(line), flush=True)


def path_subrecord(r, sky, prm, world, rank, n=48, w=1920, h=1080):
    """The first `n` frames of the reference's 'Gargantua Fly-By' path (src/camera_paths.cpp:33-43) under the recorder's
    1/24 s clock at 1080p, frame k rendered whole by rank k mod N, gathered to rank 0 and copied to pinned host memory in
    frame order (PathSequence).  Timed by the host clock between barriers; three of the gathered frames are then checked
    byte for byte against the same frames rendered by rank 0 alone.  Runs on every rank; returns the record on rank 0."""
    import numpy as np
    import torch
    import torch.distributed as dist
    import relativisticraytracer_b200 as rrt
    from relativisticraytracer_b200.parallel import PathSequence
    fx = rrt.default_effects()
    seq = PathSequence(r, w, h, depth=2)

    class Keep:                                    # a sink that keeps the frames it is handed (rank 0)
        def __init__(self):
            self.frames = []

        def write(self, t):
            self.frames.append(t.clone())

    seq.render(0, 2 * world * seq.depth, prm, fx, sky)                  # warm-up rounds
    torch.cuda.synchronize()
    dist.barrier()
    keep = Keep()
    t0 = time.perf_counter()
    done, launches = seq.render(0, n, prm, fx, sky, sink=keep if rank == 0 else None)
    torch.cuda.synchronize()
    dist.barrier()
    secs = time.perf_counter() - t0
    tm = torch.tensor([secs], dtype=torch.float64, device="cuda")
    dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    secs = float(tm.item())
    if rank != 0:
        return None
    ok = done == n and len(keep.frames) == n
    for k in (1, n // 2, n):
        t = rrt.path_clock(k, 24.0)
        cam, _ = rrt.path_state(0, t)
        want = np.zeros((h, w, 4), np.uint8)
        r.render_host(prm, cam, fx, sky, t, w, h, want)
        ok = ok and bool(np.array_equal(keep.frames[k - 1].numpy(), want))
    return {"workload": f"{n} frames of the 'Gargantua Fly-By' Catmull-Rom path at {w}x{h}, a=0.99 disk+dust, frame k on GPU k mod {world}, "
                        "gathered to rank 0 and copied to pinned host memory in frame order",
            "frames": n, "frames_per_s": n / secs, "seconds": secs, "frames_in_flight": seq.depth,
            "frames_equal_single_gpu_render": ok, "gpu_launches_rank0": launches,
            "timing": "host wall clock between barriers, max over ranks, device->host copies inside"}


# ------------------------------------------------------------------------------------------------------
def main():
    args = parse()
    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import torch.distributed as dist
    import relativisticraytracer_b200 as rrt

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    else:
        torch.cuda.set_device(0)
    dev = torch.cuda.current_device()
    w, h = args.width, args.height

    r = rrt.Renderer(dev)
    sky = r.create_sky(rrt.procedural_sky(4096, 2048))
    prm = rrt.default_params(spin_a=SPIN, flags=args.flags | (0 if args.strict else rrt.FLAG_FMAD))
    if args.workload == "path":
        run_path_workload(args, r, sky, prm, world, rank, dev)
        if world > 1:
            dist.destroy_process_group()
        return
    cams = {"C0": (CAM_POS, CAM_YAW, CAM_PITCH), "C1": ((15.0, 3.0, -30.0), -26.6, -5.1),
            "C2": ((35.0, 0.8, 10.0), -106.0, -1.2), "C3": ((4.2, 0.6, 4.2), -90.0, -5.7)}
    cam = rrt.camera_state_from(*cams[args.camera])
    fx = rrt.default_effects()
    headline = (w, h, args.flags & 3, args.camera, args.strict) == (W4K, H4K, 3, "C0", False)
    from relativisticraytracer_b200.parallel import BandedFrame
    bf = BandedFrame(r, w, h, BAND_GROUP, exchange=args.exchange)
    host_frame = torch.zeros((h, w, 4), dtype=torch.uint8).pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # > 126 MB L2
    stream = torch.cuda.current_stream()

    def one_frame(to_host: bool) -> int:
        """the hot path for one step; returns the number of OUR kernels launched"""
        if world == 1 and to_host:
            r.render_host(prm, cam, fx, sky, TIME, w, h, host_frame)   # the C-ABI call with a HOST destination
            return 1
        n = bf.render(prm, cam, fx, sky, TIME)                         # trace [+ NCCL gather + assemble on rank 0]
        if to_host and rank == 0:
            host_frame.copy_(bf.frame, non_blocking=True)
        return n

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(n_steps: int, to_host: bool):
        """K steps, each bracketed by barrier + synchronize; device time from CUDA events on the launching
        stream (host clock for the synchronous host-destination call); L2 flushed between steps."""
        total_ms, kernel_ms, launches = 0.0, 0.0, 0
        for _ in range(n_steps):
            flush.fill_(1)
            barrier()
            e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            t0 = time.perf_counter()
            e0.record(stream)
            if world == 1 and to_host:
                launches += one_frame(True)
                torch.cuda.synchronize()
                total_ms += (time.perf_counter() - t0) * 1e3
                continue
            if world == 1:
                launches += one_frame(to_host)
                e1.record(stream)
            elif bf.exchange == "peer":
                r.render(prm, cam, fx, sky, TIME, w, h, band=bf.band, out=bf.peer)      # stores land in rank 0's frame
                e1.record(stream)
                launches += 1
                dist.all_reduce(bf.token)                                               # every band has landed
                if to_host and rank == 0:
                    bf.peer.read_into(host_frame)
            else:
                r.render(prm, cam, fx, sky, TIME, w, h, band=bf.band, out=bf.packed, layout=rrt.OUT_PACKED)
                e1.record(stream)
                launches += 1
                if rank == 0:
                    dist.gather(bf.packed, list(bf.gathered.unbind(0)), dst=0)
                    r.assemble_bands(bf.gathered, bf.rows_max, w, h, world, BAND_GROUP, frame=bf.frame)
                    launches += 1
                    if to_host:
                        host_frame.copy_(bf.frame, non_blocking=True)
                else:
                    dist.gather(bf.packed, None, dst=0)
            e2.record(stream)
            torch.cuda.synchronize()
            total_ms += e0.elapsed_time(e2)
            kernel_ms += e0.elapsed_time(e1)
        return total_ms, kernel_ms, launches

    from relativisticraytracer_b200.parallel import FramePipeline

    def timed_sequence(pipe, share: int, n_steps: int):
        """K frames as a sequence with pipe.depth frames in flight (frame k on stream k % depth), each launch on
        1/share of the resident-CTA slots, the whole sequence bracketed by barrier + synchronize.
        Returns (device ms by CUDA events, host wall ms, launches)."""
        launches = 0
        r.set_frames_in_flight(share)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(stream)
        pipe.begin()
        for k in range(n_steps):
            with torch.cuda.stream(pipe.streams[pipe.submitted % pipe.depth]):
                flush.fill_(1)                                   # L2 flushed before every frame, in that frame's stream
            launches += pipe.submit(prm, cam, fx, sky, TIME)
        pipe.end()
        e1.record(stream)
        torch.cuda.synchronize()
        barrier()
        wall_ms = (time.perf_counter() - t0) * 1e3
        r.set_frames_in_flight(1)
        return e0.elapsed_time(e1), wall_ms, launches

    # How the sequence is scheduled.  A frame's kernel cannot finish faster than its critical path (one tile of
    # disk-plane rays, ~17 ms at 4K); when that is long against the frame's share of the work (band-parallel frames
    # at N >= 4) more frames in flight on a share of the CTA slots each keep the SMs busy, otherwise two frames
    # in flight on the whole GPU are best.  Unless --depth/--share pin it, both schedules are tried on a short
    # sequence at start-up and the faster one is used (the same on every rank: max over ranks decides).
    if args.depth > 0:
        depth = max(1, min(args.depth, 4))
        share = args.share if args.share > 0 else 1
        schedule_how = "fixed by --depth/--share"
    else:
        # trials of PICK_FRAMES frames each (short ones are noise-limited: 8-frame trials 1.5 % apart once picked the
        # slower schedule); the default "2 frames on the whole GPU" is kept unless the alternative is > 3 % faster
        cands = [(2, 1), (4, 2)]
        PICK_FRAMES = 24 if world > 1 else 12
        trial = []
        for d_, s_ in cands:
            pp = FramePipeline(r, w, h, BAND_GROUP, depth=d_, to_host=False, exchange=bf.exchange if world > 1 else "auto")
            timed_sequence(pp, s_, d_)                                     # warm the streams / buffers
            ms, _, _ = timed_sequence(pp, s_, PICK_FRAMES)
            tm = torch.tensor([ms], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            trial.append(float(tm.item()) / PICK_FRAMES)
            del pp
        pick = 1 if trial[1] < 0.97 * trial[0] else 0
        depth, share = cands[pick]
        schedule_how = (f"auto ({PICK_FRAMES}-frame trials, alternative must win by > 3 %): " +
                        ", ".join(f"depth {d_} on 1/{s_} of the CTA slots = {t_:.2f} ms/frame" for (d_, s_), t_ in zip(cands, trial)))
    xchg = bf.exchange if world > 1 else "auto"
    pipe_dev = FramePipeline(r, w, h, BAND_GROUP, depth=depth, to_host=False, exchange=xchg)
    pipe_host = FramePipeline(r, w, h, BAND_GROUP, depth=depth, to_host=True, exchange=xchg)

    # ---- warm-up, then the counted work of one step -------------------------------------------------
    timed(args.warmup, False)
    timed_sequence(pipe_dev, share, min(max(args.warmup, 1), depth))
    r.read_counters(reset=True)
    one_frame(False)
    torch.cuda.synchronize()
    cnt = r.read_counters(reset=True)
    steps_local = torch.tensor([cnt["rk4_steps"], cnt["disk_evals"], cnt["dust_evals"]], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(steps_local)
    rk4_per_frame, disk_evals, dust_evals = (float(x) for x in steps_local.tolist())

    # ---- single-frame latency and the kernel's own duration (each frame alone, bracketed) ----------------
    lat_ms, kern_ms, _ = timed(args.steps, False)
    # ---- timed region: K frames, device-resident, `depth` in flight -------------------------------------
    l0 = r.kernel_launches()
    with ClockSampler(dev) as clk:
        tot_ms, _, _ = timed_sequence(pipe_dev, share, args.steps)
    launches = r.kernel_launches() - l0          # kernels rank 0's context launched in the timed region (C-ABI counter)
    split = r.split_stats()
    # ---- timed region: end to end (HOST destination, device->host copy inside) --------------------------
    timed_sequence(pipe_host, share, min(2, args.steps))
    _, e2e_ms, _ = timed_sequence(pipe_host, share, args.steps)

    t = torch.tensor([tot_ms, kern_ms, e2e_ms, lat_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    tot_ms, kern_ms, e2e_ms, lat_ms = (float(x) for x in t.tolist())
    ms_per_step = tot_ms / args.steps
    kern_ms_per_step = kern_ms / args.steps
    e2e_ms_per_step = e2e_ms / args.steps
    lat_ms_per_step = lat_ms / args.steps
    value = rk4_per_frame / (ms_per_step * 1e-3)

    # ---- N > 1: BASELINE config 5 beside the headline (frame-parallel camera path, frame k on rank k mod N) ----------
    path_rec = None
    if world > 1 and not args.no_path:
        path_rec = path_subrecord(r, sky, prm, world, rank)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_frame(args.dump_outputs, pipe_dev.last_frame())     # the headline's device-resident frames; pipe_host has its own

    # ---- roofline of the dominant kernel (render_kernel): FP32 FMA pipe -------------------------------
    traffic = {"bytes": None, "source": "no ncu capture for this workload (see profiles/)"}
    if headline and world == 1:
        try:
            with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
                tj = json.load(f)
            traffic = {"bytes": float(tj["dram_bytes_read"]) + float(tj["dram_bytes_write"]),
                       "source": f"{tj['capture']} (dram__bytes_read.sum + dram__bytes_write.sum of one {tj.get('kernel', 'render_kernel')} launch, "
                                 f"ncu --set full, {tj['when']}); not measured by this run"}
        except (OSError, KeyError, ValueError):
            pass
    fp32_meas, _ = r.fp32_peak(4096)
    kern_steps_per_s = (rk4_per_frame / world) / (kern_ms_per_step * 1e-3)      # this rank's kernel (max over ranks time)
    achieved_tflops = FLOP_PER_STEP * kern_steps_per_s / 1e12
    roofline = {
        "bound": "fp32_fma", "achieved": achieved_tflops, "peak": fp32_meas, "unit": "TFLOP/s",
        "frac": achieved_tflops / fp32_meas,
        # DRAM bytes of one launch: not measurable from inside this process; the number is read from the committed
        # ncu --set full capture of this same command (profiles/ncu_traffic.json names the capture), headline workload only
        "traffic": traffic["bytes"], "traffic_source": traffic["source"],
        "peak_source": "FFMA-chain microbenchmark measured in this run (MEASURED_PEAKS.json has no FP32 entry)",
        "peak_theoretical": FP32_THEORETICAL_TFLOPS, "frac_of_theoretical": achieved_tflops / FP32_THEORETICAL_TFLOPS,
        "flop_per_step": FLOP_PER_STEP,
        "kernel": ("trace_kernel<spin> + media_kernel + fold_kernel (+ empty sweep_kernel): the launches of one frame, timed together"
                   if split["passes_enqueued"] else "render_kernel<spin,media>"),
        "kernel_ms": kern_ms_per_step,
        "note": "geodesic-step FLOPs only; disk/dust density evaluations (1.1k/4.1k FLOP each) are not credited",
    }

    line = {
        "metric": "geodesic_rk4_steps_per_s", "value": value, "unit": "steps/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD if headline else f"EXPERIMENT {w}x{h} flags={args.flags} camera={args.camera} variant of: {WORKLOAD}",
                   "width": w, "height": h, "spin_a": SPIN,
                   "media": {0: "none (geodesic only)", 1: "disk", 2: "dust", 3: "disk+dust"}[args.flags & 3], "camera": args.camera,
                   "band_group_rows": BAND_GROUP,
                   "parallelism": f"rowbands{world}", "exchange": bf.exchange, "l2": "flushed (256 MiB write) before every frame",
                   "frames_in_flight": depth, "cta_slots_per_frame": f"1/{share}", "schedule": schedule_how,
                   "rounding_contract": ("strict: unfused mul+add, the twin of the reference headers on a host" if args.strict else
                                         "fmad: the FMA fusion schedule of the reference's own CUDA build (default)"),
                   "rk4_steps_per_frame": rk4_per_frame, "disk_evals_per_frame": disk_evals, "dust_evals_per_frame": dust_evals},
        "frames_per_s": 1e3 / ms_per_step,
        "latency_ms_single_frame": lat_ms_per_step,
        "roofline": roofline,
        "e2e": {"value": rk4_per_frame / (e2e_ms_per_step * 1e-3), "unit": "steps/s",
                "frames_per_s": 1e3 / e2e_ms_per_step, "ms_per_step": e2e_ms_per_step,
                "h2d_bytes_per_step": 64 + 48 + 36 + 16, "d2h_bytes_per_step": w * h * 4,
                "timing": "host wall clock around the K-frame sequence incl. final synchronize",
                "path": ("rrt_render_host_async (C ABI, pinned host frames)" if world == 1 else
                         ("rrt_render per rank storing into rank 0's peer-mapped frame + 4-byte all-reduce + D2H to pinned host" if xchg == "peer"
                          else "rrt_render per rank + NCCL gather + rrt_assemble_bands + D2H to pinned host"))},
        "gpu_launches": launches,
        "pipeline": ({"kind": "split: trace / media / fold kernels over a sample pool in HBM (csrc/rrt_split.cuh)",
                      "passes_per_frame": split["passes_worked"], "passes_enqueued": split["passes_enqueued"],
                      "tiles_left_to_fused_sweep": split["tiles_swept"], "pool_GiB_per_stream": split["pool_kislots"] * 32 / 2 ** 20}
                     if split["passes_enqueued"] else {"kind": "fused: render_kernel"}),
        "clocks": clk.summary(),
    }

    if path_rec is not None:
        line["path"] = path_rec
    if world == 1 and not args.no_cpu_baseline:
        cw, ch = CPU_SAMPLE
        steps_c, secs, meta = cpu_reference_run(cw, ch, repeats=3)     # ~15 s of host work, best of 3
        line["cpu_baseline"] = {"value": steps_c / secs, "unit": "steps/s", "cores": meta["cores"], "kind": meta["kind"],
                                "sample": meta["sample"], "seconds": secs}
    if world == 1 and not args.no_ref_cuda:
        try:
            from oracle import RefCuda, Oracle
            if RefCuda.available():
                oc = Oracle("port")
                _, best, mean = RefCuda().render(SPIN, oc.camera_from(CAM_POS, CAM_YAW, CAM_PITCH), oc.default_effects(),
                                                 rrt.procedural_sky(4096, 2048), TIME, w, h, reps=3)
                line["ref_cuda_baseline"] = {"what": "reference src/raymarcher.cu unmodified, nvcc -O3 sm_100a, same frame",
                                             "ms_per_frame": mean, "best_ms": best, "steps_per_s": rk4_per_frame / (mean * 1e-3)}
        except Exception as e:  # a baseline, never the product: report and move on
            line["ref_cuda_baseline"] = {"unavailable": str(e)[:200]}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
