"""Multi-GPU sharding of the render path: one process per GPU, torch.distributed for the plumbing.

Every pixel is an independent pure function of (x, y, frame parameters) -- reference raymarch_kernel,
src/raymarcher.cu:15-174, has no inter-thread communication -- so a frame shards by image rows and a camera
path shards by frame.  The only exchange step is collecting finished pixels on the encoding GPU (rank 0):

* ``render_banded``: rows are cut into groups of ``group`` consecutive rows, group k goes to rank k % N
  (cyclic, because contiguous bands are 12-20 % imbalanced: the disk rows are the expensive ones); every rank
  traces its rows into a packed buffer, one NCCL gather over NVLink brings the N buffers to rank 0, and one
  small kernel (rrt_assemble_bands) scatters them into the row-flipped frame.  Bit-identical to one GPU.
* ``frame_owner`` / ``path_frames``: frame k of a path goes to rank k % N (BASELINE config 5).

Host-side index logic lives here in plain Python so it is testable on CPU with the gloo backend.
"""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch
import torch.distributed as dist

from ._capi import HOST_SLOTS, OUT_PACKED, Band

DEFAULT_GROUP = 8


def band_rows_of(rank: int, nranks: int, group: int, h: int) -> np.ndarray:
    """Global image rows owned by `rank`, in packed (local-row) order; mirrors the kernel's mapping
    y = ((l // group) * nranks + rank) * group + l % group."""
    if not (0 <= rank < nranks) or group <= 0:
        raise ValueError("bad band")
    rows = []
    ngroups = (h + group - 1) // group
    for g in range(rank, ngroups, nranks):
        rows.extend(range(g * group, min((g + 1) * group, h)))
    return np.asarray(rows, dtype=np.int64)


def max_band_rows(nranks: int, group: int, h: int) -> int:
    return max(len(band_rows_of(r, nranks, group, h)) for r in range(nranks))


def assemble_host(packed_all: np.ndarray, nranks: int, group: int, h: int) -> np.ndarray:
    """Host reference of rrt_assemble_bands: packed_all [nranks, rows_max, w, 4] -> row-flipped frame
    [h, w, 4] (pixel row y is stored at h-1-y, reference raymarcher.cu:168)."""
    w = packed_all.shape[2]
    frame = np.zeros((h, w, packed_all.shape[3]), packed_all.dtype)
    for r in range(nranks):
        ys = band_rows_of(r, nranks, group, h)
        frame[h - 1 - ys] = packed_all[r, : len(ys)]
    return frame


def gather_bands(packed: torch.Tensor, dst: int = 0, group=None) -> Optional[torch.Tensor]:
    """Collect every rank's packed band on `dst`; returns [nranks, rows_max, w, 4] there, None elsewhere.
    NCCL gather on GPU tensors (NVLink / NVSwitch), gloo on CPU tensors (tests)."""
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    if rank == dst:
        out = torch.empty((world,) + tuple(packed.shape), dtype=packed.dtype, device=packed.device)
        dist.gather(packed, list(out.unbind(0)), dst=dst, group=group)
        return out
    dist.gather(packed, None, dst=dst, group=group)
    return None


def share_peer_frames(renderer, h: int, w: int, count: int):
    """``count`` frames on rank 0's GPU that every rank's render kernel can store into (renderer.PeerFrame): rank 0
    creates them, the 64-byte CUDA IPC handles travel by broadcast_object_list, the other ranks map them.  Returns the
    list of PeerFrame objects, or None (on every rank alike) if any rank could not set the mapping up -- the caller then
    keeps the NCCL gather path."""
    from .renderer import PeerFrame
    rank = dist.get_rank()
    frames, handles, ok = [], [None] * count, 1
    if rank == 0:
        try:
            frames = [PeerFrame(renderer, h, w) for _ in range(count)]
            handles = [f.handle for f in frames]
        except Exception:
            ok, handles = 0, [None] * count
    dist.broadcast_object_list(handles, src=0)
    if rank != 0:
        try:
            if any(hd is None for hd in handles):
                raise RuntimeError("rank 0 has no peer frames")
            frames = [PeerFrame(renderer, h, w, handle=hd) for hd in handles]
        except Exception:
            ok = 0
    flag = torch.tensor([ok], dtype=torch.int32, device=renderer.device)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if int(flag.item()) == 0:
        for f in frames:
            f.close()
        return None
    return frames


def frame_owner(frame_index: int, nranks: int) -> int:
    """Frame-parallel path rendering: frame k -> rank k % N."""
    return frame_index % nranks


def path_frames(rank: int, nranks: int, n_frames: int):
    """Frames (1-based, as the recorder counts them) this rank renders."""
    return [k for k in range(1, n_frames + 1) if frame_owner(k, nranks) == rank]


def path_rounds(n_frames: int, nranks: int, first_frame: int = 1):
    """Frame-parallel schedule of ``PathSequence``: round j covers the next ``nranks`` consecutive frames and is the
    list, indexed by rank, of the frame that rank renders -- frame k belongs to rank ``frame_owner(k)`` = k % N --
    or ``None`` for a rank left without one in the last round.  Every frame first_frame .. first_frame+n_frames-1
    appears exactly once; within a round the sink takes them in increasing frame number."""
    rounds = []
    for j in range((n_frames + nranks - 1) // nranks):
        rnd = [None] * nranks
        for i in range(nranks):
            if j * nranks + i < n_frames:
                f = first_frame + j * nranks + i
                rnd[frame_owner(f, nranks)] = f
        rounds.append(rnd)
    return rounds


class BandedFrame:
    """Buffers + calls for one banded frame on this rank (see module docstring)."""

    def __init__(self, renderer, w: int, h: int, group: int = DEFAULT_GROUP, exchange: str = "auto"):
        """exchange: "peer" = every rank's kernel stores straight into rank 0's frame (CUDA IPC mapping, see
        rrt_peer_frame_*), a 4-byte all-reduce is the barrier; "nccl" = packed bands + NCCL gather + rrt_assemble_bands;
        "auto" = peer when the mapping can be set up on every rank, else nccl."""
        self.r, self.w, self.h, self.group = renderer, w, h, group
        self.world = dist.get_world_size() if dist.is_initialized() else 1
        self.rank = dist.get_rank() if dist.is_initialized() else 0
        self.band = Band(self.rank, self.world, group)
        self.rows_max = max_band_rows(self.world, group, h)
        dev = renderer.device
        self.peer = None
        if self.world > 1 and exchange in ("auto", "peer"):
            pf = share_peer_frames(renderer, h, w, 1)
            if pf is None and exchange == "peer":
                raise RuntimeError("peer frames unavailable (CUDA IPC mapping failed on some rank)")
            self.peer = pf[0] if pf else None
        self.exchange = "peer" if self.peer is not None else ("nccl" if self.world > 1 else "none")
        self.token = torch.zeros(1, dtype=torch.int32, device=dev)
        self.packed = self.gathered = None
        if self.exchange == "nccl":
            self.packed = torch.zeros((self.rows_max, w, 4), dtype=torch.uint8, device=dev)
            self.gathered = torch.zeros((self.world, self.rows_max, w, 4), dtype=torch.uint8, device=dev) if self.rank == 0 else None
        self.frame = torch.zeros((h, w, 4), dtype=torch.uint8, device=dev) if self.rank == 0 else None

    def render(self, prm, cam, fx, sky, time: float) -> int:
        """Trace this rank's rows and bring them together on rank 0.  Returns how many of OUR kernels were launched."""
        l0 = self.r.kernel_launches()   # the context counts its own kernels (1 fused, or 3 per pass + 1 in the split pipeline)
        if self.world == 1:
            self.r.render(prm, cam, fx, sky, time, self.w, self.h, out=self.frame)
            return self.r.kernel_launches() - l0
        if self.exchange == "peer":
            # the store that ends the path is the exchange; the all-reduce orders rank 0's consumers after every band
            self.r.render(prm, cam, fx, sky, time, self.w, self.h, band=self.band, out=self.peer)
            dist.all_reduce(self.token)
            if self.rank == 0:
                self.peer.read_into(self.frame)     # 33 MB device-to-device at 4K (~10 us): hands the frame to torch
            return self.r.kernel_launches() - l0
        self.r.render(prm, cam, fx, sky, time, self.w, self.h, band=self.band, out=self.packed, layout=OUT_PACKED)
        if self.rank == 0:
            dist.gather(self.packed, list(self.gathered.unbind(0)), dst=0)
            self.r.assemble_bands(self.gathered, self.rows_max, self.w, self.h, self.world, self.group, frame=self.frame)
            return self.r.kernel_launches() - l0
        dist.gather(self.packed, None, dst=0)
        return self.r.kernel_launches() - l0


class FramePipeline:
    """A sequence of frames with ``depth`` of them in flight (the recorder loop of the reference renders frame
    after frame, src/main.cpp:505-528).

    Frame k runs on CUDA stream k % depth with its own buffers: trace of this rank's rows [+ NCCL gather to
    rank 0 + rrt_assemble_bands there] [+ device->host copy into a pinned frame on rank 0].  Within one stream
    the order is kept, between streams nothing waits, so the drain of frame k -- the few warps still
    integrating the expensive disk-plane rays while most SMs are already idle -- overlaps with the start of
    frame k+1 instead of leaving the GPU empty.  Every pixel is the same pure function of its frame's inputs
    as in the unpipelined call, so results are identical.
    """

    def __init__(self, renderer, w: int, h: int, group: int = DEFAULT_GROUP, depth: int = 2, to_host: bool = False,
                 exchange: str = "auto"):
        if not 1 <= depth <= HOST_SLOTS:
            raise ValueError(f"depth must be 1..{HOST_SLOTS}")
        self.r, self.w, self.h, self.group, self.depth, self.to_host = renderer, w, h, group, depth, to_host
        self.world = dist.get_world_size() if dist.is_initialized() else 1
        self.rank = dist.get_rank() if dist.is_initialized() else 0
        self.band = Band(self.rank, self.world, group)
        self.rows_max = max_band_rows(self.world, group, h)
        dev = renderer.device
        self.streams = [torch.cuda.Stream(device=dev) for _ in range(depth)]
        # one completion event per slot: recorded at the end of the slot's work, waited on before the slot's buffers are
        # reused by a later submit() and before last_frame() hands the destination to a consumer
        self.done = [torch.cuda.Event() for _ in range(depth)]
        self.busy = [False] * depth
        root = self.rank == 0
        # exchange step of a band-parallel frame, see BandedFrame
        self.peer = None
        if self.world > 1 and exchange in ("auto", "peer"):
            self.peer = share_peer_frames(renderer, h, w, depth)
            if self.peer is None and exchange == "peer":
                raise RuntimeError("peer frames unavailable (CUDA IPC mapping failed on some rank)")
        self.exchange = "peer" if self.peer is not None else ("nccl" if self.world > 1 else "none")
        self.tokens = [torch.zeros(1, dtype=torch.int32, device=dev) for _ in range(depth)]
        nccl = self.exchange == "nccl"
        self.packed = [torch.zeros((self.rows_max, w, 4), dtype=torch.uint8, device=dev) for _ in range(depth)] if nccl else None
        self.gathered = ([torch.zeros((self.world, self.rows_max, w, 4), dtype=torch.uint8, device=dev) for _ in range(depth)]
                         if root and nccl else None)
        need_dev_frame = root and (self.world > 1 or not to_host)
        if self.peer is not None:
            need_dev_frame = root and not to_host
        self.frames = [torch.zeros((h, w, 4), dtype=torch.uint8, device=dev) for _ in range(depth)] if need_dev_frame else None
        self.host_frames = ([torch.zeros((h, w, 4), dtype=torch.uint8).pin_memory() for _ in range(depth)]
                            if root and to_host else None)
        self.submitted = 0

    def begin(self) -> None:
        """Order every pipeline stream after the work already queued on the current stream."""
        cur = torch.cuda.current_stream(self.r.device)
        for s in self.streams:
            s.wait_stream(cur)

    def submit(self, prm, cam, fx, sky, time: float) -> int:
        """Enqueue one frame; returns how many of OUR kernels that launched on this rank."""
        k = self.submitted % self.depth
        self.submitted += 1
        s = self.streams[k]
        l0 = self.r.kernel_launches()   # the context counts its own kernels (1 fused, or 3 per pass + 1 in the split pipeline)
        if self.world == 1:
            if self.to_host:   # the C-ABI call with a HOST destination, asynchronous flavour
                self.r.render_host_async(prm, cam, fx, sky, time, self.w, self.h, self.host_frames[k], slot=k, stream=s)
            else:
                self.r.render(prm, cam, fx, sky, time, self.w, self.h, out=self.frames[k], stream=s)
            self.done[k].record(s)
            self.busy[k] = True
            return self.r.kernel_launches() - l0
        if self.exchange == "peer":
            with torch.cuda.stream(s):
                # every rank's kernel stores its rows straight into slot k of rank 0's frames; all-reduce #1 tells rank 0
                # that all bands have landed, all-reduce #2 (after rank 0's device->host copy) tells the others that the
                # slot may be overwritten by frame k + depth
                self.r.render(prm, cam, fx, sky, time, self.w, self.h, band=self.band, out=self.peer[k], stream=s)
                dist.all_reduce(self.tokens[k])
                if self.rank == 0:
                    self.peer[k].read_into(self.host_frames[k] if self.to_host else self.frames[k], stream=s)
                dist.all_reduce(self.tokens[k])
                self.done[k].record(s)
            self.busy[k] = True
            return self.r.kernel_launches() - l0
        with torch.cuda.stream(s):
            self.r.render(prm, cam, fx, sky, time, self.w, self.h, band=self.band, out=self.packed[k], layout=OUT_PACKED, stream=s)
            if self.rank == 0:
                dist.gather(self.packed[k], list(self.gathered[k].unbind(0)), dst=0)
                self.r.assemble_bands(self.gathered[k], self.rows_max, self.w, self.h, self.world, self.group,
                                      frame=self.frames[k], stream=s)
                if self.to_host:
                    self.host_frames[k].copy_(self.frames[k], non_blocking=True)
            else:
                dist.gather(self.packed[k], None, dst=0)
            self.done[k].record(s)
        self.busy[k] = True
        return self.r.kernel_launches() - l0

    def wait_slot(self, k: int) -> None:
        """Block the host until the frame last submitted to slot k is complete (its destination may then be read, and
        the slot's buffers are free for the next submit; submits to one slot are ordered by its stream anyway)."""
        if self.busy[k]:
            self.done[k].synchronize()
            self.busy[k] = False

    def end(self) -> None:
        """Order the current stream after every frame submitted so far (no host synchronisation)."""
        cur = torch.cuda.current_stream(self.r.device)
        for s in self.streams:
            cur.wait_stream(s)

    def last_frame(self):
        """The most recently submitted frame's destination on rank 0 (host tensor if to_host, else device), complete:
        the slot's event is synchronised first, so a consumer never reads a half-copied frame.  It stays valid until
        `depth` further submits reuse the slot."""
        if self.submitted == 0:
            return None
        k = (self.submitted - 1) % self.depth
        self.wait_slot(k)
        if self.rank != 0:
            return None
        return self.host_frames[k] if self.to_host else self.frames[k]


class PathSequence:
    """Frame-parallel rendering of a keyframe camera path (BASELINE config 5; reference P + R keys:
    PathController playback under the recorder's fixed 1/fps clock, src/main.cpp:171-220, 505-528).

    Frames are 1-based like the recorder counts them.  Round j covers frames j*N+1 .. j*N+N; frame k is rendered
    whole by rank k % N (``frame_owner``, ``path_rounds``), one NCCL gather per round brings the N frames to
    rank 0 (the encoding GPU), which copies them to pinned host memory and hands them to the sink in frame order.  Rounds
    are pipelined ``depth`` deep on separate streams like ``FramePipeline``.  Camera and clock come from the
    C-ABI host functions (``rrt_path_state`` / ``rrt_path_clock``), so frame k is the same pure function of k
    on every rank count.  ``ss`` > 1 renders every frame anti-aliased with ss x ss rays per pixel (``Renderer.render_ss``
    into the slot's device frame, then the same pinned copy), which keeps the photon ring, the disk's inner edge and the
    stars from crawling between frames.  ``samples`` > 1 renders every frame motion-blurred (``Renderer.render_mb``): a
    shutter open for ``shutter`` (0..1) of the frame interval, centred on the frame's clock, with ``samples`` sub-frames at
    ``shutter_times(path_clock(k, fps), shutter, fps, samples)``, each with the path's camera at its own time, so that the
    disk's rotation and the camera's motion smear instead of strobing.  ``samples`` > 1 does not combine with ``ss`` > 1
    here; the C ABI composes the two (rrt_resolve_time, then rrt_resolve)."""

    def __init__(self, renderer, w: int, h: int, depth: int = 2, ss: int = 1, shutter: float = 0.0, samples: int = 1):
        if not 1 <= depth <= HOST_SLOTS:
            raise ValueError(f"depth must be 1..{HOST_SLOTS}")
        if not 1 <= ss <= 8:
            raise ValueError("ss must be 1..8")
        if not 1 <= samples <= 64:
            raise ValueError("samples must be 1..64")
        if not 0.0 <= shutter <= 1.0:
            raise ValueError("shutter must be in [0, 1]")
        if ss > 1 and samples > 1:
            raise ValueError("ss > 1 together with samples > 1 is not supported by PathSequence")
        self.r, self.w, self.h, self.depth, self.ss = renderer, w, h, depth, ss
        self.shutter, self.samples = float(shutter), samples
        self.world = dist.get_world_size() if dist.is_initialized() else 1
        self.rank = dist.get_rank() if dist.is_initialized() else 0
        dev = renderer.device
        self.streams = [torch.cuda.Stream(device=dev) for _ in range(depth)]
        self.events = [torch.cuda.Event() for _ in range(depth)]
        root = self.rank == 0
        self.local = ([torch.zeros((h, w, 4), dtype=torch.uint8, device=dev) for _ in range(depth)]
                      if self.world > 1 or ss > 1 or samples > 1 else None)
        self.gathered = ([torch.zeros((self.world, h, w, 4), dtype=torch.uint8, device=dev) for _ in range(depth)]
                         if root and self.world > 1 else None)
        self.host = [torch.zeros((self.world, h, w, 4), dtype=torch.uint8).pin_memory() for _ in range(depth)] if root else None

    def render(self, path_index: int, n_frames: int, prm, fx, sky, fps: float = 24.0, sink=None, first_frame: int = 1):
        """Render frames first_frame .. first_frame+n_frames-1 of the path.  Returns (frames_done, launches)."""
        from .renderer import path_clock, path_state, shutter_times
        cur = torch.cuda.current_stream(self.r.device)
        for s in self.streams:
            s.wait_stream(cur)
        schedule = path_rounds(n_frames, self.world, first_frame)
        rounds = len(schedule)
        in_flight = [None] * self.depth     # per slot: list of frame numbers it holds
        done = 0
        l0 = self.r.kernel_launches()       # the context counts its own kernels

        def retire(k):
            nonlocal done
            if in_flight[k] is None:
                return
            self.events[k].synchronize()
            if self.rank == 0:
                for f, i in sorted((f, i) for i, f in enumerate(in_flight[k]) if f is not None):   # frame order
                    if sink is not None:
                        sink.write(self.host[k][i])
                    done += 1
            in_flight[k] = None

        for j in range(rounds):
            k = j % self.depth
            retire(k)
            frames = schedule[j]
            mine = frames[self.rank]
            s = self.streams[k]
            with torch.cuda.stream(s):
                if self.world == 1 and self.ss == 1 and self.samples == 1:
                    t = path_clock(mine, fps)
                    cam, _ = path_state(path_index, t)
                    self.r.render_host_async(prm, cam, fx, sky, t, self.w, self.h, self.host[k][0], slot=k, stream=s)
                else:
                    if mine is not None:
                        t = path_clock(mine, fps)
                        cam, _ = path_state(path_index, t)
                        if self.samples > 1:
                            times = shutter_times(t, self.shutter, fps, self.samples)
                            cams = [path_state(path_index, ti)[0] for ti in times]
                            self.r.render_mb(prm, cams, fx, sky, times, self.w, self.h, out=self.local[k], stream=s)
                        elif self.ss == 1:
                            self.r.render(prm, cam, fx, sky, t, self.w, self.h, out=self.local[k], stream=s)
                        else:
                            self.r.render_ss(prm, cam, fx, sky, t, self.w, self.h, self.ss, out=self.local[k], stream=s)
                    if self.world == 1:
                        self.host[k][0].copy_(self.local[k], non_blocking=True)
                    elif self.rank == 0:
                        dist.gather(self.local[k], list(self.gathered[k].unbind(0)), dst=0)
                        self.host[k].copy_(self.gathered[k], non_blocking=True)
                    else:
                        dist.gather(self.local[k], None, dst=0)
                self.events[k].record(s)
            in_flight[k] = frames
        for j in range(rounds, rounds + self.depth):
            retire(j % self.depth)
        for s in self.streams:
            cur.wait_stream(s)
        return done, self.r.kernel_launches() - l0
