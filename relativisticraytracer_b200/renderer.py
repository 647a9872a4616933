"""Host-side mirror of the reference's render interface over the C ABI.

The reference exposes one call, ``launch_raymarch(d_out, w, h, time, cam, skyboxTex, effects)``
(include/raymarcher.h:19), fed by ``CameraController::getCUDAStateFrom`` (src/main.cpp:141-167) and
``loadSkybox`` (src/main.cpp:237-266).  This module keeps those names and argument meanings.  PyTorch is
used for what it is good at here -- device buffers, streams and (in ``parallel.py``) ``torch.distributed``;
every pixel is computed by the hand-written sm_100a kernels in ``csrc/`` through ``librrt_b200.so``.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np
import torch

from . import _capi
from ._capi import (Band, Camera, Counters, Effects, Params, Planes, RrtError, OUT_FRAME, OUT_PACKED,
                    default_effects, default_params, effects_off)

CameraState = Camera      # reference name (include/raymarcher.h:11)
CameraEffects = Effects   # reference name (camera_settings.h:4)


def camera_state_from(pos, yaw_deg: float, pitch_deg: float) -> Camera:
    """CameraController::getCUDAStateFrom (src/main.cpp:141-167); angles in degrees.  Host only."""
    cam = Camera()
    arr = (C.c_float * 3)(*[float(x) for x in pos])
    _capi.load().rrt_camera_from(C.byref(arr), float(yaw_deg), float(pitch_deg), C.byref(cam))
    return cam


def path_names():
    lib = _capi.load()
    return [lib.rrt_path_name(i).decode() for i in range(lib.rrt_path_count())]


def path_state(path_index: int, t: float):
    """PathController::getInterpolatedState (src/main.cpp:176-203) -> (Camera, [x,y,z,yaw,pitch])."""
    cam = Camera()
    pyp = np.zeros(5, np.float32)
    rc = _capi.load().rrt_path_state(int(path_index), float(t), C.byref(cam), pyp.ctypes.data_as(C.c_void_p))
    if rc != 0:
        raise RrtError(rc, f"rrt_path_state({path_index}, {t})")
    return cam, pyp


def path_clock(frame: int, fps: float = 24.0) -> float:
    """pathTime after `frame` float accumulations of 1/fps (recording clock, src/main.cpp:511-516)."""
    return float(_capi.load().rrt_path_clock(int(frame), float(fps)))


def path_duration(path_index: int) -> float:
    return float(_capi.load().rrt_path_duration(int(path_index)))


def shutter_times(t: float, shutter: float, fps: float, n: int) -> list:
    """rrt_shutter_times: the n sub-frame times of a shutter open for ``shutter`` (0..1) of the frame interval 1/fps,
    centred on t: t + (shutter/fps) * ((i + 0.5)/n - 0.5), each operation in float32.  n = 1 gives [t].  Host only."""
    out = (C.c_float * max(int(n), 1))()
    rc = _capi.load().rrt_shutter_times(float(t), float(shutter), float(fps), int(n), out)
    if rc != 0:
        raise RrtError(rc, f"rrt_shutter_times({t}, {shutter}, {fps}, {n}): shutter must be in [0, 1], fps > 0, n in 1..64")
    return [float(v) for v in out]


def _f32_array(values) -> C.Array:
    values = [float(v) for v in values]
    return (C.c_float * len(values))(*values)


class Sky:
    """A skybox texture object (rrt_sky) -- the device half of the reference's loadSkybox."""

    def __init__(self, renderer: "Renderer", rgba: np.ndarray):
        rgba = np.ascontiguousarray(rgba, dtype=np.uint8)
        if rgba.ndim != 3 or rgba.shape[2] != 4:
            raise ValueError("sky must be [h, w, 4] uint8 (RGBA8, rows top-down as stbi_load returns them)")
        self._r = renderer
        self._h = C.c_void_p()
        self.height, self.width = int(rgba.shape[0]), int(rgba.shape[1])
        renderer._check(renderer._lib.rrt_sky_create(renderer._ctx, rgba.ctypes.data_as(C.c_void_p), self.width,
                                                     self.height, C.byref(self._h)))
        self.texture = int(renderer._lib.rrt_sky_texture(self._h))   # cudaTextureObject_t

    def close(self):
        if self._h:
            self._r._lib.rrt_sky_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Capture:
    """One traced frame kept for renders at other times (rrt_capture): ``Renderer.capture`` traces once, ``render`` evaluates
    the disk and dust at a new time and folds, shades and stores without tracing again.  ``render(prm, fx, sky, t)`` gives
    the bytes of ``Renderer.render`` with the capture's parameters, camera, size and band, ``prm``'s exposure, ``fx``'s
    bloom / vignette / CA settings, ``sky`` and time ``t``; ``prm`` must keep the capture's FLAG_FMAD bit and ``fx`` its lens
    fields."""

    def __init__(self, renderer: "Renderer", prm: Params, cam: Camera, fx: Effects, sky: "Sky | int", w: int, h: int, *,
                 band: Optional[Band] = None, max_bytes: int = 0, stream: Optional[torch.cuda.Stream] = None):
        tex = sky.texture if isinstance(sky, Sky) else int(sky)
        self._r, self.w, self.h, self.band = renderer, int(w), int(h), band
        self._h = C.c_void_p()
        st = stream if stream is not None else torch.cuda.current_stream(renderer.device)
        renderer._check(renderer._lib.rrt_capture_create(renderer._ctx, C.byref(prm), C.byref(cam), C.byref(fx), C.c_uint64(tex),
                                                         self.w, self.h, C.byref(band) if band is not None else None,
                                                         C.c_size_t(int(max_bytes)), C.c_void_p(st.cuda_stream), C.byref(self._h)))

    def render(self, prm: Params, fx: Effects, sky: "Sky | int", time: float, *, out=None, layout: int = OUT_FRAME,
               hdr_out: Optional[torch.Tensor] = None, stream: Optional[torch.cuda.Stream] = None) -> torch.Tensor:
        """rrt_capture_render: the captured frame (or band) at ``time``; asynchronous.  ``out`` (a tensor or a PeerFrame),
        ``layout`` and ``hdr_out`` ((h, w, 4) float32) as in ``Renderer.render`` / ``Renderer.shade``; returns the frame."""
        r = self._r
        tex = sky.texture if isinstance(sky, Sky) else int(sky)
        out, out_ptr = r._frame_out(out, layout, self.band, self.w, self.h)
        hdr_ptr = r._plane_ptr("hdr", hdr_out, self.w, self.h) if hdr_out is not None else None
        st = stream if stream is not None else torch.cuda.current_stream(r.device)
        r._check(r._lib.rrt_capture_render(self._h, C.byref(prm), C.byref(fx), C.c_uint64(tex), float(time), C.c_void_p(out_ptr),
                                           int(layout), C.c_void_p(hdr_ptr), C.c_void_p(st.cuda_stream)))
        return out

    def render_mb(self, prm: Params, fx: Effects, sky: "Sky | int", times, *, out=None, layout: int = OUT_FRAME,
                  hdr_out: Optional[torch.Tensor] = None, stream: Optional[torch.cuda.Stream] = None) -> torch.Tensor:
        """rrt_capture_render_mb: the captured frame motion-blurred over ``times`` (1..64 sub-frames), without a new trace;
        asynchronous.  Gives the bytes of ``Renderer.render_mb`` with the capture's camera for every sub-frame, under the
        rules of ``render``.  ``out``, ``layout`` and ``hdr_out`` (the mean) as in ``render``; returns the frame."""
        r = self._r
        tex = sky.texture if isinstance(sky, Sky) else int(sky)
        ts = _f32_array(times)
        out, out_ptr = r._frame_out(out, layout, self.band, self.w, self.h)
        hdr_ptr = r._plane_ptr("hdr", hdr_out, self.w, self.h) if hdr_out is not None else None
        st = stream if stream is not None else torch.cuda.current_stream(r.device)
        r._check(r._lib.rrt_capture_render_mb(self._h, C.byref(prm), C.byref(fx), C.c_uint64(tex), ts, len(ts), C.c_void_p(out_ptr),
                                              int(layout), C.c_void_p(hdr_ptr), C.c_void_p(st.cuda_stream)))
        return out

    def info(self) -> dict:
        """rrt_capture_info: what the capture holds."""
        out = (C.c_uint64 * 8)()
        self._r._check(self._r._lib.rrt_capture_info(self._h, out))
        return {"samples": int(out[0]), "slots": int(out[1]), "bytes": int(out[2]), "groups_queued": int(out[3]),
                "tiles_left": int(out[4]), "packed": bool(out[5]), "tiles": int(out[6]), "pool_bytes": int(out[7])}

    def close(self):
        if self._h:
            self._r._lib.rrt_capture_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


PLANE_SPECS = {"hdr": (4, torch.float32), "dir": (4, torch.float32), "emis": (4, torch.float32),
               "pos": (4, torch.float32), "vel": (4, torch.float32), "cls": (0, torch.uint8), "steps": (0, torch.int32)}
# the planes Renderer.shade / rrt_shade re-shade a traced frame from (16 + 16 + 16 + 1 bytes per pixel)
TRACE_PLANES = ("hdr", "emis", "vel", "cls")


class PeerFrame:
    """A device frame on the encoding GPU that other processes' render kernels store into directly (C ABI
    rrt_peer_frame_*; CUDA IPC).  The owner (rank 0) creates it and passes ``handle`` (64 bytes) to the other ranks,
    which ``open`` it; the owner reads the assembled frame out with ``read_into`` (pinned host or device tensor)."""

    def __init__(self, renderer: "Renderer", h: int, w: int, handle: Optional[bytes] = None):
        self.r, self.h, self.w, self.nbytes = renderer, h, w, h * w * 4
        self.owner = handle is None
        ptr = C.c_void_p()
        if self.owner:
            buf = (C.c_uint8 * 64)()
            renderer._check(renderer._lib.rrt_peer_frame_create(renderer._ctx, C.c_size_t(self.nbytes), C.byref(ptr), buf))
            self.handle = bytes(buf)
        else:
            assert len(handle) == 64
            self.handle = bytes(handle)
            buf = (C.c_uint8 * 64).from_buffer_copy(self.handle)
            renderer._check(renderer._lib.rrt_peer_frame_open(renderer._ctx, buf, C.byref(ptr)))
        self.ptr = int(ptr.value)

    def read_into(self, dst: torch.Tensor, stream: Optional[torch.cuda.Stream] = None) -> None:
        """Stream-ordered copy of the frame into `dst` (pinned host or device uint8 tensor of the frame's size)."""
        assert dst.dtype == torch.uint8 and dst.is_contiguous() and dst.numel() == self.nbytes
        st = stream if stream is not None else torch.cuda.current_stream(self.r.device)
        self.r._check(self.r._lib.rrt_peer_frame_read(self.r._ctx, C.c_void_p(self.ptr), C.c_size_t(self.nbytes),
                                                      C.c_void_p(dst.data_ptr()), C.c_void_p(st.cuda_stream)))

    def close(self):
        if self.ptr:
            self.r._lib.rrt_peer_frame_close(self.r._ctx, C.c_void_p(self.ptr), 1 if self.owner else 0)
            self.ptr = 0


class Renderer:
    """One rrt_context on one B200.  Thread-compatible; launches are asynchronous on the given stream."""

    def __init__(self, device: int | None = None):
        self._lib = _capi.load()
        if not torch.cuda.is_available():
            raise RuntimeError("relativisticraytracer_b200 needs a CUDA device (no CPU fallback exists)")
        self.device_index = torch.cuda.current_device() if device is None else int(device)
        self.device = torch.device("cuda", self.device_index)
        self._ctx = C.c_void_p()
        rc = self._lib.rrt_context_create(self.device_index, C.byref(self._ctx))
        if rc != 0:
            raise RrtError(rc, (self._lib.rrt_last_error(None) or b"").decode())

    # ---- plumbing -------------------------------------------------------------------------------
    def _check(self, rc: int):
        if rc != 0:
            raise RrtError(rc, (self._lib.rrt_last_error(self._ctx) or b"").decode())

    def close(self):
        if self._ctx:
            self._lib.rrt_context_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def create_sky(self, rgba: np.ndarray) -> Sky:
        return Sky(self, rgba)

    @staticmethod
    def band_rows(band: Optional[Band], h: int) -> int:
        return int(_capi.load().rrt_band_rows(C.byref(band) if band is not None else None, int(h)))

    def alloc_planes(self, w: int, h: int, names=("hdr", "dir", "emis", "pos", "vel", "cls", "steps")):
        out = {}
        for n in names:
            ch, dt = PLANE_SPECS[n]
            shape = (h, w, ch) if ch else (h, w)
            out[n] = torch.zeros(shape, dtype=dt, device=self.device)
        return out

    # ---- the hot path -----------------------------------------------------------------------------
    def render(self, prm: Params, cam: Camera, fx: Effects, sky: Sky | int, time: float, w: int, h: int, *,
               band: Optional[Band] = None, out: Optional[torch.Tensor] = None, layout: int = OUT_FRAME,
               planes: Optional[dict] = None, stream: Optional[torch.cuda.Stream] = None) -> torch.Tensor:
        """rrt_render: one frame (or one band of it) into a device uchar4 tensor; asynchronous."""
        tex = sky.texture if isinstance(sky, Sky) else int(sky)
        out, out_ptr = self._frame_out(out, layout, band, w, h)
        pl = self._planes(planes, w, h) if planes else None
        st = stream if stream is not None else torch.cuda.current_stream(self.device)
        self._check(self._lib.rrt_render(self._ctx, C.byref(prm), C.byref(cam), C.byref(fx), C.c_uint64(tex),
                                         float(time), int(w), int(h), C.byref(band) if band is not None else None,
                                         C.c_void_p(out_ptr), int(layout),
                                         C.byref(pl) if pl is not None else None, C.c_void_p(st.cuda_stream)))
        return out

    def shade(self, prm: Params, fx: Effects, sky: Sky | int, traced: dict, w: int, h: int, *, band: Optional[Band] = None,
              out: Optional[torch.Tensor] = None, layout: int = OUT_FRAME, hdr_out: Optional[torch.Tensor] = None,
              stream: Optional[torch.cuda.Stream] = None) -> torch.Tensor:
        """rrt_shade: the step after the ray loop (sky, bloom, vignette, chromatic aberration, exposure tonemap, store)
        again from the planes of an earlier ``render(..., planes=traced)`` with at least TRACE_PLANES, without tracing;
        asynchronous.  Gives the bytes (and ``hdr_out`` values) of a fresh render with this sky, exposure and bloom /
        vignette / CA settings; ``prm`` must keep the trace's FLAG_FMAD bit and ``fx`` its lens fields.  ``band``,
        ``out`` (a tensor or a PeerFrame) and ``layout`` as in ``render``; returns the frame."""
        tex = sky.texture if isinstance(sky, Sky) else int(sky)
        out, out_ptr = self._frame_out(out, layout, band, w, h)
        pl = self._planes(traced, w, h)
        hdr_ptr = self._plane_ptr("hdr", hdr_out, w, h) if hdr_out is not None else None
        st = stream if stream is not None else torch.cuda.current_stream(self.device)
        self._check(self._lib.rrt_shade(self._ctx, C.byref(prm), C.byref(fx), C.c_uint64(tex), int(w), int(h),
                                        C.byref(band) if band is not None else None, C.byref(pl), C.c_void_p(out_ptr),
                                        int(layout), C.c_void_p(hdr_ptr), C.c_void_p(st.cuda_stream)))
        return out

    def render_ss(self, prm: Params, cam: Camera, fx: Effects, sky: Sky | int, time: float, w: int, h: int, ss: int, *,
                  band: Optional[Band] = None, out=None, layout: int = OUT_FRAME, hdr_out: Optional[torch.Tensor] = None,
                  stream: Optional[torch.cuda.Stream] = None) -> torch.Tensor:
        """rrt_render_ss: one anti-aliased frame (or band) with ss x ss rays per pixel, 1 <= ss <= 8; asynchronous.
        Pixel (x, y) is the box-filtered mean of pixels (ss*x + i, ss*y + j) of the ss*w x ss*h render, then the render's
        own bloom / vignette / tonemap; ss = 1 is ``render``.  ``hdr_out`` (h, w, 4) float32 receives the averaged linear
        value (.w = mean T).  ``band``, ``out`` (a tensor or a PeerFrame) and ``layout`` as in ``render``."""
        tex = sky.texture if isinstance(sky, Sky) else int(sky)
        out, out_ptr = self._frame_out(out, layout, band, w, h)
        hdr_ptr = self._plane_ptr("hdr", hdr_out, w, h) if hdr_out is not None else None
        st = stream if stream is not None else torch.cuda.current_stream(self.device)
        self._check(self._lib.rrt_render_ss(self._ctx, C.byref(prm), C.byref(cam), C.byref(fx), C.c_uint64(tex), float(time),
                                            int(w), int(h), int(ss), C.byref(band) if band is not None else None,
                                            C.c_void_p(out_ptr), int(layout), C.c_void_p(hdr_ptr), C.c_void_p(st.cuda_stream)))
        return out

    def resolve(self, prm: Params, fx: Effects, hdr_hi: torch.Tensor, ss: int, w: int, h: int, *, band: Optional[Band] = None,
                out=None, layout: int = OUT_FRAME, hdr_out: Optional[torch.Tensor] = None,
                stream: Optional[torch.cuda.Stream] = None) -> torch.Tensor:
        """rrt_resolve: box-filters ``hdr_hi``, the (ss*h, ss*w, 4) float32 hdr plane of a ``render`` or ``shade`` at
        ss*w x ss*h, into a w x h frame and runs the post step (bloom, vignette, exposure tonemap, store) on it;
        asynchronous.  ``hdr_out`` ((h, w, 4) float32, not overlapping ``hdr_hi``) receives the mean.  ``band``, ``out``
        and ``layout`` as in ``render``; returns the frame."""
        out, out_ptr = self._frame_out(out, layout, band, w, h)
        assert tuple(hdr_hi.shape) == (ss * h, ss * w, 4), "hdr_hi must be (ss*h, ss*w, 4)"
        hi_ptr = self._plane_ptr("hdr", hdr_hi, ss * w, ss * h)
        hdr_ptr = self._plane_ptr("hdr", hdr_out, w, h) if hdr_out is not None else None
        st = stream if stream is not None else torch.cuda.current_stream(self.device)
        self._check(self._lib.rrt_resolve(self._ctx, C.byref(prm), C.byref(fx), int(ss), int(w), int(h),
                                          C.byref(band) if band is not None else None, C.c_void_p(hi_ptr),
                                          C.c_void_p(out_ptr), int(layout), C.c_void_p(hdr_ptr), C.c_void_p(st.cuda_stream)))
        return out

    def resolve_time(self, prm: Params, fx: Effects, hdr_stack: torch.Tensor, w: int, h: int, *, band: Optional[Band] = None,
                     out=None, layout: int = OUT_FRAME, hdr_out: Optional[torch.Tensor] = None,
                     stream: Optional[torch.cuda.Stream] = None) -> torch.Tensor:
        """rrt_resolve_time: the mean of the n planes of ``hdr_stack`` ((n, h, w, 4) float32, 1 <= n <= 64, e.g. the hdr
        planes of n renders), summed from plane 0 in float32 and divided by n, then the post step (bloom, vignette, exposure
        tonemap, store) on it; asynchronous.  ``hdr_out`` ((h, w, 4) float32, not overlapping ``hdr_stack``) receives the
        mean.  ``band``, ``out`` and ``layout`` as in ``render``; returns the frame."""
        out, out_ptr = self._frame_out(out, layout, band, w, h)
        assert hdr_stack.dim() == 4 and tuple(hdr_stack.shape[1:]) == (h, w, 4), "hdr_stack must be (n, h, w, 4)"
        n = int(hdr_stack.shape[0])
        stack_ptr = self._plane_ptr("hdr", hdr_stack, w, n * h)
        hdr_ptr = self._plane_ptr("hdr", hdr_out, w, h) if hdr_out is not None else None
        st = stream if stream is not None else torch.cuda.current_stream(self.device)
        self._check(self._lib.rrt_resolve_time(self._ctx, C.byref(prm), C.byref(fx), n, int(w), int(h),
                                               C.byref(band) if band is not None else None, C.c_void_p(stack_ptr),
                                               C.c_void_p(out_ptr), int(layout), C.c_void_p(hdr_ptr), C.c_void_p(st.cuda_stream)))
        return out

    def render_mb(self, prm: Params, cam, fx: Effects, sky: Sky | int, times, w: int, h: int, *, band: Optional[Band] = None,
                  out=None, layout: int = OUT_FRAME, hdr_out: Optional[torch.Tensor] = None,
                  stream: Optional[torch.cuda.Stream] = None) -> torch.Tensor:
        """rrt_render_mb: one motion-blurred frame (or band), the mean of n = len(times) renders (1 <= n <= 64) with the
        render's own bloom / vignette / tonemap on it; asynchronous.  Sub-frame i is ``render`` at ``times[i]`` with camera
        ``cam`` (one Camera for every sub-frame) or ``cam[i]`` (a sequence of n); n = 1 is ``render``.  ``hdr_out``
        (h, w, 4) float32 receives the mean (.w = mean T).  ``band``, ``out`` (a tensor or a PeerFrame) and ``layout`` as
        in ``render``."""
        tex = sky.texture if isinstance(sky, Sky) else int(sky)
        ts = _f32_array(times)
        cams = [cam] * len(ts) if isinstance(cam, Camera) else list(cam)
        if len(cams) != len(ts):
            raise ValueError(f"render_mb: {len(cams)} cameras for {len(ts)} times")
        cam_arr = (Camera * max(len(cams), 1))(*cams)
        out, out_ptr = self._frame_out(out, layout, band, w, h)
        hdr_ptr = self._plane_ptr("hdr", hdr_out, w, h) if hdr_out is not None else None
        st = stream if stream is not None else torch.cuda.current_stream(self.device)
        self._check(self._lib.rrt_render_mb(self._ctx, C.byref(prm), cam_arr, C.byref(fx), C.c_uint64(tex), ts, len(ts),
                                            int(w), int(h), C.byref(band) if band is not None else None,
                                            C.c_void_p(out_ptr), int(layout), C.c_void_p(hdr_ptr), C.c_void_p(st.cuda_stream)))
        return out

    def capture(self, prm: Params, cam: Camera, fx: Effects, sky: Sky | int, w: int, h: int, *, band: Optional[Band] = None,
                max_bytes: int = 0, stream: Optional[torch.cuda.Stream] = None) -> Capture:
        """rrt_capture_create: trace the frame (or band) once and keep it for ``Capture.render`` at any time; synchronises.
        Needs a medium (FLAG_DISK / FLAG_DUST).  ``max_bytes``: the sample pool the trace runs in (0: the context's sizing
        rule); tiles that do not fit it are rendered by the fused code at every ``Capture.render``."""
        return Capture(self, prm, cam, fx, sky, w, h, band=band, max_bytes=max_bytes, stream=stream)

    def _frame_out(self, out, layout: int, band: Optional[Band], w: int, h: int):
        """(out, device pointer) of a uchar4 destination: a PeerFrame, a device tensor, or None (allocated here)."""
        if isinstance(out, PeerFrame):      # a frame that lives on the encoding GPU (possibly another process's)
            assert layout == OUT_FRAME and out.nbytes >= h * w * 4
            return out, out.ptr
        rows = h if layout == OUT_FRAME else self.band_rows(band, h)
        if out is None:
            out = torch.empty((rows, w, 4), dtype=torch.uint8, device=self.device)
        assert out.is_cuda and out.dtype == torch.uint8 and out.is_contiguous() and out.numel() >= rows * w * 4
        return out, out.data_ptr()

    @staticmethod
    def _plane_ptr(name: str, t: torch.Tensor, w: int, h: int) -> int:
        ch, dt = PLANE_SPECS[name]
        assert t.is_cuda and t.dtype == dt and t.is_contiguous() and t.numel() == h * w * max(ch, 1), name
        return t.data_ptr()

    @classmethod
    def _planes(cls, planes: dict, w: int, h: int) -> Planes:
        pl = Planes()
        for n, t in planes.items():
            setattr(pl, n, cls._plane_ptr(n, t, w, h))
        return pl

    def render_host(self, prm: Params, cam: Camera, fx: Effects, sky: Sky | int, time: float, w: int, h: int,
                    host_out) -> None:
        """rrt_render_host: end-to-end call, HOST destination (numpy array or pinned torch tensor)."""
        tex = sky.texture if isinstance(sky, Sky) else int(sky)
        if isinstance(host_out, torch.Tensor):
            assert not host_out.is_cuda and host_out.is_contiguous() and host_out.numel() * host_out.element_size() >= w * h * 4
            ptr = host_out.data_ptr()
        else:
            assert host_out.flags["C_CONTIGUOUS"] and host_out.nbytes >= w * h * 4
            ptr = host_out.ctypes.data
        self._check(self._lib.rrt_render_host(self._ctx, C.byref(prm), C.byref(cam), C.byref(fx), C.c_uint64(tex),
                                              float(time), int(w), int(h), C.c_void_p(ptr)))

    def render_host_async(self, prm: Params, cam: Camera, fx: Effects, sky: Sky | int, time: float, w: int, h: int,
                          host_out: torch.Tensor, slot: int = 0, stream: Optional[torch.cuda.Stream] = None) -> None:
        """rrt_render_host_async: trace + device->host copy enqueued on `stream`, no synchronisation.
        ``host_out`` must be a pinned CPU tensor; ``slot`` < HOST_SLOTS selects the context's device frame."""
        tex = sky.texture if isinstance(sky, Sky) else int(sky)
        assert (not host_out.is_cuda) and host_out.is_pinned() and host_out.is_contiguous()
        assert host_out.numel() * host_out.element_size() >= w * h * 4
        st = stream if stream is not None else torch.cuda.current_stream(self.device)
        self._check(self._lib.rrt_render_host_async(self._ctx, C.byref(prm), C.byref(cam), C.byref(fx), C.c_uint64(tex),
                                                    float(time), int(w), int(h), C.c_void_p(host_out.data_ptr()),
                                                    int(slot), C.c_void_p(st.cuda_stream)))

    def assemble_bands(self, packed: torch.Tensor, rows_per_rank: int, w: int, h: int, nranks: int, group: int,
                       frame: Optional[torch.Tensor] = None, stream: Optional[torch.cuda.Stream] = None) -> torch.Tensor:
        if frame is None:
            frame = torch.empty((h, w, 4), dtype=torch.uint8, device=self.device)
        st = stream if stream is not None else torch.cuda.current_stream(self.device)
        self._check(self._lib.rrt_assemble_bands(self._ctx, C.c_void_p(packed.data_ptr()), int(rows_per_rank), int(w),
                                                 int(h), int(nranks), int(group), C.c_void_p(frame.data_ptr()),
                                                 C.c_void_p(st.cuda_stream)))
        return frame

    def read_counters(self, reset: bool = True) -> dict:
        c = Counters()
        self._check(self._lib.rrt_read_counters(self._ctx, C.byref(c), 1 if reset else 0))
        return c.as_dict()

    def fp32_peak(self, iters: int = 4096):
        tf, ms = C.c_double(), C.c_double()
        self._check(self._lib.rrt_fp32_peak_probe(self._ctx, int(iters), C.byref(tf), C.byref(ms)))
        return tf.value, ms.value

    def set_frames_in_flight(self, n: int) -> None:
        """rrt_set_frames_in_flight: each launch takes 1/n of the resident-CTA slots (n concurrent frames)."""
        self._check(self._lib.rrt_set_frames_in_flight(self._ctx, int(n)))

    def set_pipeline(self, mode) -> None:
        """rrt_set_pipeline: "auto" (split whenever a medium is on), "fused" (one kernel) or "split"
        (trace / media / fold kernels over the sample pool); same frames either way."""
        modes = {"auto": _capi.PIPELINE_AUTO, "fused": _capi.PIPELINE_FUSED, "split": _capi.PIPELINE_SPLIT}
        self._check(self._lib.rrt_set_pipeline(self._ctx, int(modes.get(mode, mode))))

    def set_sample_pool(self, max_bytes_per_stream: int = 0, max_passes: int = 0) -> None:
        """rrt_set_sample_pool: size limit of one sample pool and the passes a frame may be cut into (0 = unchanged)."""
        self._check(self._lib.rrt_set_sample_pool(self._ctx, C.c_size_t(int(max_bytes_per_stream)), int(max_passes)))

    def kernel_launches(self) -> int:
        """rrt_kernel_launches: kernels launched so far by this context's render / assemble calls."""
        return int(self._lib.rrt_kernel_launches(self._ctx))

    def split_stats(self) -> dict:
        """rrt_split_stats: bookkeeping of the last frame the split pipeline completed (synchronises)."""
        out = (C.c_uint32 * 8)()
        self._check(self._lib.rrt_split_stats(self._ctx, out))
        return {"passes_worked": int(out[0]), "tiles_swept": int(out[1]), "tiles_split": int(out[2]),
                "passes_enqueued": int(out[3]), "tiles": int(out[4]), "pool_kislots": int(out[5])}

    def tile_log(self, log: Optional[torch.Tensor]) -> None:
        """rrt_debug_tile_log: per-tile (start ns, end ns, row<<32|col, sm<<32|max steps) into `log` ([n, 4] int64/uint64
        device tensor), or None to switch it off."""
        if log is None:
            self._check(self._lib.rrt_debug_tile_log(self._ctx, None, 0))
        else:
            assert log.is_cuda and log.is_contiguous() and log.element_size() == 8 and log.shape[-1] == 4
            self._check(self._lib.rrt_debug_tile_log(self._ctx, C.c_void_p(log.data_ptr()), C.c_size_t(log.shape[0])))

    def set_probe_contract(self, fmad: bool) -> None:
        """Rounding contract of hash31 / noise3d / fbm (the probes without a parameter block)."""
        self._check(self._lib.rrt_set_probe_contract(self._ctx, 1 if fmad else 0))

    def exact_math_selftest(self, seed: int = 1, n: int = 1 << 30):
        """(div mismatches, sqrt mismatches) of the loop's branch-free div/sqrt vs the IEEE intrinsics."""
        a, b = C.c_uint64(), C.c_uint64()
        self._check(self._lib.rrt_exact_math_selftest(self._ctx, C.c_uint64(seed), C.c_uint64(n), C.byref(a), C.byref(b)))
        return int(a.value), int(b.value)

    def exact_pow_selftest(self, seed: int = 1, n: int = 1 << 30):
        """rrt_exact_pow_selftest: (mismatches with the media code's exponents, mismatches with random exponents)."""
        a, b = C.c_uint64(), C.c_uint64()
        self._check(self._lib.rrt_exact_pow_selftest(self._ctx, C.c_uint64(seed), C.c_uint64(n), C.byref(a), C.byref(b)))
        return int(a.value), int(b.value)

    # ---- function-level probes (host numpy in / out) --------------------------------------------------
    @staticmethod
    def _f32(a):
        return np.ascontiguousarray(np.asarray(a, dtype=np.float32))

    @staticmethod
    def _p(a):
        return a.ctypes.data_as(C.c_void_p)

    def geodesic_acc(self, prm, q, v):
        q, v = self._f32(q), self._f32(v)
        out = np.empty_like(q)
        self._check(self._lib.rrt_geodesic_acc_batch(self._ctx, C.byref(prm), len(q), self._p(q), self._p(v), self._p(out)))
        return out

    def _step(self, fn, prm, p, v, h):
        p, v = self._f32(p).copy(), self._f32(v).copy()
        h = self._f32(np.broadcast_to(np.asarray(h, np.float32), (len(p),)))
        self._check(fn(self._ctx, C.byref(prm), len(p), self._p(p), self._p(v), self._p(h)))
        return p, v

    def rk4_step(self, prm, p, v, h):
        return self._step(self._lib.rrt_rk4_step_batch, prm, p, v, h)

    def euler_step(self, prm, p, v, h):
        return self._step(self._lib.rrt_euler_step_batch, prm, p, v, h)

    def redshift(self, prm, q, v):
        q, v = self._f32(q), self._f32(v)
        out = np.empty(len(q), np.float32)
        self._check(self._lib.rrt_redshift_batch(self._ctx, C.byref(prm), len(q), self._p(q), self._p(v), self._p(out)))
        return out

    def hash31(self, p):
        p = self._f32(p)
        out = np.empty(len(p), np.float32)
        self._check(self._lib.rrt_hash31_batch(self._ctx, len(p), self._p(p), self._p(out)))
        return out

    def noise3d(self, p):
        p = self._f32(p)
        out = np.empty(len(p), np.float32)
        self._check(self._lib.rrt_noise3d_batch(self._ctx, len(p), self._p(p), self._p(out)))
        return out

    def fbm(self, p, octaves: int):
        p = self._f32(p)
        out = np.empty(len(p), np.float32)
        self._check(self._lib.rrt_fbm_batch(self._ctx, len(p), self._p(p), int(octaves), self._p(out)))
        return out

    def disk_temperature(self, prm, r):
        r = self._f32(r)
        out = np.empty_like(r)
        self._check(self._lib.rrt_disk_temperature_batch(self._ctx, C.byref(prm), len(r), self._p(r), self._p(out)))
        return out

    def disk_density(self, prm, q, time):
        q = self._f32(q)
        out = np.empty(len(q), np.float32)
        self._check(self._lib.rrt_disk_density_batch(self._ctx, C.byref(prm), len(q), self._p(q), float(time), self._p(out)))
        return out

    def dust_density(self, prm, q, time):
        q = self._f32(q)
        out = np.empty(len(q), np.float32)
        self._check(self._lib.rrt_dust_density_batch(self._ctx, C.byref(prm), len(q), self._p(q), float(time), self._p(out)))
        return out

    def sky_sample(self, sky: Sky | int, tx, ty):
        tex = sky.texture if isinstance(sky, Sky) else int(sky)
        tx, ty = self._f32(tx), self._f32(ty)
        out = np.empty((len(tx), 4), np.float32)
        self._check(self._lib.rrt_sky_sample_batch(self._ctx, C.c_uint64(tex), len(tx), self._p(tx), self._p(ty), self._p(out)))
        return out


# ---- the reference's own entry point, same name and argument order (include/raymarcher.h:19) ------------
_default: dict[int, Renderer] = {}
_launch_params: Optional[Params] = None


def set_launch_params(prm: Optional[Params]) -> None:
    """Parameter block used by launch_raymarch (the reference compiles these in; default = config.h)."""
    global _launch_params
    _launch_params = prm


def launch_raymarch(d_out: torch.Tensor, w: int, h: int, time: float, cam: Camera, skyboxTex, effects: Effects) -> None:
    """Drop-in for the reference launcher: renders into the caller-owned device buffer ``d_out``
    (uchar4 per pixel, pixel (x,y) at [(h-1-y)*w + x]) on the current stream, asynchronously."""
    dev = d_out.device.index if d_out.device.index is not None else torch.cuda.current_device()
    r = _default.get(dev)
    if r is None:
        r = _default[dev] = Renderer(dev)
    prm = _launch_params if _launch_params is not None else default_params()
    r.render(prm, cam, effects, skyboxTex, time, w, h, out=d_out, layout=OUT_FRAME)
