"""relativisticraytracer_b200 -- a B200-native (sm_100a) implementation of ONE path of
levi2234/RelativisticRayTracer: per-pixel geodesic RK4 integration, volumetric disk/dust transfer and
skybox lookup, behind the reference's own launch surface.  See DESIGN.md and INTEGRATION.md.

The package is a thin host layer over ``librrt_b200.so`` (C ABI in ``include/rrt.h``); importing it does not
need a GPU, calling any render or probe entry point does.
"""
from ._capi import (Band, Camera, Counters, Effects, Params, Planes, RrtError, FLAG_DISK, FLAG_DUST, FLAG_FMAD, CLS_CAPTURED,
                    CLS_DISK_HIT, CLS_ESCAPED, CLS_MASK, CLSF_EXHAUSTED, CLSF_TOUCHED, OUT_FRAME, OUT_PACKED, LIB_PATH,
                    default_effects, default_params, effects_off)
from .renderer import (TRACE_PLANES, CameraEffects, Capture, CameraState, PeerFrame, Renderer, Sky, camera_state_from, launch_raymarch,
                       path_clock, path_duration, path_names, path_state, set_launch_params, shutter_times)
from .skybox import decode_image, load_skybox, procedural_sky
from .sink import FrameSink, ffmpeg_command
from ._capi import SINK_RGBA, SINK_Y4M, HOST_SLOTS

__all__ = [n for n in dir() if not n.startswith("_")]
