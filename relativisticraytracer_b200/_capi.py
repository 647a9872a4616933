"""ctypes binding of the C ABI in include/rrt.h (librrt_b200.so).

There is deliberately no fallback: if the shared library is missing or was not built, importing a
compute entry point raises, and every compute call needs a B200 (the library itself refuses other
devices).  Nothing here imports ``oracle``.
"""
from __future__ import annotations

import ctypes as C
import os

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RRT_B200_LIB") or os.path.join(PKG_DIR, "librrt_b200.so")   # env: A/B builds only

OK, ERR_BAD_ARG, ERR_CUDA, ERR_NO_DEVICE, ERR_NOMEM, ERR_IO, ERR_UNSUPPORTED = 0, -1, -2, -3, -4, -5, -6
SINK_RGBA, SINK_Y4M = 0, 1
FLAG_DISK, FLAG_DUST, FLAG_FMAD = 1, 2, 4
CLS_CAPTURED, CLS_DISK_HIT, CLS_ESCAPED, CLS_MASK = 0, 1, 2, 3
CLSF_EXHAUSTED, CLSF_TOUCHED = 4, 8
OUT_FRAME, OUT_PACKED = 0, 1
HOST_SLOTS = 4   # RRT_HOST_SLOTS
PIPELINE_AUTO, PIPELINE_FUSED, PIPELINE_SPLIT = 0, 1, 2


class RrtError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"librrt_b200 error {code}: {msg}")
        self.code = code


class Params(C.Structure):
    """rrt_params: the reference's include/config.h macros as run-time fields."""
    _fields_ = [(n, C.c_float) for n in (
        "spin_a", "event_horizon", "isco_radius", "disk_out", "disk_h", "disk_luminosity", "disk_opacity",
        "exposure", "cloud_h", "cloud_out", "cloud_opacity", "cloud_luminosity", "step_size", "disk_temp_ref")] + [
        ("max_steps", C.c_int32), ("flags", C.c_uint32)]


class Camera(C.Structure):
    """rrt_camera == reference struct CameraState (include/raymarcher.h:11-16)."""
    _fields_ = [("pos", C.c_float * 3), ("forward", C.c_float * 3), ("right", C.c_float * 3), ("up", C.c_float * 3)]


class Effects(C.Structure):
    """rrt_effects == reference struct CameraEffects (camera_settings.h:4-17) with int32 booleans."""
    _fields_ = [("use_bloom", C.c_int32), ("bloom_threshold", C.c_float), ("bloom_intensity", C.c_float),
                ("use_vignette", C.c_int32), ("vignette_intensity", C.c_float),
                ("use_ca", C.c_int32), ("ca_amount", C.c_float),
                ("use_lens", C.c_int32), ("distortion_amount", C.c_float)]


class Band(C.Structure):
    _fields_ = [("rank", C.c_int32), ("nranks", C.c_int32), ("group", C.c_int32)]


class Planes(C.Structure):
    _fields_ = [("hdr", C.c_void_p), ("dir", C.c_void_p), ("emis", C.c_void_p), ("pos", C.c_void_p),
                ("vel", C.c_void_p), ("cls", C.c_void_p), ("steps", C.c_void_p)]


class Counters(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("rk4_steps", "disk_evals", "dust_evals", "dense_samples",
                                          "n_captured", "n_escaped", "n_exhausted", "n_touched")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


# every symbol include/rrt.h declares (tests/test_capi_symbols.py checks the header against this list)
SYMBOLS = [
    "rrt_abi_version", "rrt_build_info", "rrt_context_create", "rrt_context_destroy", "rrt_last_error",
    "rrt_default_params", "rrt_default_effects", "rrt_sky_create", "rrt_sky_texture", "rrt_sky_destroy",
    "rrt_render", "rrt_shade", "rrt_resolve", "rrt_render_ss", "rrt_capture_create", "rrt_capture_render", "rrt_capture_info",
    "rrt_capture_destroy", "rrt_resolve_time", "rrt_render_mb", "rrt_capture_render_mb", "rrt_shutter_times", "rrt_render_host", "rrt_render_host_async", "rrt_band_rows", "rrt_assemble_bands", "rrt_read_counters",
    "rrt_geodesic_acc_batch", "rrt_rk4_step_batch", "rrt_euler_step_batch", "rrt_redshift_batch",
    "rrt_hash31_batch", "rrt_noise3d_batch", "rrt_fbm_batch", "rrt_disk_temperature_batch",
    "rrt_disk_density_batch", "rrt_dust_density_batch", "rrt_sky_sample_batch", "rrt_fp32_peak_probe",
    "rrt_camera_from", "rrt_path_count", "rrt_path_name", "rrt_path_num_keys", "rrt_path_duration",
    "rrt_path_state", "rrt_path_clock", "rrt_exact_math_selftest", "rrt_exact_pow_selftest",
    "rrt_image_load", "rrt_image_decode", "rrt_image_free", "rrt_image_last_error", "rrt_sky_load",
    "rrt_peer_frame_create", "rrt_peer_frame_open", "rrt_peer_frame_read", "rrt_peer_frame_close",
    "rrt_debug_tile_log", "rrt_set_probe_contract", "rrt_set_frames_in_flight", "rrt_set_pipeline", "rrt_set_sample_pool", "rrt_split_stats", "rrt_kernel_launches", "rrt_sink_open", "rrt_sink_write", "rrt_sink_frames", "rrt_sink_close", "rrt_sink_ffmpeg_command",
]

_lib = None


def load() -> C.CDLL:
    """Load librrt_b200.so (built by ``__graft_entry__.build()`` / ``make -C csrc``).  Raises if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FileNotFoundError(
            f"{LIB_PATH} is not built; run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU or PyTorch fallback for the render path)")
    lib = C.CDLL(LIB_PATH)
    P, vp, ci, cf = C.POINTER, C.c_void_p, C.c_int, C.c_float
    lib.rrt_abi_version.restype = ci
    lib.rrt_build_info.restype = C.c_char_p
    lib.rrt_context_create.argtypes = [ci, P(vp)]
    lib.rrt_context_destroy.argtypes = [vp]
    lib.rrt_context_destroy.restype = None
    lib.rrt_last_error.argtypes = [vp]
    lib.rrt_last_error.restype = C.c_char_p
    lib.rrt_default_params.argtypes = [P(Params)]
    lib.rrt_default_params.restype = None
    lib.rrt_default_effects.argtypes = [P(Effects)]
    lib.rrt_default_effects.restype = None
    lib.rrt_sky_create.argtypes = [vp, vp, ci, ci, P(vp)]
    lib.rrt_sky_texture.argtypes = [vp]
    lib.rrt_sky_texture.restype = C.c_uint64
    lib.rrt_sky_destroy.argtypes = [vp]
    lib.rrt_sky_destroy.restype = None
    lib.rrt_render.argtypes = [vp, P(Params), P(Camera), P(Effects), C.c_uint64, cf, ci, ci, P(Band), vp, ci,
                               P(Planes), vp]
    lib.rrt_shade.argtypes = [vp, P(Params), P(Effects), C.c_uint64, ci, ci, P(Band), P(Planes), vp, ci, vp, vp]
    lib.rrt_resolve.argtypes = [vp, P(Params), P(Effects), ci, ci, ci, P(Band), vp, vp, ci, vp, vp]
    lib.rrt_render_ss.argtypes = [vp, P(Params), P(Camera), P(Effects), C.c_uint64, cf, ci, ci, ci, P(Band), vp, ci, vp,
                                  vp]
    lib.rrt_capture_create.argtypes = [vp, P(Params), P(Camera), P(Effects), C.c_uint64, ci, ci, P(Band), C.c_size_t, vp, P(vp)]
    lib.rrt_capture_render.argtypes = [vp, P(Params), P(Effects), C.c_uint64, cf, vp, ci, vp, vp]
    lib.rrt_capture_info.argtypes = [vp, P(C.c_uint64)]
    lib.rrt_capture_destroy.argtypes = [vp]
    lib.rrt_capture_destroy.restype = None
    lib.rrt_resolve_time.argtypes = [vp, P(Params), P(Effects), ci, ci, ci, P(Band), vp, vp, ci, vp, vp]
    lib.rrt_render_mb.argtypes = [vp, P(Params), P(Camera), P(Effects), C.c_uint64, P(cf), ci, ci, ci, P(Band), vp, ci, vp, vp]
    lib.rrt_capture_render_mb.argtypes = [vp, P(Params), P(Effects), C.c_uint64, P(cf), ci, vp, ci, vp, vp]
    lib.rrt_shutter_times.argtypes = [cf, cf, cf, ci, P(cf)]
    lib.rrt_render_host.argtypes = [vp, P(Params), P(Camera), P(Effects), C.c_uint64, cf, ci, ci, vp]
    lib.rrt_render_host_async.argtypes = [vp, P(Params), P(Camera), P(Effects), C.c_uint64, cf, ci, ci, vp, ci, vp]
    lib.rrt_band_rows.argtypes = [P(Band), ci]
    lib.rrt_assemble_bands.argtypes = [vp, vp, ci, ci, ci, ci, ci, vp, vp]
    lib.rrt_read_counters.argtypes = [vp, P(Counters), ci]
    lib.rrt_image_load.argtypes = [C.c_char_p, P(P(C.c_uint8)), P(ci), P(ci)]
    lib.rrt_image_decode.argtypes = [vp, C.c_size_t, P(P(C.c_uint8)), P(ci), P(ci)]
    lib.rrt_image_free.argtypes = [P(C.c_uint8)]
    lib.rrt_image_free.restype = None
    lib.rrt_image_last_error.restype = C.c_char_p
    lib.rrt_sky_load.argtypes = [vp, C.c_char_p, P(vp)]
    lib.rrt_peer_frame_create.argtypes = [vp, C.c_size_t, P(vp), vp]
    lib.rrt_peer_frame_open.argtypes = [vp, vp, P(vp)]
    lib.rrt_peer_frame_read.argtypes = [vp, vp, C.c_size_t, vp, vp]
    lib.rrt_peer_frame_close.argtypes = [vp, vp, ci]
    lib.rrt_geodesic_acc_batch.argtypes = [vp, P(Params), ci, vp, vp, vp]
    lib.rrt_rk4_step_batch.argtypes = [vp, P(Params), ci, vp, vp, vp]
    lib.rrt_euler_step_batch.argtypes = [vp, P(Params), ci, vp, vp, vp]
    lib.rrt_redshift_batch.argtypes = [vp, P(Params), ci, vp, vp, vp]
    lib.rrt_hash31_batch.argtypes = [vp, ci, vp, vp]
    lib.rrt_noise3d_batch.argtypes = [vp, ci, vp, vp]
    lib.rrt_fbm_batch.argtypes = [vp, ci, vp, ci, vp]
    lib.rrt_disk_temperature_batch.argtypes = [vp, P(Params), ci, vp, vp]
    lib.rrt_disk_density_batch.argtypes = [vp, P(Params), ci, vp, cf, vp]
    lib.rrt_dust_density_batch.argtypes = [vp, P(Params), ci, vp, cf, vp]
    lib.rrt_sky_sample_batch.argtypes = [vp, C.c_uint64, ci, vp, vp, vp]
    lib.rrt_fp32_peak_probe.argtypes = [vp, ci, P(C.c_double), P(C.c_double)]
    lib.rrt_exact_math_selftest.argtypes = [vp, C.c_uint64, C.c_uint64, P(C.c_uint64), P(C.c_uint64)]
    lib.rrt_exact_pow_selftest.argtypes = [vp, C.c_uint64, C.c_uint64, P(C.c_uint64), P(C.c_uint64)]
    lib.rrt_camera_from.argtypes = [P(C.c_float * 3), cf, cf, P(Camera)]
    lib.rrt_camera_from.restype = None
    lib.rrt_path_count.restype = ci
    lib.rrt_path_name.argtypes = [ci]
    lib.rrt_path_name.restype = C.c_char_p
    lib.rrt_path_num_keys.argtypes = [ci]
    lib.rrt_path_duration.argtypes = [ci]
    lib.rrt_path_duration.restype = cf
    lib.rrt_path_state.argtypes = [ci, cf, P(Camera), vp]
    lib.rrt_path_clock.argtypes = [ci, cf]
    lib.rrt_path_clock.restype = cf
    lib.rrt_debug_tile_log.argtypes = [vp, vp, C.c_size_t]
    lib.rrt_set_probe_contract.argtypes = [vp, ci]
    lib.rrt_set_frames_in_flight.argtypes = [vp, ci]
    lib.rrt_set_pipeline.argtypes = [vp, ci]
    lib.rrt_set_sample_pool.argtypes = [vp, C.c_size_t, ci]
    lib.rrt_split_stats.argtypes = [vp, P(C.c_uint32)]
    lib.rrt_kernel_launches.argtypes = [vp]
    lib.rrt_kernel_launches.restype = C.c_uint64
    lib.rrt_sink_open.argtypes = [C.c_char_p, ci, ci, ci, ci, P(vp)]
    lib.rrt_sink_write.argtypes = [vp, vp]
    lib.rrt_sink_frames.argtypes = [vp]
    lib.rrt_sink_close.argtypes = [vp]
    lib.rrt_sink_ffmpeg_command.argtypes = [ci, ci, ci, C.c_char_p, C.c_char_p, ci]
    for name in SYMBOLS:
        getattr(lib, name)  # AttributeError here = header and library disagree
    _lib = lib
    return lib


def default_params(**over) -> Params:
    p = Params()
    load().rrt_default_params(C.byref(p))
    for k, v in over.items():
        setattr(p, k, v)
    return p


def default_effects(**over) -> Effects:
    e = Effects()
    load().rrt_default_effects(C.byref(e))
    for k, v in over.items():
        setattr(e, k, v)
    return e


def effects_off() -> Effects:
    return default_effects(use_bloom=0, use_vignette=0, use_ca=0, use_lens=0)
