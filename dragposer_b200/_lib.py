"""ctypes binding of the dp_engine_* C ABI (include/dp_engine.h).

There is NO CPU fallback: if `libdp_engine.so` is missing or fails to load, every
entry point raises.  Build it with `python -m dragposer_b200.build` (or
`__graft_entry__.build()`).
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
ENGINE_SO = os.path.join(HERE, "libdp_engine.so")

c_float_p = C.POINTER(C.c_float)
c_int32_p = C.POINTER(C.c_int32)


class RunParams(C.Structure):
    _fields_ = [
        ("stop_eps_pos", C.c_double),
        ("stop_eps_rot", C.c_double),
        ("min_loss_incr", C.c_double),
        ("max_iter", C.c_int32),
        ("learning_rate", C.c_float),
        ("lambda_rot", C.c_float),
        ("lambda_temporal", C.c_float),
        ("temporal_future_window", C.c_int32),
        ("joint_adjust_joint", C.c_int32),
        ("joint_adjust_slot", C.c_int32),
        ("joint_adjust_weight", C.c_float),
        ("decoder_path", C.c_int32),
        ("targets_world", C.c_int32),
        ("extension_losses", C.c_int32),
        ("floor_level", C.c_float),
    ]


class ClipSettings(C.Structure):
    _fields_ = [
        ("stop_eps_pos", C.c_double),
        ("stop_eps_rot", C.c_double),
        ("min_loss_incr", C.c_double),
        ("max_iter", C.c_int32),
        ("learning_rate", C.c_float),
        ("lambda_rot", C.c_float),
        ("lambda_temporal", C.c_float),
        ("joint_adjust_joint", C.c_int32),
        ("joint_adjust_slot", C.c_int32),
        ("joint_adjust_weight", C.c_float),
    ]


MAX_CLIP_SETTINGS = 32  # DP_MAX_CLIP_SETTINGS


class EncoderModelC(C.Structure):
    _fields_ = [(n, c_float_p) for n in ("A0", "b0", "A1", "b1", "A2", "b2", "mu_w", "mu_b", "logvar_w", "logvar_b")]


class PoseModelC(C.Structure):
    _fields_ = [(n, c_float_p) for n in ("A0", "b0", "A1", "b1", "A2", "b2", "mean_q", "std_q", "mean_d", "std_d")] + [
        ("parents", c_int32_p),
        ("offsets", c_float_p),
    ]


# every symbol include/dp_engine.h declares: name -> (restype, argtypes)
_VP = C.c_void_p
SIGNATURES = {
    "dp_engine_create": (C.c_int, [C.POINTER(_VP), C.c_int, C.c_int]),
    "dp_engine_destroy": (C.c_int, [_VP]),
    "dp_engine_last_error": (C.c_char_p, []),
    "dp_engine_version": (C.c_int, []),
    "dp_engine_set_pose_model": (C.c_int, [_VP, C.POINTER(PoseModelC)]),
    "dp_engine_temporal_blob_floats": (C.c_size_t, []),
    "dp_engine_set_temporal_model": (C.c_int, [_VP, _VP, C.c_size_t, _VP, _VP]),
    "dp_engine_init_clips": (C.c_int, [_VP, C.c_int, _VP, _VP, _VP, _VP]),
    "dp_engine_set_global_pos": (C.c_int, [_VP, C.c_int, C.c_int, _VP]),
    "dp_engine_n_clips": (C.c_int, [_VP]),
    "dp_engine_run_frame_device": (C.c_int, [_VP, C.POINTER(RunParams), _VP, _VP, _VP, C.c_int, _VP, _VP, C.c_int, _VP, _VP, _VP]),
    "dp_engine_run_frame_host": (C.c_int, [_VP, C.POINTER(RunParams), _VP, _VP, _VP, C.c_int, _VP, _VP, C.c_int, _VP, _VP]),
    "dp_engine_run_frames_host": (C.c_int, [_VP, C.POINTER(RunParams), C.c_int, _VP, _VP, _VP, C.c_int, _VP, _VP, C.c_int, _VP, _VP]),
    "dp_engine_run_frames_device": (C.c_int, [_VP, C.POINTER(RunParams), C.c_int, _VP, _VP, _VP, C.c_int, _VP, _VP, C.c_int, _VP, _VP, _VP]),
    "dp_engine_get_frame_stats": (C.c_int, [_VP, _VP, _VP]),
    "dp_engine_enable_trace": (C.c_int, [_VP, C.c_int]),
    "dp_engine_get_trace": (C.c_int, [_VP, _VP, C.c_int]),
    "dp_engine_eval_gradient": (C.c_int, [_VP, C.c_int, _VP, _VP, _VP, _VP, _VP, _VP, C.c_int, _VP, _VP, C.c_int, C.c_float, C.c_float, C.c_int, _VP, _VP, _VP, C.c_int, C.c_float, _VP]),
    "dp_engine_get_state": (C.c_int, [_VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, C.POINTER(C.c_int)]),
    "dp_engine_set_ring_buffers": (C.c_int, [_VP, _VP, _VP, _VP]),
    "dp_engine_predict_targets": (C.c_int, [_VP, C.c_int, _VP]),
    "dp_engine_launch_count": (C.c_longlong, [_VP]),
    "dp_engine_last_decoder_path": (C.c_int, [_VP]),
    "dp_engine_set_predictor_path": (C.c_int, [_VP, C.c_int]),
    "dp_engine_set_profiling": (C.c_int, [_VP, C.c_int]),
    "dp_engine_pose_error_host": (C.c_int, [_VP, C.c_int, _VP, _VP, _VP]),
    "dp_engine_set_encoder_model": (C.c_int, [_VP, C.POINTER(EncoderModelC)]),
    "dp_engine_encode_host": (C.c_int, [_VP, C.c_int, _VP, _VP, _VP]),
    "dp_engine_get_phase_cycles": (C.c_int, [_VP, C.POINTER(C.c_ulonglong)]),
    "dp_engine_get_timeline": (C.c_int, [_VP, C.POINTER(C.c_ulonglong)]),
    "dp_engine_get_profile": (C.c_int, [_VP, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_longlong)]),
    "dp_engine_restart_clips": (C.c_int, [_VP, C.c_int, _VP, _VP, _VP, _VP, _VP, _VP]),
    "dp_engine_get_clip_index": (C.c_int, [_VP, C.c_int, _VP]),
    "dp_engine_frames_to_boundary": (C.c_int, [_VP, C.c_int]),
    "dp_engine_set_clip_settings": (C.c_int, [_VP, C.c_int, _VP, _VP]),
}

_lib = None


class EngineError(RuntimeError):
    pass


def load():
    """Load libdp_engine.so (no GPU needed to load it); raises if it was not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(ENGINE_SO):
            raise EngineError(
                f"{ENGINE_SO} is missing: build the CUDA engine first (python -m dragposer_b200.build). "
                "There is no CPU fallback."
            )
        lib = C.CDLL(ENGINE_SO)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def check(rc):
    if rc != 0:
        raise EngineError(f"dp_engine error {rc}: {load().dp_engine_last_error().decode()}")
