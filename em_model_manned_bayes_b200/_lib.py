"""ctypes binding of libemb200.so (include/emb200.h).  Fails loudly when the library is missing:
there is no Python/CPU fallback for sampling."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("EMB200_LIB") or os.path.join(HERE, "libemb200.so")   # EMB200_LIB: tuning variants (build.py --variant)

EMB_MAX_VARS = 24
EMB_MAX_DYN = 8
EMB_MAX_PARENTS = 8
EMB_MAX_GATED = 16

EMB_MEM_HOST = 0
EMB_MEM_DEVICE = 1
EMB_MEM_ASYNC = 0x100
EMB_PRIOR_CONSTANT, EMB_PRIOR_DBE, EMB_PRIOR_STAY = 0, 1, 2
EMB_REJECT_NONE, EMB_REJECT_UNCOR, EMB_REJECT_BOX = 0, 1, 2

EMB_E_IO, EMB_E_PARSE, EMB_E_MODEL, EMB_E_ARG, EMB_E_CUDA, EMB_E_LIMIT, EMB_E_REJECT = -1, -2, -3, -4, -5, -6, -7


class EmbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("[emb %d] %s" % (code, msg))
        self.code = code
        self.message = msg


class ModelInfo(C.Structure):
    _fields_ = [
        ("n_initial", C.c_int32), ("n_transition", C.c_int32), ("n_dyn", C.c_int32), ("n_gated", C.c_int32),
        ("is_dynvar_depend", C.c_int32), ("n_timevarying", C.c_int32),
        ("len_N_initial", C.c_int64), ("len_N_transition", C.c_int64),
        ("r_initial", C.c_int32 * EMB_MAX_VARS),
        ("r_transition", C.c_int32 * (EMB_MAX_VARS + EMB_MAX_DYN)),
        ("order_initial", C.c_int32 * EMB_MAX_VARS),
        ("order_transition", C.c_int32 * (EMB_MAX_VARS + EMB_MAX_DYN)),
        ("temporal_map", (C.c_int32 * 2) * EMB_MAX_DYN),
        ("zero_bins", C.c_int32 * EMB_MAX_VARS),
        ("boundaries_len", C.c_int32 * EMB_MAX_VARS),
        ("timevarying_vars", C.c_int32 * EMB_MAX_VARS),
        ("resample_rates", C.c_double * EMB_MAX_VARS),
        ("bounds_initial", (C.c_double * 2) * EMB_MAX_VARS),
    ]


class Rng(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("first_sample", C.c_uint64)]


class SampleOpts(C.Structure):
    _fields_ = [
        ("start", C.c_int32 * EMB_MAX_VARS),
        ("reject_mode", C.c_int32),
        ("idx_v", C.c_int32), ("idx_dh", C.c_int32), ("idx_L", C.c_int32),
        ("box_lo", C.c_double * EMB_MAX_VARS), ("box_hi", C.c_double * EMB_MAX_VARS),
        ("is_quantize500", C.c_int32),
        ("n_layers", C.c_int32),
        ("layers", (C.c_double * 2) * 8),
        ("max_attempts", C.c_int32),
        ("mem", C.c_int32),
        ("device", C.c_int32),
        ("stream", C.c_void_p),
        ("start_per_sample", C.c_void_p),
        ("correct_dbn", C.c_int32),
    ]


class DynLimits(C.Structure):
    _fields_ = [("minVel_ft_s", C.c_double), ("maxVel_ft_s", C.c_double), ("maxTurnRate_deg_s", C.c_double),
                ("maxAltitude_ft", C.c_double), ("maxVertRate_ft_s", C.c_double)]


class TerminalModels(C.Structure):
    _fields_ = [("own_fwd", C.c_void_p * 2), ("own_bck", C.c_void_p * 2), ("int_fwd", C.c_void_p * 3),
                ("int_bck", C.c_void_p * 3)]


class TrajOut(C.Structure):
    _fields_ = [("traj", C.c_void_p), ("len", C.c_void_p)]


class ScreenOut(C.Structure):
    _fields_ = [("hmd_ft", C.c_void_p), ("vmd_ft", C.c_void_p), ("tcpa", C.c_void_p), ("enc_time_s", C.c_void_p),
                ("runway", C.c_void_p)]


class IntegrateOpts(C.Structure):
    _fields_ = [("idx_altitude", C.c_int32), ("idx_speed", C.c_int32), ("idx_acceleration", C.c_int32),
                ("idx_vertrate", C.c_int32), ("idx_turnrate", C.c_int32),
                ("ur_speed", C.c_double), ("ur_vertrate", C.c_double), ("ur_heading", C.c_double),
                ("min_speed", C.c_double), ("max_speed", C.c_double),
                ("mem", C.c_int32), ("device", C.c_int32), ("stream", C.c_void_p)]


class TrackOut(C.Structure):
    _fields_ = [
        ("bins", C.c_void_p), ("values", C.c_void_p), ("init_bins", C.c_void_p), ("init_values", C.c_void_p),
        ("attempts", C.c_void_p), ("hist_initial", C.c_void_p), ("hist_transition", C.c_void_p),
    ]


_lib = None


def lib():
    """Load libemb200.so (once).  Raises if it has not been built: `python -m em_model_manned_bayes_b200.build`."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise EmbError(EMB_E_CUDA, "libemb200.so not found at %s -- build it with "
                       "`python -m em_model_manned_bayes_b200.build` (there is no CPU fallback)" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, i32, i64, u64, u32 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64, C.c_uint32
    P = C.POINTER
    sig = {
        "emb_abi_version": (C.c_int, []),
        "emb_last_error": (C.c_char_p, []),
        "emb_launch_count": (i64, []),
        "emb_debug_force_generic": (None, [C.c_int]),
        "emb_debug_last_kernel_fast": (C.c_int, []),
        "emb_device_count": (C.c_int, []),
        "emb_host_alloc": (C.c_int, [P(vp), i64]),
        "emb_host_free": (C.c_int, [vp]),
        "emb_trim_device_memory": (C.c_int, [C.c_int]),
        "emb_async_status": (C.c_int, [C.c_int]),
        "emb_rng_word": (u32, [u64, u64, u32, u32, u32, u32, u32]),
        "emb_model_load": (C.c_int, [C.c_char_p, C.c_int, P(i32), i32, P(vp)]),
        "emb_model_from_arrays": (C.c_int, [i32, vp, vp, vp, i64, i32, vp, vp, vp, i64, vp, i32, vp, vp, vp, P(vp)]),
        "emb_model_free": (None, [vp]),
        "emb_model_get_info": (C.c_int, [vp, P(ModelInfo)]),
        "emb_model_get_labels": (i64, [vp, C.c_int, C.c_char_p, i64]),
        "emb_model_get_G": (i64, [vp, C.c_int, vp, i64]),
        "emb_model_get_N": (i64, [vp, C.c_int, vp, i64]),
        "emb_model_get_boundaries": (i64, [vp, vp, i64]),
        "emb_model_get_packed": (i64, [vp, C.c_int, vp, i64]),
        "emb_set_prior": (C.c_int, [vp, C.c_int, C.c_int, C.c_double]),
        "emb_sample_opts_init": (None, [P(SampleOpts)]),
        "emb_sample_initial": (C.c_int, [vp, P(Rng), i64, P(SampleOpts), vp, vp, vp]),
        "emb_sample_initial_f32": (C.c_int, [vp, P(Rng), i64, P(SampleOpts), vp, vp, vp]),
        "emb_sample_tracks": (C.c_int, [vp, P(Rng), i64, i32, P(SampleOpts), P(TrackOut)]),
        "emb_sample_track_events": (C.c_int, [vp, P(Rng), i64, i32, P(SampleOpts), i64, vp, vp, P(TrackOut), P(i64)]),
        "emb_sample_track_events_packed": (C.c_int, [vp, P(Rng), i64, i32, P(SampleOpts), i64, vp, vp, vp, P(TrackOut), P(i64)]),
        "emb_model_get_gated": (i64, [vp, vp, i64]),
        "emb_shard_range": (None, [i64, i32, i32, P(i64), P(i64)]),
        "emb_sample_tracks_multi": (C.c_int, [vp, P(Rng), i64, i32, P(SampleOpts), i32, vp, vp, vp]),
        "emb_allreduce_histograms": (C.c_int, [i32, vp, vp, i64]),
        "emb_nccl_available": (C.c_int, []),
        "emb_multi_last_error": (C.c_char_p, []),
        "emb_dyn_limits_named": (C.c_int, [C.c_char_p, P(DynLimits)]),
        "emb_terminal_propagate": (C.c_int, [P(TerminalModels), P(Rng), i64, vp, i64, P(i32), C.c_double, P(DynLimits),
                                             P(SampleOpts), P(TrajOut)]),
        "emb_terminal_traj_len": (i64, [i64, C.c_double]),
        "emb_terminal_screen": (C.c_int, [vp, vp, i64, C.c_double, C.c_double, C.c_double, P(SampleOpts), P(ScreenOut)]),
        "emb_tracks_integrate": (C.c_int, [vp, i64, i32, vp, vp, P(IntegrateOpts), vp, vp]),
        "emb_sample_tracks_xyz": (C.c_int, [vp, P(Rng), i64, i32, P(SampleOpts), P(IntegrateOpts), P(TrackOut), vp, vp]),
        "emb_tracks_bins_len": (i64, [vp, i64, i32]),
        "emb_tracks_values_len": (i64, [vp, i64, i32]),
        "emb_loglik_initial": (C.c_int, [vp, i64, vp, P(SampleOpts), vp, vp]),
        "emb_loglik_tracks": (C.c_int, [vp, i64, i32, vp, vp, P(SampleOpts), vp, vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)  # AttributeError if a declared symbol is missing
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


EXPORTED = [
    "emb_abi_version", "emb_last_error", "emb_launch_count", "emb_debug_force_generic", "emb_debug_last_kernel_fast", "emb_device_count", "emb_host_alloc", "emb_host_free", "emb_trim_device_memory", "emb_async_status",
    "emb_rng_word", "emb_shard_range", "emb_sample_tracks_multi", "emb_allreduce_histograms", "emb_nccl_available", "emb_multi_last_error", "emb_sample_initial_f32", "emb_sample_track_events_packed", "emb_model_get_gated", "emb_model_load", "emb_model_from_arrays", "emb_model_free", "emb_model_get_info",
    "emb_model_get_labels", "emb_model_get_G", "emb_model_get_N", "emb_model_get_boundaries",
    "emb_model_get_packed", "emb_set_prior", "emb_sample_opts_init", "emb_sample_initial", "emb_sample_tracks",
    "emb_tracks_bins_len", "emb_tracks_values_len", "emb_sample_track_events",
    "emb_dyn_limits_named", "emb_terminal_propagate", "emb_terminal_traj_len", "emb_tracks_integrate", "emb_sample_tracks_xyz",
    "emb_terminal_screen", "emb_loglik_initial", "emb_loglik_tracks",
]
TRAJ_FIELDS = ("x_nm", "y_nm", "z_ft", "heading_deg", "v_ft_s")

# numpy view of emb_event (include/emb200.h)
EVENT_DTYPE = [("dt", "<u2"), ("var", "u1"), ("bin", "u1"), ("value", "<f4")]


def check(rc):
    if rc != 0:
        raise EmbError(rc, lib().emb_last_error().decode("utf-8", "replace"))
