"""ctypes binding of the C ABI in include/same_engine.h (sameold_b200/_build/libsame_b200.so).

The library is the product: if it cannot be built/loaded this module raises — there is no Python or CPU fallback.
"""
import ctypes as C
import os

from . import build as _build


class SameConfig(C.Structure):
    """== include/same_engine.h:same_config == SameReceiverBuilder + EqualizerBuilder (builder.rs:14-29, 360-365)."""

    _fields_ = [
        ("input_rate", C.c_uint32),
        ("dc_blocker_len", C.c_float),
        ("agc_bandwidth", C.c_float),
        ("agc_gain_min", C.c_float),
        ("agc_gain_max", C.c_float),
        ("timing_bw_unlocked", C.c_float),
        ("timing_bw_locked", C.c_float),
        ("timing_max_deviation", C.c_float),
        ("squelch_power_open", C.c_float),
        ("squelch_power_close", C.c_float),
        ("squelch_bandwidth", C.c_float),
        ("preamble_max_errors", C.c_uint32),
        ("eq_enabled", C.c_uint32),
        ("eq_nff", C.c_uint32),
        ("eq_nfb", C.c_uint32),
        ("eq_relaxation", C.c_float),
        ("eq_regularization", C.c_float),
        ("frame_prefix_max_errors", C.c_uint32),
        ("frame_max_invalid_bytes", C.c_uint32),
    ]


class SameEvent(C.Structure):
    _fields_ = [
        ("stream", C.c_uint32), ("seq", C.c_uint32),
        ("input_sample_counter", C.c_uint64), ("symbol_count", C.c_uint64),
        ("kind", C.c_uint32), ("err", C.c_uint32),
        ("data_offset", C.c_uint32), ("data_len", C.c_uint32),
        ("parity_errors", C.c_uint16), ("voting_bytes", C.c_uint16), ("flags", C.c_uint32),
    ]


class SameSoftSymbol(C.Structure):
    _fields_ = [("input_sample_counter", C.c_uint64), ("zero", C.c_float), ("sym", C.c_float)]


class SameDerived(C.Structure):
    _fields_ = [(n, C.c_float) for n in (
        "sps", "agc_bw", "agc_gain0", "samples_per_ted", "period_min", "period_max",
        "alpha_unlocked", "beta_unlocked", "alpha_locked", "beta_locked")] + [("dc_len", C.c_uint32), ("ntaps", C.c_uint32)]


# every symbol include/same_engine.h declares: (restype, argtypes)
_P = C.c_void_p
API = {
    "same_abi_version": (C.c_uint32, []),
    "same_config_default": (None, [C.POINTER(SameConfig), C.c_uint32]),
    "same_config_samedec": (None, [C.POINTER(SameConfig), C.c_uint32]),
    "same_config_sanitize": (None, [C.POINTER(SameConfig)]),
    "same_engine_create": (C.c_int, [C.POINTER(SameConfig), C.c_int, C.c_uint32, C.POINTER(_P)]),
    "same_engine_destroy": (None, [_P]),
    "same_last_error": (C.c_char_p, []),
    "same_engine_last_error": (C.c_char_p, [_P]),
    "same_engine_num_streams": (C.c_uint32, [_P]),
    "same_engine_input_rate": (C.c_uint32, [_P]),
    "same_engine_input_sample_counters": (C.c_int, [_P, _P]),
    "same_engine_reset": (C.c_int, [_P, _P, C.c_uint32]),
    "same_engine_snapshot": (C.c_int, [_P, C.POINTER(_P)]),
    "same_engine_restore": (C.c_int, [_P, _P]),
    "same_snapshot_free": (None, [_P]),
    "same_engine_state_bytes": (C.c_size_t, [_P, C.c_uint32]),
    "same_engine_export_streams": (C.c_int, [_P, _P, C.c_uint32, _P, C.c_size_t, C.POINTER(C.c_size_t)]),
    "same_engine_import_streams": (C.c_int, [_P, _P, C.c_uint32, _P, C.c_size_t]),
    "same_state_info": (C.c_int, [_P, C.c_size_t, C.POINTER(SameConfig), C.POINTER(C.c_uint32)]),
    "same_engine_set_event_capacity": (C.c_int, [_P, C.c_size_t, C.c_size_t]),
    "same_engine_submit_s16": (C.c_int, [_P, _P, C.c_uint64, _P, _P]),
    "same_engine_submit_s16_2d": (C.c_int, [_P, _P, C.c_uint64, C.c_uint64, C.c_uint32]),
    "same_engine_submit_s16_device": (C.c_int, [_P, _P, C.c_uint64, _P, _P]),
    "same_engine_submit_f32": (C.c_int, [_P, _P, C.c_uint64, _P, _P]),
    "same_engine_submit_f32_device": (C.c_int, [_P, _P, C.c_uint64, _P, _P]),
    "same_engine_submit_zeros": (C.c_int, [_P, _P]),
    "same_engine_lost_events": (C.c_int, [_P, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "same_engine_sync": (C.c_int, [_P]),
    "same_engine_pending": (C.c_int, [_P, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "same_engine_drain_events": (C.c_int, [_P, _P, C.c_size_t, C.POINTER(C.c_size_t), _P, C.c_size_t, C.POINTER(C.c_size_t)]),
    "same_engine_enable_soft_trace": (C.c_int, [_P, C.c_uint32]),
    "same_engine_read_soft_trace": (C.c_int, [_P, C.c_uint32, _P, C.c_size_t, C.POINTER(C.c_size_t)]),
    "same_engine_set_option": (C.c_int, [_P, C.c_char_p, C.c_int]),
    "same_engine_get_option": (C.c_int, [_P, C.c_char_p, C.POINTER(C.c_int)]),
    "same_engine_frontend_probe": (C.c_int, [_P, _P, C.c_uint64, _P, _P, C.c_int, C.POINTER(C.c_float)]),
    "same_engine_last_timing": (C.c_int, [_P, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "same_engine_launch_count": (C.c_uint64, [_P]),
    "same_engine_timer_start": (C.c_int, [_P]),
    "same_engine_timer_stop": (C.c_int, [_P, C.POINTER(C.c_float)]),
    "same_engine_cuda_stream": (_P, [_P]),
    "same_host_alloc": (_P, [C.c_size_t]),
    "same_host_free": (None, [_P]),
    "same_h2d_probe": (C.c_int, [C.c_int, _P, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, C.POINTER(C.c_float)]),
    "same_engine_get_derived": (C.c_int, [_P, C.POINTER(SameDerived), _P, _P, C.c_size_t]),
    # several devices in one process
    "same_multi_create": (C.c_int, [C.POINTER(SameConfig), C.POINTER(C.c_int), C.c_uint32, C.c_uint32, C.POINTER(_P)]),
    "same_multi_destroy": (None, [_P]),
    "same_multi_last_error": (C.c_char_p, [_P]),
    "same_multi_num_shards": (C.c_uint32, [_P]),
    "same_multi_num_streams": (C.c_uint32, [_P]),
    "same_multi_shard_info": (C.c_int, [_P, C.c_uint32, C.POINTER(C.c_int), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "same_multi_engine": (_P, [_P, C.c_uint32]),
    "same_multi_submit_s16": (C.c_int, [_P, _P, C.c_uint64, _P, _P]),
    "same_multi_submit_f32": (C.c_int, [_P, _P, C.c_uint64, _P, _P]),
    "same_multi_submit_s16_2d": (C.c_int, [_P, _P, C.c_uint64, C.c_uint64, C.c_uint32]),
    "same_multi_submit_zeros": (C.c_int, [_P, _P]),
    "same_multi_sync": (C.c_int, [_P]),
    "same_multi_reset": (C.c_int, [_P]),
    "same_multi_input_sample_counters": (C.c_int, [_P, _P]),
    "same_multi_pending": (C.c_int, [_P, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "same_multi_drain_events": (C.c_int, [_P, _P, C.c_size_t, C.POINTER(C.c_size_t), _P, C.c_size_t, C.POINTER(C.c_size_t)]),
    "same_multi_state_bytes": (C.c_size_t, [_P, C.c_uint32]),
    "same_multi_export_streams": (C.c_int, [_P, _P, C.c_uint32, _P, C.c_size_t, C.POINTER(C.c_size_t)]),
    "same_multi_import_streams": (C.c_int, [_P, _P, C.c_uint32, _P, C.c_size_t]),
    # synthetic corpus generator (bench / test tooling, same library)
    "same_synth_generate": (C.c_int, [C.c_int, _P, C.c_uint32, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, _P, _P, C.c_uint32,
                                      _P, C.c_uint64, _P, _P, C.c_float, C.c_float, _P]),
}

_LIB = None


def lib_path():
    return _build.LIB


def load():
    """Load (building first if the sources are newer) the native library; raises if that is impossible."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = _build.build_native() if _build.needs_build() else _build.LIB
    alt = os.environ.get("SAME_B200_LIB")   # diagnostic: A/B-time another in-tree build of the same ABI
    if alt:
        path = alt
    try:
        lib = C.CDLL(path)
    except OSError as e:  # pragma: no cover
        raise ImportError(f"cannot load {path}: {e}. The CUDA engine is mandatory; there is no CPU fallback.") from e
    for name, (res, args) in API.items():
        fn = getattr(lib, name)  # AttributeError here = header and library out of sync: fail loudly
        fn.restype = res
        fn.argtypes = args
    _LIB = lib
    return lib
