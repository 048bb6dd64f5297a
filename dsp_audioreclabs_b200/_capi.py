"""ctypes binding of libdspfront.so (include/dspfront.h).

This is the stub a maintainer of the reference would add (INTEGRATION.md): plain
pointers and sizes, no torch types.  Importing this module without the built
CUDA library raises -- there is no CPU implementation to fall back to.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DSP_LIB_PATH") or os.path.join(_HERE, "libdspfront.so")   # override: tuning builds only

DSP_S16, DSP_U8, DSP_F32, DSP_F64 = 0, 1, 2, 3
WINDOW_IDS = {"rectangular": 0, "hamming": 1, "hanning": 2}
DSP_UTT_EMPTY, DSP_UTT_NO_FRAMES, DSP_UTT_EXACT = 1, 2, 0x100
DSP_ERR_INVALID, DSP_ERR_CUDA, DSP_ERR_NO_DEVICE, DSP_ERR_UNSUPPORTED, DSP_ERR_NOMEM = -1, -2, -3, -4, -5


class DspError(RuntimeError):
    """CUDA / environment failure (not a caller error)."""


class FrontendParams(C.Structure):
    _fields_ = [
        ("frame_length", C.c_int32), ("frame_shift", C.c_int32), ("window", C.c_int32),
        ("do_endpoint_detection", C.c_int32),
        ("energy_high_ratio", C.c_double), ("energy_low_ratio", C.c_double),
        ("zcr_threshold_ratio", C.c_double),
        ("channels", C.c_int32), ("force_exact", C.c_int32), ("aligned16", C.c_int32),
    ]


class FrontendOutputs(C.Structure):
    _fields_ = [
        ("start", C.c_void_p), ("end", C.c_void_p), ("n_epd_frames", C.c_void_p),
        ("n_frames", C.c_void_p), ("status", C.c_void_p),
        ("energy", C.c_void_p), ("magnitude", C.c_void_p), ("zcr", C.c_void_p),
        ("stats", C.c_void_p), ("epd_energy", C.c_void_p), ("epd_zcr", C.c_void_p),
        ("energy_f64", C.c_void_p), ("magnitude_f64", C.c_void_p), ("zcr_f64", C.c_void_p),
        ("stats_f64", C.c_void_p), ("epd_zcr_f64", C.c_void_p), ("frames_f64", C.c_void_p),
    ]


class MfccParams(C.Structure):
    _fields_ = [
        ("frame_length", C.c_int32), ("frame_shift", C.c_int32), ("n_fft", C.c_int32), ("n_mels", C.c_int32),
        ("n_ceps", C.c_int32), ("window", C.c_int32), ("pre_emphasis", C.c_double), ("log_floor", C.c_double),
    ]


class WavInfo(C.Structure):
    _fields_ = [
        ("status", C.c_int32), ("channels", C.c_int32), ("sample_width", C.c_int32), ("sample_rate", C.c_int32),
        ("n_frames", C.c_int64), ("data_offset", C.c_int64), ("data_bytes", C.c_int64),
    ]


# every symbol include/dspfront.h declares: name -> (restype, argtypes)
_P = C.c_void_p
_I64 = C.c_int64
_I32 = C.c_int32
SIGNATURES = {
    "dsp_abi_version": (C.c_int, []),
    "dsp_last_error": (C.c_char_p, []),
    "dsp_create": (C.c_int, [C.c_int, C.POINTER(_P)]),
    "dsp_destroy": (C.c_int, [_P]),
    "dsp_set_stream": (C.c_int, [_P, _P]),
    "dsp_use_own_stream": (C.c_int, [_P]),
    "dsp_set_tuning": (C.c_int, [_P, C.c_char_p, C.c_int]),
    "dsp_sync": (C.c_int, [_P]),
    "dsp_launch_count": (_I64, [_P]),
    "dsp_device_sm_count": (C.c_int, [_P]),
    "dsp_frontend_plan": (C.c_int, [_P, _P, _I64, C.POINTER(FrontendParams), _P, _P, C.POINTER(_I64)]),
    "dsp_window": (C.c_int, [C.c_int, _I32, _P]),
    "dsp_frontend_batch_device": (C.c_int, [_P, _P, C.c_int, _P, _P, _P, _P, _I64, _I64,
                                            C.POINTER(FrontendParams), C.POINTER(FrontendOutputs)]),
    "dsp_frontend_batch_host": (C.c_int, [_P, _P, C.c_int, _P, _P, _I64, C.POINTER(FrontendParams),
                                          C.POINTER(FrontendOutputs)]),
    "dsp_preprocess_host": (C.c_int, [_P, _P, _I64, C.c_int, _P]),
    "dsp_endpoint_detection_host": (C.c_int, [_P, _P, _I64, C.POINTER(FrontendParams), C.POINTER(_I32),
                                              C.POINTER(_I32), C.POINTER(_I32), _P, _P]),
    "dsp_frame_count": (_I64, [_I64, _I32, _I32]),
    "dsp_frame_signal_host": (C.c_int, [_P, _P, _I64, _I32, _I32, C.c_int, _P]),
    "dsp_frame_features_host": (C.c_int, [_P, _P, _I64, _I32, _P, _P, _P, _P]),
    "dsp_sequence_stats_host": (C.c_int, [_P, _P, _I64, _P]),
    "dsp_zscore_host": (C.c_int, [_P, _P, _I64, _I32, C.c_int, _P, _P, _P]),
    "dsp_zscore_device": (C.c_int, [_P, _P, _I64, _I32, C.c_int, _P, _P, _P]),
    "dsp_zscore_apply_f32_device": (C.c_int, [_P, _P, _I64, _I32, _P, _P, _P]),
    "dsp_knn_fit_host": (C.c_int, [_P, _P, _P, _I64, _I32, _I32, _I64, C.POINTER(_P)]),
    "dsp_knn_fit_device": (C.c_int, [_P, _P, _P, _I64, _I32, _I32, _I64, C.POINTER(_P)]),
    "dsp_knn_free": (C.c_int, [_P]),
    "dsp_knn_topk_host": (C.c_int, [_P, _P, _I64, _P, _P, _P]),
    "dsp_knn_topk_device": (C.c_int, [_P, _P, _I64, _P, _P, _P]),
    "dsp_knn_topk_bounded_device": (C.c_int, [_P, _P, _I64, _P, _P, _P, _P]),
    "dsp_knn_predict_host": (C.c_int, [_P, _P, _I64, _P]),
    "dsp_knn_predict_device": (C.c_int, [_P, _P, _I64, _P]),
    "dsp_knn_last_stats": (C.c_int, [_P, C.POINTER(_I64), C.POINTER(_I32)]),
    "dsp_knn_merge_vote_device": (C.c_int, [_P, _P, _P, _P, _I32, _I64, _I32, _P, _P, _P]),
    "dsp_mfcc_batch_host": (C.c_int, [_P, _P, _P, _P, _P, _P, _I64, C.POINTER(MfccParams), _P, _P, _P, _P, _P]),
    "dsp_dtw_topk_host": (C.c_int, [_P, _P, _P, _I64, _P, _P, _P, _I64, _I32, _I32, _I64, _P, _P, _P, _P]),
    "dsp_mfcc_batch_device": (C.c_int, [_P, _P, _P, _P, _P, _P, _I64, C.POINTER(MfccParams), _P, _P, _P, _P, _P]),
    "dsp_dtw_fit_device": (C.c_int, [_P, _P, _P, _P, _P, _I64, _I32, _I32, _I64, C.POINTER(_P)]),
    "dsp_dtw_topk_device": (C.c_int, [_P, _P, _P, _P, _I64, _I32, _P, _P, _P]),
    "dsp_dtw_topk_bounded_device": (C.c_int, [_P, _P, _P, _P, _I64, _I32, _P, _P, _P, _P]),
    "dsp_dtw_last_stats": (C.c_int, [_P, C.POINTER(_I64), C.POINTER(_I64)]),
    "dsp_dtw_free": (C.c_int, [_P]),
    "dsp_wav_scan": (C.c_int, [_P, _I64, _I32, _P]),
    "dsp_wav_read": (C.c_int, [_P, _I64, _I32, _P, _P, _P, _I64]),
    "dsp_host_alloc": (C.c_int, [_I64, C.POINTER(_P)]),
    "dsp_host_free": (C.c_int, [_P]),
}

_lib = None


def load_library():
    """dlopen libdspfront.so and attach prototypes; raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DspError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make`.  There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the ABI is incomplete
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error():
    return load_library().dsp_last_error().decode("utf-8", "replace")


def check(rc):
    """Map a dsp_status to the exception the reference's callers expect: caller errors are
    ValueError (they catch it per file, experiments/run_experiments.py:109-111)."""
    if rc == 0:
        return
    msg = last_error()
    if rc in (DSP_ERR_INVALID, DSP_ERR_UNSUPPORTED):
        raise ValueError(msg)
    raise DspError(f"libdspfront error {rc}: {msg}")
