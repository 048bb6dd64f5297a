"""Batched host-buffer API over the C ABI (NumPy in, NumPy out).

These are the additive ``*_batch`` entry points of SURVEY.md section 8(b): one call processes a
packed ragged batch of utterances (``samples`` + ``offsets[B+1]``) through the CUDA kernels.
The per-call functions of the drop-in ``src`` package are batch-of-one wrappers around them.
"""
import ctypes as C
import threading

import numpy as np

from . import _capi
from ._capi import FrontendOutputs, FrontendParams, WINDOW_IDS, check, load_library

_DTYPES = {np.dtype(np.int16): _capi.DSP_S16, np.dtype(np.uint8): _capi.DSP_U8,
           np.dtype(np.float32): _capi.DSP_F32, np.dtype(np.float64): _capi.DSP_F64}

STAT_NAMES = ("mean", "std", "max", "min", "median")
FEATURE_NAMES = [f"{f}_{s}" for f in ("energy", "magnitude", "zcr") for s in STAT_NAMES]


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Context:
    """One CUDA context handle (device ordinal + stream + scratch)."""

    def __init__(self, device=0):
        self.lib = load_library()
        h = C.c_void_p()
        check(self.lib.dsp_create(int(device), C.byref(h)))
        self.handle = h
        self.device = int(device)

    def close(self):
        if getattr(self, "handle", None):
            self.lib.dsp_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, cuda_stream_ptr):
        check(self.lib.dsp_set_stream(self.handle, C.c_void_p(cuda_stream_ptr)))

    def use_own_stream(self):
        check(self.lib.dsp_use_own_stream(self.handle))

    def set_tuning(self, key, value):
        check(self.lib.dsp_set_tuning(self.handle, key.encode(), int(value)))

    def sync(self):
        check(self.lib.dsp_sync(self.handle))

    @property
    def launch_count(self):
        return int(self.lib.dsp_launch_count(self.handle))

    @property
    def sm_count(self):
        return int(self.lib.dsp_device_sm_count(self.handle))


_default = {}
_lock = threading.Lock()


def default_context(device=0):
    with _lock:
        ctx = _default.get(device)
        if ctx is None:
            ctx = _default[device] = Context(device)
        return ctx


def _host_ctx(ctx):
    """Context for a host-pointer call: host entry points run on the context's own stream (a torch
    stream installed earlier by the device API may no longer exist)."""
    ctx = ctx or default_context()
    ctx.use_own_stream()
    return ctx


def make_params(frame_length, frame_shift, window_type="hamming", do_endpoint_detection=True,
                energy_high_ratio=0.5, energy_low_ratio=0.1, zcr_threshold_ratio=1.5, channels=1,
                force_exact=False):
    if window_type not in WINDOW_IDS:
        raise ValueError(f"unsupported window type: {window_type}")     # audio_processing.py:296
    return FrontendParams(int(frame_length), int(frame_shift), WINDOW_IDS[window_type],
                          int(bool(do_endpoint_detection)), float(energy_high_ratio),
                          float(energy_low_ratio), float(zcr_threshold_ratio), int(channels),
                          int(bool(force_exact)), 0)


def plan(offsets, params, lengths=None):
    """(feat_offsets, epd_offsets, max_len) -- host arithmetic only (dsp_frontend_plan)."""
    lib = load_library()
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    if lengths is not None:
        lengths = np.ascontiguousarray(lengths, dtype=np.int32)
    b = len(offsets) - 1
    fo = np.zeros(b + 1, dtype=np.int64)
    eo = np.zeros(b + 1, dtype=np.int64)
    mx = C.c_int64(0)
    check(lib.dsp_frontend_plan(_ptr(offsets), _ptr(lengths), b, C.byref(params), _ptr(fo), _ptr(eo), C.byref(mx)))
    return fo, eo, int(mx.value)


class FrontendResult:
    """Outputs of one front-end batch (ragged arrays + offsets)."""

    def __init__(self, **kw):
        self.__dict__.update(kw)

    def __len__(self):
        return len(self.start)

    def ok(self, b):
        return (int(self.status[b]) & 0xff) == 0

    def frames(self, b):
        o = int(self.feat_offsets[b])
        n = int(self.n_frames[b])
        return self.energy[o:o + n], self.magnitude[o:o + n], self.zcr[o:o + n]

    def dense(self, b):
        """frame_signal's (n_frames, frame_length) float64 matrix of utterance b (emit_dense_frames=True)."""
        o = int(self.feat_offsets[b])
        return self.dense_frames[o:o + int(self.n_frames[b])]

    def epd_lists(self, b):
        o = int(self.epd_offsets[b])
        n = int(self.n_epd_frames[b])
        return self.epd_energy[o:o + n], self.epd_zcr[o:o + n]


def pack_aligned(utterances, align=8):
    """Concatenate PCM utterances with every start rounded up to a multiple of `align` samples
    (16 bytes for int16): returns (samples, offsets[B+1], lengths[B]) for frontend_batch(...,
    lengths=...), the layout on which the aligned TMA / streaming loads apply to ragged data."""
    lengths = np.array([len(u) for u in utterances], dtype=np.int32)
    room = (lengths.astype(np.int64) + align - 1) // align * align
    offsets = np.zeros(len(utterances) + 1, dtype=np.int64)
    np.cumsum(room, out=offsets[1:])
    dtype = utterances[0].dtype if len(utterances) else np.int16
    samples = np.zeros(int(offsets[-1]), dtype=dtype)
    for u, o in zip(utterances, offsets[:-1]):
        samples[o:o + len(u)] = u
    return samples, offsets, lengths


def frontend_batch(samples, offsets, frame_length, frame_shift, window_type="hamming",
                   do_endpoint_detection=True, energy_high_ratio=0.5, energy_low_ratio=0.1,
                   zcr_threshold_ratio=1.5, channels=1, emit_epd_lists=False, force_exact=False,
                   emit_frames=True, lengths=None, ctx=None, float64_outputs=False, emit_dense_frames=False):
    """preprocess -> endpoint_detection -> frame_signal -> extract_frame_features -> 15 statistics
    for every utterance of a packed batch (src/audio_processing.py:364-394 and
    src/feature_extraction.py:91-112, batched).  `samples` is int16 / uint8 PCM or float32/64.
    emit_frames=False skips the download of the per-frame sequences (the callers of the
    'statistical' method only consume the 15 statistics, run_experiments.py:102-107).
    float64_outputs=True returns energy / magnitude / zcr / stats / epd_zcr as float64 computed by the
    float64 replay kernel (bit-identical to the NumPy path; what the drop-in per-file API hands to the
    reference's callers); emit_dense_frames=True adds `dense_frames`, the [total frames, frame_length]
    float64 matrix of frame_signal (row feat_offsets[b] + t)."""
    ctx = _host_ctx(ctx)
    samples = np.ascontiguousarray(samples)
    if samples.dtype not in _DTYPES:
        raise ValueError(f"unsupported sample dtype {samples.dtype}")
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    b = len(offsets) - 1
    p = make_params(frame_length, frame_shift, window_type, do_endpoint_detection, energy_high_ratio,
                    energy_low_ratio, zcr_threshold_ratio, channels, force_exact)
    if lengths is not None:
        lengths = np.ascontiguousarray(lengths, dtype=np.int32)
    fo, eo, max_len = plan(offsets, p, lengths)
    if b and (offsets[0] < 0 or offsets[-1] > samples.size):
        raise ValueError("offsets exceed the sample buffer")
    ft = np.float64 if float64_outputs else np.float32
    res = FrontendResult(
        start=np.zeros(b, np.int32), end=np.zeros(b, np.int32), n_epd_frames=np.zeros(b, np.int32),
        n_frames=np.zeros(b, np.int32), status=np.zeros(b, np.int32),
        energy=np.zeros(int(fo[-1]), ft) if emit_frames else None,
        magnitude=np.zeros(int(fo[-1]), ft) if emit_frames else None,
        zcr=np.zeros(int(fo[-1]), ft) if emit_frames else None, stats=np.zeros((b, 15), ft),
        feat_offsets=fo, epd_offsets=eo, max_len=max_len,
        epd_energy=np.zeros(int(eo[-1]), np.float64) if emit_epd_lists else None,
        epd_zcr=np.zeros(int(eo[-1]), ft) if emit_epd_lists else None,
        dense_frames=np.zeros((int(fo[-1]), int(frame_length)), np.float64) if emit_dense_frames else None)
    if float64_outputs:
        out = FrontendOutputs(_ptr(res.start), _ptr(res.end), _ptr(res.n_epd_frames), _ptr(res.n_frames),
                              _ptr(res.status), None, None, None, None, _ptr(res.epd_energy), None,
                              _ptr(res.energy), _ptr(res.magnitude), _ptr(res.zcr), _ptr(res.stats),
                              _ptr(res.epd_zcr), _ptr(res.dense_frames))
    else:
        out = FrontendOutputs(_ptr(res.start), _ptr(res.end), _ptr(res.n_epd_frames), _ptr(res.n_frames),
                              _ptr(res.status), _ptr(res.energy), _ptr(res.magnitude), _ptr(res.zcr),
                              _ptr(res.stats), _ptr(res.epd_energy), _ptr(res.epd_zcr),
                              None, None, None, None, None, _ptr(res.dense_frames))
    check(ctx.lib.dsp_frontend_batch_host(ctx.handle, _ptr(samples), _DTYPES[samples.dtype],
                                          _ptr(offsets), _ptr(lengths), b, C.byref(p), C.byref(out)))
    return res


# ---- single-signal calls (float64, NumPy operation order replayed on the GPU) ----------------
def _f64(x):
    return np.ascontiguousarray(x, dtype=np.float64)


def window(window_type, length):
    if window_type not in WINDOW_IDS:
        raise ValueError(f"unsupported window type: {window_type}")
    out = np.empty(int(length), np.float64)
    check(load_library().dsp_window(WINDOW_IDS[window_type], int(length), _ptr(out)))
    return out


def preprocess(x, mode=2, ctx=None):
    """mode 0 remove_dc, 1 normalize_audio, 2 preprocess (src/audio_processing.py:49-90)."""
    ctx = _host_ctx(ctx)
    x = _f64(x)
    out = np.empty_like(x)
    check(ctx.lib.dsp_preprocess_host(ctx.handle, _ptr(x), x.size, int(mode), _ptr(out)))
    return out


def endpoint_detection(x, frame_length, frame_shift, energy_high_ratio=0.5, energy_low_ratio=0.1,
                       zcr_threshold_ratio=1.5, ctx=None):
    ctx = _host_ctx(ctx)
    x = _f64(x)
    p = make_params(frame_length, frame_shift, "rectangular", True, energy_high_ratio,
                    energy_low_ratio, zcr_threshold_ratio)
    n = x.size
    f1 = (n - int(frame_length)) // int(frame_shift) + 1 if n >= int(frame_length) else 0
    el = np.empty(f1, np.float64)
    zl = np.empty(f1, np.float64)
    s, e, nf = C.c_int32(), C.c_int32(), C.c_int32()
    check(ctx.lib.dsp_endpoint_detection_host(ctx.handle, _ptr(x), n, C.byref(p), C.byref(s), C.byref(e),
                                              C.byref(nf), _ptr(el), _ptr(zl)))
    return int(s.value), int(e.value), el, zl


def frame_signal(x, frame_length, frame_shift, window_type="hamming", ctx=None):
    ctx = _host_ctx(ctx)
    if window_type not in WINDOW_IDS:
        raise ValueError(f"unsupported window type: {window_type}")
    x = _f64(x)
    nf = int(load_library().dsp_frame_count(x.size, int(frame_length), int(frame_shift)))
    out = np.zeros((nf, int(frame_length)), np.float64)
    if nf:
        check(ctx.lib.dsp_frame_signal_host(ctx.handle, _ptr(x), x.size, int(frame_length),
                                            int(frame_shift), WINDOW_IDS[window_type], _ptr(out)))
    return out


def frame_features(frames, want_stats=True, ctx=None):
    """extract_frame_features (+ the 15 statistics) of an arbitrary [F, fl] float64 matrix."""
    ctx = _host_ctx(ctx)
    frames = _f64(frames)
    if frames.ndim == 1:
        frames = frames.reshape(1, -1)
    nf, fl = frames.shape
    if nf == 0:
        raise ValueError("No frames provided for feature extraction.")
    e, m, z = (np.empty(nf, np.float64) for _ in range(3))
    st = np.empty(15, np.float64) if want_stats else None
    check(ctx.lib.dsp_frame_features_host(ctx.handle, _ptr(frames), nf, fl, _ptr(e), _ptr(m), _ptr(z), _ptr(st)))
    return e, m, z, st


def sequence_stats(seq, ctx=None):
    ctx = _host_ctx(ctx)
    seq = _f64(seq).ravel()
    out = np.empty(5, np.float64)
    check(ctx.lib.dsp_sequence_stats_host(ctx.handle, _ptr(seq), seq.size, _ptr(out)))
    return out


def _axis0_is_inner(x):
    """True when NumPy's reduction over axis 0 of `x` (np.mean / np.std, axis=0) runs along its inner loop, i.e. sums
    every column with its pairwise algorithm; False when it adds the rows one after another.  The iterator puts axis 0
    innermost when, after dropping length-1 axes, it is the only axis left, or its |stride| is strictly below every
    other axis's and no stride involved is zero (zero or equal strides leave the axes in C order).  `x` is a NumPy
    array or a torch tensor; decide on the caller's array, before any contiguous copy."""
    strides = x.strides if isinstance(x, np.ndarray) else tuple(x.stride())
    if x.ndim == 0 or x.shape[0] <= 1:
        return True                      # a single row: both orders give the same sums
    s0 = abs(strides[0])
    rest = [abs(s) for n, s in zip(x.shape[1:], strides[1:]) if n != 1]
    return not rest or (s0 != 0 and all(s != 0 and s0 < s for s in rest))


def zscore(features, mean=None, std=None, ctx=None):
    """normalize_features (src/feature_extraction.py:157-181).  The fit sums each column in the order NumPy would
    for this array's layout (_axis0_is_inner), so mean and std are bit-identical to np.mean / np.std(axis=0)."""
    ctx = _host_ctx(ctx)
    features = np.asarray(features)
    pairwise = _axis0_is_inner(features)
    x = _f64(features)
    one_d = x.ndim == 1
    x2 = x.reshape(-1, 1) if one_d else x.reshape(x.shape[0], -1)
    n, d = x2.shape
    fit_mean, fit_std = mean is None, std is None
    # mean / std have the shape of one row (np.mean(axis=0)); given ones broadcast to it
    row = (1,) if one_d else x.shape[1:]
    m = np.empty(d, np.float64) if fit_mean else _f64(np.broadcast_to(mean, row)).reshape(d).copy()
    s = np.empty(d, np.float64) if fit_std else _f64(np.broadcast_to(std, row)).reshape(d).copy()
    out = np.empty_like(x2)
    if fit_mean or fit_std:
        fm, fsd = np.empty(d, np.float64), np.empty(d, np.float64)
        check(ctx.lib.dsp_zscore_host(ctx.handle, _ptr(x2), n, d, 2 if pairwise else 1, _ptr(fm), _ptr(fsd), None))
        if fit_mean:
            m = fm
        if fit_std:
            s = fsd
    check(ctx.lib.dsp_zscore_host(ctx.handle, _ptr(x2), n, d, 0, _ptr(m), _ptr(s), _ptr(out)))
    if one_d:
        return out.reshape(x.shape), m[0], s[0]
    return out.reshape(x.shape), m.reshape(x.shape[1:]), s.reshape(x.shape[1:])


class KNN:
    """KNeighborsClassifier(n_neighbors=k) restated on the GPU: exact float64 neighbours
    (ties to the lower train index), majority vote with ties to the smallest label."""

    def __init__(self, n_neighbors=3, ctx=None, index_base=0):
        self.k = int(n_neighbors)
        self.ctx = _host_ctx(ctx)
        self.index_base = int(index_base)
        self.handle = None
        self.classes_ = None

    def fit(self, X, y):
        X = _f64(X)
        y = np.asarray(y)
        self.classes_, enc = np.unique(y, return_inverse=True)
        enc = np.ascontiguousarray(enc, dtype=np.int32)
        self._free()
        self.ctx.use_own_stream()
        h = C.c_void_p()
        check(self.ctx.lib.dsp_knn_fit_host(self.ctx.handle, _ptr(X), _ptr(enc), X.shape[0], X.shape[1],
                                            self.k, self.index_base, C.byref(h)))
        self.handle = h
        self.n_features_in_ = X.shape[1]
        return self

    def kneighbors(self, Q):
        Q = _f64(Q)
        self.ctx.use_own_stream()
        m = Q.shape[0]
        idx = np.empty((m, self.k), np.int64)
        d2 = np.empty((m, self.k), np.float64)
        lab = np.empty((m, self.k), np.int32)
        check(self.ctx.lib.dsp_knn_topk_host(self.handle, _ptr(Q), m, _ptr(idx), _ptr(d2), _ptr(lab)))
        return np.sqrt(d2), idx, lab

    def predict(self, Q):
        Q = _f64(Q)
        if Q.ndim != 2 or Q.shape[1] != self.n_features_in_:
            raise ValueError(f"X has {Q.shape[-1]} features, but KNN is expecting {self.n_features_in_}")
        out = np.empty(Q.shape[0], np.int32)
        self.ctx.use_own_stream()
        check(self.ctx.lib.dsp_knn_predict_host(self.handle, _ptr(Q), Q.shape[0], _ptr(out)))
        return self.classes_[out]

    def last_stats(self):
        """(queries rescanned in float64, scan kind) of the last kneighbors / predict call: 0 float64 only,
        1 fp32 tiled scan, 2 tensor-core scan."""
        n, kind = C.c_int64(), C.c_int32()
        check(self.ctx.lib.dsp_knn_last_stats(self.handle, C.byref(n), C.byref(kind)))
        return int(n.value), int(kind.value)

    def _free(self):
        if self.handle:
            self.ctx.lib.dsp_knn_free(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self._free()
        except Exception:
            pass
