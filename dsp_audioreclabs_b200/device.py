"""The same entry points on torch CUDA tensors (device pointers straight into the C ABI).

torch is plumbing here -- device memory, streams, torch.distributed -- the compute is
libdspfront.so.  Nothing in this module creates a host copy of the samples.
"""
import ctypes as C

import numpy as np
import torch

from . import _capi
from ._capi import FrontendOutputs, check
from .batch import _axis0_is_inner, default_context, make_params, plan

_TORCH_DTYPES = {torch.int16: _capi.DSP_S16, torch.uint8: _capi.DSP_U8,
                 torch.float32: _capi.DSP_F32, torch.float64: _capi.DSP_F64}


def _dp(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class DeviceFrontend:
    """Plans one packed batch layout (host offsets) and runs the front end on device tensors.

    The plan (ragged output offsets, longest utterance) depends only on `offsets` and the frame
    parameters, so it is computed once and reused for every launch over batches of that shape.
    """

    def __init__(self, offsets, frame_length, frame_shift, window_type="hamming",
                 do_endpoint_detection=True, energy_high_ratio=0.5, energy_low_ratio=0.1,
                 zcr_threshold_ratio=1.5, emit_epd_lists=False, force_exact=False, device=None, ctx=None,
                 lengths=None):
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.ctx = ctx or default_context(self.device.index or 0)
        self.params = make_params(frame_length, frame_shift, window_type, do_endpoint_detection,
                                  energy_high_ratio, energy_low_ratio, zcr_threshold_ratio, 1, force_exact)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        self.n_utts = len(offsets) - 1
        self.h_offsets = offsets
        self.h_lengths = None if lengths is None else np.ascontiguousarray(lengths, dtype=np.int32)
        self.h_feat_offsets, self.h_epd_offsets, self.max_len = plan(offsets, self.params, self.h_lengths)
        dev = self.device
        self.offsets = torch.from_numpy(offsets).to(dev)
        self.lengths = None if self.h_lengths is None else torch.from_numpy(self.h_lengths).to(dev)
        self.feat_offsets = torch.from_numpy(self.h_feat_offsets).to(dev)
        self.epd_offsets = torch.from_numpy(self.h_epd_offsets).to(dev)
        b, nf, ne = self.n_utts, int(self.h_feat_offsets[-1]), int(self.h_epd_offsets[-1])
        i32 = dict(dtype=torch.int32, device=dev)
        f32 = dict(dtype=torch.float32, device=dev)
        self.start = torch.zeros(b, **i32)
        self.end = torch.zeros(b, **i32)
        self.n_epd_frames = torch.zeros(b, **i32)
        self.n_frames = torch.zeros(b, **i32)
        self.status = torch.zeros(b, **i32)
        self.energy = torch.zeros(max(nf, 1), **f32)
        self.magnitude = torch.zeros(max(nf, 1), **f32)
        self.zcr = torch.zeros(max(nf, 1), **f32)
        self.stats = torch.zeros(b, 15, **f32)
        self.epd_energy = torch.zeros(max(ne, 1), dtype=torch.float64, device=dev) if emit_epd_lists else None
        self.epd_zcr = torch.zeros(max(ne, 1), **f32) if emit_epd_lists else None
        self._out = FrontendOutputs(_dp(self.start), _dp(self.end), _dp(self.n_epd_frames), _dp(self.n_frames),
                                    _dp(self.status), _dp(self.energy), _dp(self.magnitude), _dp(self.zcr),
                                    _dp(self.stats), _dp(self.epd_energy), _dp(self.epd_zcr))
        # the uploads and fills above were enqueued on torch's current stream; run() may use another one
        self._ready = torch.cuda.Event()
        self._ready.record(torch.cuda.current_stream(dev))
        self._waited = set()

    def set_window(self, window_type):
        self.params.window = _capi.WINDOW_IDS[window_type]

    def algorithmic_bytes(self, sample_bytes=2):
        """SURVEY.md section 8(d): s*L + 4*(3*F2 + 15 + 2) [+ 8*F1 when the EPD lists are written],
        with F2 the frames actually produced (call after a run)."""
        f2 = int(self.n_frames.sum().item())
        total = sample_bytes * int(self.h_offsets[-1] - self.h_offsets[0]) + 4 * (3 * f2 + 17 * self.n_utts)
        if self.epd_energy is not None:
            total += 8 * int(self.n_epd_frames.sum().item())
        return total

    def run(self, samples, stream=None):
        """Enqueue the front end over `samples` (1-D CUDA tensor laid out by `offsets`) on
        `stream` (default: torch's current stream).  Asynchronous."""
        if not samples.is_cuda or samples.dtype not in _TORCH_DTYPES:
            raise ValueError("samples must be a CUDA tensor of int16 / uint8 / float32 / float64")
        # utterances that all start on 16-byte boundaries may use the streaming build of the kernel
        self.params.aligned16 = int(samples.data_ptr() % 16 == 0 and
                                    bool(np.all(self.h_offsets[:-1] * samples.element_size() % 16 == 0)))
        st = stream if stream is not None else torch.cuda.current_stream(self.device)
        if st.cuda_stream not in self._waited:            # once per stream: order the launch after the construction work
            st.wait_event(self._ready)
            self._waited.add(st.cuda_stream)
        self.ctx.set_stream(st.cuda_stream)
        check(self.ctx.lib.dsp_frontend_batch_device(
            self.ctx.handle, _dp(samples), _TORCH_DTYPES[samples.dtype], _dp(self.offsets), _dp(self.lengths),
            _dp(self.feat_offsets), _dp(self.epd_offsets), self.n_utts, self.max_len,
            C.byref(self.params), C.byref(self._out)))
        return self


class DeviceKNN:
    """KNN over device tensors: fit on a (row shard of the) train matrix, top-k / predict for
    device-resident queries."""

    def __init__(self, n_neighbors=3, ctx=None, device=None, index_base=0):
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.ctx = ctx or default_context(self.device.index or 0)
        self.k = int(n_neighbors)
        self.index_base = int(index_base)
        self.handle = None

    def _stream(self):
        self.ctx.set_stream(torch.cuda.current_stream(self.device).cuda_stream)

    def fit(self, train, labels):
        assert train.is_cuda and train.dtype == torch.float64 and train.is_contiguous()
        assert labels.is_cuda and labels.dtype == torch.int32
        self._stream()
        self.free()
        h = C.c_void_p()
        check(self.ctx.lib.dsp_knn_fit_device(self.ctx.handle, _dp(train), _dp(labels), train.shape[0],
                                              train.shape[1], self.k, self.index_base, C.byref(h)))
        self.handle = h
        return self

    def topk(self, queries, bound=None):
        """(sqdist, idx, label) [m, k].  bound (optional float64 [m]): an upper bound on each query's k-th squared
        distance in the WHOLE train set when this handle holds a row shard of it (dsp_knn_topk_bounded_device): the
        shard returns its rows inside that radius -- possibly fewer than k, the rest (-1, inf, -1)."""
        assert queries.is_cuda and queries.dtype == torch.float64 and queries.is_contiguous()
        self._stream()
        m = queries.shape[0]
        idx = torch.empty(m, self.k, dtype=torch.int64, device=self.device)
        d2 = torch.empty(m, self.k, dtype=torch.float64, device=self.device)
        lab = torch.empty(m, self.k, dtype=torch.int32, device=self.device)
        if bound is None:
            check(self.ctx.lib.dsp_knn_topk_device(self.handle, _dp(queries), m, _dp(idx), _dp(d2), _dp(lab)))
        else:
            assert bound.is_cuda and bound.dtype == torch.float64 and bound.is_contiguous() and bound.numel() == m
            check(self.ctx.lib.dsp_knn_topk_bounded_device(self.handle, _dp(queries), m, _dp(bound), _dp(idx), _dp(d2), _dp(lab)))
        return d2, idx, lab

    def predict(self, queries):
        assert queries.is_cuda and queries.dtype == torch.float64 and queries.is_contiguous()
        self._stream()
        out = torch.empty(queries.shape[0], dtype=torch.int32, device=self.device)
        check(self.ctx.lib.dsp_knn_predict_device(self.handle, _dp(queries), queries.shape[0], _dp(out)))
        return out

    def last_stats(self):
        """(queries rescanned in float64, scan kind: 0 float64 only / 1 fp32 tiled / 2 tensor cores) of the last call."""
        import ctypes as C
        n, kind = C.c_int64(), C.c_int32()
        check(self.ctx.lib.dsp_knn_last_stats(self.handle, C.byref(n), C.byref(kind)))
        return int(n.value), int(kind.value)

    def merge_vote(self, cand_d2, cand_idx, cand_lab):
        """[R, m, k] candidate lists (e.g. all-gathered from R row shards) -> labels, idx, d2."""
        self._stream()
        r, m, k = cand_d2.shape
        labels = torch.empty(m, dtype=torch.int32, device=self.device)
        idx = torch.empty(m, k, dtype=torch.int64, device=self.device)
        d2 = torch.empty(m, k, dtype=torch.float64, device=self.device)
        check(self.ctx.lib.dsp_knn_merge_vote_device(self.ctx.handle, _dp(cand_d2.contiguous()),
                                                     _dp(cand_idx.contiguous()), _dp(cand_lab.contiguous()),
                                                     r, m, k, _dp(labels), _dp(idx), _dp(d2)))
        return labels, idx, d2

    def free(self):
        if self.handle:
            self.ctx.lib.dsp_knn_free(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def zscore_device(x, mean=None, std=None, ctx=None):
    """normalize_features on a CUDA float64 [n, d] tensor: the result of normalize_features(x.cpu().numpy()), whose
    column sums follow the tensor's layout (batch._axis0_is_inner), e.g. pairwise for a transposed tensor."""
    assert x.is_cuda and x.dtype == torch.float64 and x.dim() == 2
    ctx = ctx or default_context(x.device.index or 0)
    ctx.set_stream(torch.cuda.current_stream(x.device).cuda_stream)
    pairwise = _axis0_is_inner(x)
    x = x.contiguous()
    n, d = x.shape
    fit = mean is None or std is None
    fm = torch.empty(d, dtype=torch.float64, device=x.device)
    fs = torch.empty(d, dtype=torch.float64, device=x.device)
    if fit:
        check(ctx.lib.dsp_zscore_device(ctx.handle, _dp(x), n, d, 2 if pairwise else 1, _dp(fm), _dp(fs), None))
    m = fm if mean is None else mean.clone()
    s = fs if std is None else std.clone()
    out = torch.empty_like(x)
    check(ctx.lib.dsp_zscore_device(ctx.handle, _dp(x), n, d, 0, _dp(m), _dp(s), _dp(out)))
    return out, m, s


def zscore_apply_f32(stats, mean, std, out=None, ctx=None):
    """(float32 [n, d] statistics of the fused front end) -> float64 z-scores with the given train mean / std:
    one kernel between DeviceFrontend.stats and DeviceKNN.predict, no torch arithmetic on the path."""
    assert stats.is_cuda and stats.dtype == torch.float32 and stats.is_contiguous() and stats.dim() == 2
    ctx = ctx or default_context(stats.device.index or 0)
    ctx.set_stream(torch.cuda.current_stream(stats.device).cuda_stream)
    n, d = stats.shape
    if out is None:
        out = torch.empty(n, d, dtype=torch.float64, device=stats.device)
    check(ctx.lib.dsp_zscore_apply_f32_device(ctx.handle, _dp(stats), n, d, _dp(mean), _dp(std), _dp(out)))
    return out
