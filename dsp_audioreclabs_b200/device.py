"""The same entry points on torch CUDA tensors (device pointers straight into the C ABI).

torch is plumbing here -- device memory, streams, torch.distributed -- the compute is
libdspfront.so.  Nothing in this module creates a host copy of the samples.
"""
import ctypes as C

import numpy as np
import torch

from . import _capi
from ._capi import FrontendOutputs, check
from .batch import _axis0_is_inner, _window_id, default_context, make_params, plan
from .mfcc_dtw import DEFAULTS, _mfcc_setup

_TORCH_DTYPES = {torch.int16: _capi.DSP_S16, torch.uint8: _capi.DSP_U8,
                 torch.float32: _capi.DSP_F32, torch.float64: _capi.DSP_F64}


def _dp(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _device(device):
    """torch.device of `device`, by default torch's current CUDA device."""
    return torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)


def _bind(device, ctx=None, stream=None):
    """`ctx` (default: the default context of `device`) with `stream` (default: torch's current stream of `device`)
    installed, so the C entry points called with it enqueue there."""
    ctx = ctx or default_context(device.index or 0)
    ctx.set_stream((torch.cuda.current_stream(device) if stream is None else stream).cuda_stream)
    return ctx


class _Uploads:
    """Orders launches after the work a constructor enqueued on torch's current stream.  Each stream waits once, before
    its first launch: a CUDA graph captured on a stream that has already run records no wait on this event."""

    def __init__(self, device):
        self._done = torch.cuda.Event()
        self._done.record(torch.cuda.current_stream(device))
        self._waited = set()

    def wait(self, stream):
        if stream.cuda_stream not in self._waited:
            stream.wait_event(self._done)
            self._waited.add(stream.cuda_stream)


def _frontend_outputs(n_utts, n_frames, n_epd, device, epd_lists):
    """Zero-filled outputs of one front-end batch (n_frames per-frame rows, n_epd endpoint-detection rows when
    epd_lists) by FrontendOutputs field name, and the FrontendOutputs of their device pointers."""
    i32 = lambda *shape: torch.zeros(*shape, dtype=torch.int32, device=device)
    f32 = lambda *shape: torch.zeros(*shape, dtype=torch.float32, device=device)
    nf, ne = max(n_frames, 1), max(n_epd, 1)
    outs = dict(start=i32(n_utts), end=i32(n_utts), n_epd_frames=i32(n_utts), n_frames=i32(n_utts), status=i32(n_utts),
                energy=f32(nf), magnitude=f32(nf), zcr=f32(nf), stats=f32(n_utts, 15),
                epd_energy=torch.zeros(ne, dtype=torch.float64, device=device) if epd_lists else None,
                epd_zcr=f32(ne) if epd_lists else None)
    return outs, FrontendOutputs(**{name: _dp(t) for name, t in outs.items()})


class DeviceFrontend:
    """Plans one packed batch layout (host offsets) and runs the front end on device tensors.

    The plan (ragged output offsets, longest utterance) depends only on `offsets` and the frame
    parameters, so it is computed once and reused for every launch over batches of that shape.
    """

    def __init__(self, offsets, frame_length, frame_shift, window_type="hamming",
                 do_endpoint_detection=True, energy_high_ratio=0.5, energy_low_ratio=0.1,
                 zcr_threshold_ratio=1.5, emit_epd_lists=False, force_exact=False, device=None, ctx=None,
                 lengths=None):
        self.device = _device(device)
        self.ctx = _bind(self.device, ctx)
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
        outs, self._out = _frontend_outputs(self.n_utts, int(self.h_feat_offsets[-1]), int(self.h_epd_offsets[-1]), dev,
                                            emit_epd_lists)
        vars(self).update(outs)                   # self.start, self.end, ..., self.epd_zcr
        self._uploads = _Uploads(dev)

    def set_window(self, window_type):
        self.params.window = _window_id(window_type)

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
        self._uploads.wait(st)
        _bind(self.device, self.ctx, st)
        check(self.ctx.lib.dsp_frontend_batch_device(
            self.ctx.handle, _dp(samples), _TORCH_DTYPES[samples.dtype], _dp(self.offsets), _dp(self.lengths),
            _dp(self.feat_offsets), _dp(self.epd_offsets), self.n_utts, self.max_len,
            C.byref(self.params), C.byref(self._out)))
        return self


class DeviceKNN:
    """KNN over device tensors: fit on a (row shard of the) train matrix, top-k / predict for
    device-resident queries."""

    def __init__(self, n_neighbors=3, ctx=None, device=None, index_base=0):
        self.device = _device(device)
        self.ctx = _bind(self.device, ctx)
        self.k = int(n_neighbors)
        self.index_base = int(index_base)
        self.handle = None

    def fit(self, train, labels):
        assert train.is_cuda and train.dtype == torch.float64 and train.is_contiguous()
        assert labels.is_cuda and labels.dtype == torch.int32
        _bind(self.device, self.ctx)
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
        _bind(self.device, self.ctx)
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
        _bind(self.device, self.ctx)
        out = torch.empty(queries.shape[0], dtype=torch.int32, device=self.device)
        check(self.ctx.lib.dsp_knn_predict_device(self.handle, _dp(queries), queries.shape[0], _dp(out)))
        return out

    def last_stats(self):
        """(queries rescanned in float64, scan kind) of the last call: 0 float64 only, 1 fp32 tiled scan, 2 dense
        tensor-core scan, 3 tensor-core filter (D <= 15)."""
        n, kind = C.c_int64(), C.c_int32()
        check(self.ctx.lib.dsp_knn_last_stats(self.handle, C.byref(n), C.byref(kind)))
        return int(n.value), int(kind.value)

    def merge_vote(self, cand_d2, cand_idx, cand_lab):
        """[R, m, k] candidate lists (e.g. all-gathered from R row shards) -> labels, idx, d2."""
        _bind(self.device, self.ctx)
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
    ctx = _bind(x.device, ctx)
    pairwise = _axis0_is_inner(x)
    x = x.contiguous()
    n, d = x.shape
    fm, fs = _zscore_fit(ctx, x, pairwise) if mean is None or std is None else (None, None)
    # the apply kernel replaces std == 0 with 1 in place (csrc/misc.cu), so a caller's mean and std are copied first
    m = fm if mean is None else mean.clone()
    s = fs if std is None else std.clone()
    out = torch.empty_like(x)
    check(ctx.lib.dsp_zscore_device(ctx.handle, _dp(x), n, d, 0, _dp(m), _dp(s), _dp(out)))
    return out, m, s


def _zscore_fit(ctx, x, pairwise):
    """Column (mean, std) of a contiguous float64 [n, d] CUDA tensor, std == 0 kept; the column sums are pairwise or
    row by row (batch._axis0_is_inner of the caller's layout)."""
    n, d = x.shape
    mean = torch.empty(d, dtype=torch.float64, device=x.device)
    std = torch.empty(d, dtype=torch.float64, device=x.device)
    check(ctx.lib.dsp_zscore_device(ctx.handle, _dp(x), n, d, 2 if pairwise else 1, _dp(mean), _dp(std), None))
    return mean, std


def zscore_apply_f32(stats, mean, std, out=None, ctx=None):
    """(float32 [n, d] statistics of the fused front end) -> float64 z-scores with the given train mean / std:
    one kernel between DeviceFrontend.stats and DeviceKNN.predict, no torch arithmetic on the path."""
    assert stats.is_cuda and stats.dtype == torch.float32 and stats.is_contiguous() and stats.dim() == 2
    ctx = _bind(stats.device, ctx)
    n, d = stats.shape
    if out is None:
        out = torch.empty(n, d, dtype=torch.float64, device=stats.device)
    check(ctx.lib.dsp_zscore_apply_f32_device(ctx.handle, _dp(stats), n, d, _dp(mean), _dp(std), _dp(out)))
    return out


class DeviceMFCC:
    """MFCC of the trimmed segments [start, end) of one packed int16 batch layout, on device tensors.

    The output rows are planned on the host from `offsets` alone: utterance b may use rows
    [mfcc_offsets[b], mfcc_offsets[b + 1]), its untrimmed frame count (dsp_frontend_plan), which bounds the frame count
    of any segment of it.  So the front end's start / end never leave the device.  Parameters as mfcc_dtw.DEFAULTS."""

    def __init__(self, offsets, frame_length=1102, frame_shift=441, lengths=None, ctx=None, device=None, **params):
        p = dict(DEFAULTS)
        p.update(params, frame_length=int(frame_length), frame_shift=int(frame_shift))
        self.params, self.filterbank, self.dct = _mfcc_setup(p)
        self.device = _device(device)
        self.ctx = _bind(self.device, ctx)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        self.n_utts = len(offsets) - 1
        h_lengths = None if lengths is None else np.ascontiguousarray(lengths, dtype=np.int32)
        self.h_mfcc_offsets, _, _ = plan(offsets, make_params(frame_length, frame_shift), h_lengths)
        self.total_frames = int(self.h_mfcc_offsets[-1])
        self.n_ceps = int(p["n_ceps"])
        dev = self.device
        self.offsets = torch.from_numpy(offsets).to(dev)
        self.lengths = None if h_lengths is None else torch.from_numpy(h_lengths).to(dev)
        self.mfcc_offsets = torch.from_numpy(self.h_mfcc_offsets).to(dev)
        self._uploads = _Uploads(dev)

    def run(self, samples, start, end, out=None):
        """Enqueue the MFCC of `samples` (1-D int16 CUDA tensor laid out by `offsets`) over the segments given by the
        int32 CUDA tensors start / end (e.g. DeviceFrontend's) on torch's current stream.  Returns (mfcc float32
        [total_frames, n_ceps], mfcc_offsets int64 [B + 1], n_frames int32 [B]): utterance b's frames are rows
        mfcc_offsets[b] .. + n_frames[b]; the rest of its rows are left as they were in `out` (if given)."""
        if not samples.is_cuda or samples.dtype != torch.int16:
            raise ValueError("samples must be an int16 CUDA tensor")
        for name, t in (("start", start), ("end", end)):
            if not t.is_cuda or t.dtype != torch.int32 or not t.is_contiguous() or t.numel() != self.n_utts:
                raise ValueError(f"{name} must be a contiguous int32 CUDA tensor of {self.n_utts} entries")
        rows = max(self.total_frames, 1)
        if out is None:
            out = torch.empty(rows, self.n_ceps, dtype=torch.float32, device=self.device)
        elif out.dtype != torch.float32 or not out.is_contiguous() or tuple(out.shape) != (rows, self.n_ceps):
            raise ValueError(f"out must be a contiguous float32 tensor of shape ({rows}, {self.n_ceps})")
        n_frames = torch.empty(self.n_utts, dtype=torch.int32, device=self.device)
        st = torch.cuda.current_stream(self.device)
        self._uploads.wait(st)
        _mfcc_device(_bind(self.device, self.ctx, st), samples.contiguous(), self.offsets, self.lengths, start, end,
                     self.params, self.filterbank, self.dct, self.mfcc_offsets, out, n_frames)
        return out[:self.total_frames], self.mfcc_offsets, n_frames


def _mfcc_device(ctx, samples, offsets, lengths, start, end, params, filterbank, dct, mfcc_offsets, out, n_frames):
    """dsp_mfcc_batch_device over contiguous CUDA tensors: int16 samples, int64 offsets / mfcc_offsets [B + 1], int32
    lengths (or None) / start / end / n_frames [B], float32 out; MfccParams and the host tables of mfcc_dtw."""
    check(ctx.lib.dsp_mfcc_batch_device(
        ctx.handle, _dp(samples), _dp(offsets), _dp(lengths), _dp(start), _dp(end), offsets.numel() - 1,
        C.byref(params), filterbank.ctypes.data_as(C.c_void_p), dct.ctypes.data_as(C.c_void_p), _dp(mfcc_offsets),
        _dp(out), _dp(n_frames)))


class DeviceDTW:
    """k cheapest templates under DTW for device-resident sequences: fit keeps a device copy of the templates, topk
    scores every (query, template) pair without a cost matrix and abandons pairs that cannot enter the top k."""

    def __init__(self, n_neighbors=1, ctx=None, device=None, index_base=0):
        self.device = _device(device)
        self.ctx = _bind(self.device, ctx)
        self.k = int(n_neighbors)
        self.index_base = int(index_base)
        self.handle = None

    @staticmethod
    def _check_seqs(feats, offsets, lengths):
        if not feats.is_cuda or feats.dtype != torch.float32 or feats.dim() != 2 or not feats.is_contiguous():
            raise ValueError("feats must be a contiguous float32 CUDA tensor [frames, dim]")
        if not offsets.is_cuda or offsets.dtype != torch.int64 or offsets.dim() != 1 or not offsets.is_contiguous():
            raise ValueError("offsets must be a contiguous int64 CUDA tensor [n + 1] (in frames)")
        if lengths is not None and (not lengths.is_cuda or lengths.dtype != torch.int32 or not lengths.is_contiguous()
                                    or lengths.numel() != offsets.numel() - 1):
            raise ValueError("lengths must be a contiguous int32 CUDA tensor [n]")

    def fit(self, feats, offsets, labels, lengths=None):
        """Templates: sequence i is lengths[i] (default offsets[i + 1] - offsets[i]) rows of feats from offsets[i];
        labels int32 [n] (None: 0).  Synchronises once."""
        self._check_seqs(feats, offsets, lengths)
        if labels is not None and (not labels.is_cuda or labels.dtype != torch.int32 or not labels.is_contiguous()):
            raise ValueError("labels must be a contiguous int32 CUDA tensor")
        _bind(self.device, self.ctx)
        self.free()
        h = C.c_void_p()
        check(self.ctx.lib.dsp_dtw_fit_device(self.ctx.handle, _dp(feats), _dp(offsets), _dp(lengths), _dp(labels),
                                              offsets.numel() - 1, feats.shape[1], self.k, self.index_base, C.byref(h)))
        self.handle = h
        self.dim = feats.shape[1]
        return self

    def topk(self, feats, offsets, lengths=None, max_q_frames=None, bound=None):
        """(cost float64, template index int64, label int32), each [nq, k], ties to the lower index, (inf, -1, -1)
        where fewer than k templates have a finite cost.  max_q_frames (optional) only picks the kernel build.

        bound (optional contiguous float64 CUDA tensor [nq], dsp_dtw_topk_bounded_device): a cost bound per query.
        Only templates whose cost is <= bound[q] (ties included) are returned: every such template is either returned
        or displaced by k templates ordered before it by (cost, index), and the query's other slots are (inf, -1, -1).
        A negative or NaN bound returns an empty list, +inf is no bound.  Returned costs are the unbounded call's, bit
        for bit.  Uses: rejecting queries no template is close enough to, and row shards of a template set given a
        cost the caller already knows (pairs above it are abandoned from the first template on)."""
        self._check_seqs(feats, offsets, lengths)
        if feats.shape[1] != self.dim:
            raise ValueError(f"queries have {feats.shape[1]} features, the templates {self.dim}")
        nq = offsets.numel() - 1
        if bound is not None and (not bound.is_cuda or bound.dtype != torch.float64 or not bound.is_contiguous()
                                  or bound.numel() != nq):
            raise ValueError(f"bound must be a contiguous float64 CUDA tensor of {nq} entries")
        _bind(self.device, self.ctx)
        cost = torch.empty(nq, self.k, dtype=torch.float64, device=self.device)
        idx = torch.empty(nq, self.k, dtype=torch.int64, device=self.device)
        lab = torch.empty(nq, self.k, dtype=torch.int32, device=self.device)
        check(self.ctx.lib.dsp_dtw_topk_bounded_device(self.handle, _dp(feats), _dp(offsets), _dp(lengths), nq,
                                                       int(max_q_frames or 0), _dp(bound), _dp(cost), _dp(idx), _dp(lab)))
        return cost, idx, lab

    def predict(self, feats, offsets, lengths=None, max_q_frames=None, bound=None):
        """Majority label of the k cheapest templates, ties to the smallest label: int32 [nq].  With a bound (see
        topk) the vote is over the templates within it, and a query with none gets -1."""
        cost, idx, lab = self.topk(feats, offsets, lengths, max_q_frames, bound)
        nq = cost.shape[0]
        out = torch.empty(nq, dtype=torch.int32, device=self.device)
        if nq:
            check(self.ctx.lib.dsp_knn_merge_vote_device(self.ctx.handle, _dp(cost), _dp(idx), _dp(lab), 1, nq, self.k,
                                                         _dp(out), None, None))
        return out

    def last_stats(self):
        """(pairs scored to their last cell, pairs abandoned early) of the last topk / predict call; the pairs of a
        query whose bound admits nothing count as abandoned."""
        scored, abandoned = C.c_int64(), C.c_int64()
        check(self.ctx.lib.dsp_dtw_last_stats(self.handle, C.byref(scored), C.byref(abandoned)))
        return int(scored.value), int(abandoned.value)

    def free(self):
        if self.handle:
            self.ctx.lib.dsp_dtw_free(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass
