"""torch.library custom ops over the C ABI, for callers whose tensors are already torch CUDA tensors
(BASELINE.json north_star: "a thin ctypes/C-ABI layer, or torch custom ops where tensors are already torch").

    import dsp_audioreclabs_b200.torch_ops            # registers torch.ops.dsp_audioreclabs.*
    plan = torch_ops.plan(offsets, 256, 128)           # host arithmetic: ragged output layout of one batch shape
    start, end, n_frames, status, stats, energy, magnitude, zcr = torch.ops.dsp_audioreclabs.frontend_batch(
        samples, plan.offsets, plan.feat_offsets, plan.n_utts, plan.max_len, plan.total_frames, 256, 128, 1, True, 0.5, 0.1, 1.5)
    qn = torch.ops.dsp_audioreclabs.zscore_apply(stats, mean, std)
    labels = torch.ops.dsp_audioreclabs.knn_predict(train_norm, train_labels, qn, 3)
    p5 = torch_ops.plan(offsets, 1102, 441)            # MFCC rows: the untrimmed frame counts bound every segment's
    mfcc, n_frames = torch.ops.dsp_audioreclabs.mfcc_batch(   # (start / end of a frontend_batch at 1102 / 441)
        samples, p5.offsets, start, end, p5.feat_offsets, p5.total_frames, 1102, 441, 2048, 26, 13, 1, 0.97, 1e-10)
    cost, idx, label = torch.ops.dsp_audioreclabs.dtw_topk(t_feats, t_offsets, t_labels, q_feats, q_offsets, 1)

Each op enqueues libdspfront kernels on torch's CURRENT stream with the tensors' device pointers -- no host copies,
no torch arithmetic on the path -- and has a fake (meta) implementation, so the ops trace under torch.compile /
torch.export as opaque calls.  They are tensor-in / tensor-out mirrors of src/audio_processing.py:336-396 +
src/feature_extraction.py:91-112 (front end), :157-181 (z-score) and src/models.py:52-58 (KNN predict), plus the
self-specified MFCC + DTW template matching of mfcc_dtw.py.
"""
import ctypes as C
from collections import OrderedDict
from typing import Tuple

import numpy as np
import torch

from ._capi import check
from .batch import _axis0_is_inner, make_params, plan as _host_plan
from .device import (_TORCH_DTYPES, DeviceDTW, DeviceKNN, _bind, _dp, _frontend_outputs, _mfcc_device, _zscore_fit,
                     zscore_apply_f32, zscore_device)
from .mfcc_dtw import DEFAULTS, _mfcc_setup

NS = "dsp_audioreclabs"


class BatchPlan:
    """Ragged layout of one batch shape: device copies of the CSR offsets and of the per-utterance output offsets
    (dsp_frontend_plan), plus the integers the op needs to size its outputs."""

    def __init__(self, offsets, frame_length, frame_shift, device="cuda"):
        p = make_params(frame_length, frame_shift)
        h = np.ascontiguousarray(offsets, dtype=np.int64)
        fo, _eo, mx = _host_plan(h, p)
        self.n_utts, self.max_len, self.total_frames = len(h) - 1, int(mx), int(fo[-1])
        self.h_offsets, self.h_feat_offsets = h, fo
        self.offsets = torch.from_numpy(h).to(device)
        self.feat_offsets = torch.from_numpy(fo).to(device)


def plan(offsets, frame_length, frame_shift, device="cuda"):
    return BatchPlan(offsets, frame_length, frame_shift, device)


@torch.library.custom_op(f"{NS}::frontend_batch", mutates_args=(), device_types="cuda")
def frontend_batch(samples: torch.Tensor, offsets: torch.Tensor, feat_offsets: torch.Tensor, n_utts: int, max_len: int,
                   total_frames: int, frame_length: int, frame_shift: int, window: int, do_endpoint_detection: bool,
                   energy_high_ratio: float, energy_low_ratio: float, zcr_threshold_ratio: float
                   ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """-> (start[B] i32, end[B] i32, n_frames[B] i32, status[B] i32, stats[B,15] f32, energy, magnitude, zcr [total_frames] f32)."""
    if samples.dtype not in _TORCH_DTYPES:
        raise ValueError("samples must be int16 / uint8 / float32 / float64")
    ctx = _bind(samples.device)
    p = make_params(frame_length, frame_shift, "hamming", do_endpoint_detection, energy_high_ratio, energy_low_ratio,
                    zcr_threshold_ratio)
    p.window = window                             # an id; the C ABI rejects one outside 0..2
    # aligned16 stays 0: only device offsets are known here (DeviceFrontend.run decides it from its host offsets)
    o, out = _frontend_outputs(n_utts, total_frames, 0, samples.device, False)
    check(ctx.lib.dsp_frontend_batch_device(ctx.handle, _dp(samples.contiguous()), _TORCH_DTYPES[samples.dtype], _dp(offsets), None,
                                            _dp(feat_offsets), None, n_utts, max_len, C.byref(p), C.byref(out)))
    return (o["start"], o["end"], o["n_frames"], o["status"], o["stats"], o["energy"][:total_frames],
            o["magnitude"][:total_frames], o["zcr"][:total_frames])


@frontend_batch.register_fake
def _(samples, offsets, feat_offsets, n_utts, max_len, total_frames, frame_length, frame_shift, window, do_endpoint_detection,
      energy_high_ratio, energy_low_ratio, zcr_threshold_ratio):
    i = lambda: samples.new_empty(n_utts, dtype=torch.int32)
    f = lambda: samples.new_empty(total_frames, dtype=torch.float32)
    return i(), i(), i(), i(), samples.new_empty((n_utts, 15), dtype=torch.float32), f(), f(), f()


@torch.library.custom_op(f"{NS}::zscore_fit", mutates_args=(), device_types="cuda")
def zscore_fit(x: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """normalize_features' statistics (feature_extraction.py:171-177): (mean[d], std[d] with 0 -> 1), float64; the
    column sums follow x's layout like NumPy's on x.cpu().numpy() (batch._axis0_is_inner)."""
    assert x.dtype == torch.float64 and x.dim() == 2
    mean, std = _zscore_fit(_bind(x.device), x.contiguous(), _axis0_is_inner(x))
    # the rule zscore_device's std gets from the apply kernel
    return mean, torch.where(std == 0, torch.ones_like(std), std)


@zscore_fit.register_fake
def _(x):
    return x.new_empty(x.shape[1]), x.new_empty(x.shape[1])


@torch.library.custom_op(f"{NS}::zscore_apply", mutates_args=(), device_types="cuda")
def zscore_apply(x: torch.Tensor, mean: torch.Tensor, std: torch.Tensor) -> torch.Tensor:
    """(x - mean) / std in float64 (feature_extraction.py:179); x is float64, or the float32 statistics of the front end."""
    assert x.dim() == 2 and mean.dtype == torch.float64 and std.dtype == torch.float64
    x = x.contiguous()
    if x.dtype == torch.float32:
        return zscore_apply_f32(x, mean.contiguous(), std.contiguous())
    return zscore_device(x, mean, std)[0]


@zscore_apply.register_fake
def _(x, mean, std):
    return x.new_empty(x.shape, dtype=torch.float64)


_knn_cache, _dtw_cache = OrderedDict(), OrderedDict()


def _fitted(cache, key, fit):
    """The handle `cache` holds for `key`, or fit()'s: a call on the same tensors (storage, version, k) does not copy or
    re-pack them again.  A cache keeps the 4 handles fitted last and frees the others."""
    h = cache.get(key)
    if h is None:
        h = cache[key] = fit()
        while len(cache) > 4:
            cache.popitem(last=False)[1].free()
    return h


def _knn_handle(train, labels, k):
    key = (train.data_ptr(), tuple(train.shape), train._version, labels.data_ptr(), labels._version, int(k), train.device.index)
    return _fitted(_knn_cache, key, lambda: DeviceKNN(k, device=train.device).fit(train.contiguous(), labels.contiguous()))


@torch.library.custom_op(f"{NS}::knn_predict", mutates_args=(), device_types="cuda")
def knn_predict(train: torch.Tensor, labels: torch.Tensor, queries: torch.Tensor, k: int) -> torch.Tensor:
    """KNeighborsClassifier(n_neighbors=k).fit(train, labels).predict(queries) (models.py:33-35,52-58): exact float64
    neighbours, vote ties to the smallest label.  train / queries float64 [*, d], labels int32 >= 0 -> int32 [m]."""
    assert train.dtype == torch.float64 and queries.dtype == torch.float64 and labels.dtype == torch.int32
    return _knn_handle(train, labels, k).predict(queries.contiguous())


@knn_predict.register_fake
def _(train, labels, queries, k):
    return queries.new_empty(queries.shape[0], dtype=torch.int32)


@torch.library.custom_op(f"{NS}::knn_topk", mutates_args=(), device_types="cuda")
def knn_topk(train: torch.Tensor, labels: torch.Tensor, queries: torch.Tensor, k: int) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """-> (squared distances f64 [m,k], train row indices i64 [m,k], their labels i32 [m,k]), ties to the lower index."""
    assert train.dtype == torch.float64 and queries.dtype == torch.float64 and labels.dtype == torch.int32
    return _knn_handle(train, labels, k).topk(queries.contiguous())


@knn_topk.register_fake
def _(train, labels, queries, k):
    m = queries.shape[0]
    return (queries.new_empty((m, k)), queries.new_empty((m, k), dtype=torch.int64), queries.new_empty((m, k), dtype=torch.int32))


@torch.library.custom_op(f"{NS}::mfcc_batch", mutates_args=(), device_types="cuda")
def mfcc_batch(samples: torch.Tensor, offsets: torch.Tensor, start: torch.Tensor, end: torch.Tensor, mfcc_offsets: torch.Tensor,
               total_frames: int, frame_length: int, frame_shift: int, n_fft: int, n_mels: int, n_ceps: int, window: int,
               pre_emphasis: float, log_floor: float) -> Tuple[torch.Tensor, torch.Tensor]:
    """MFCC of the segments [start, end) of a packed int16 batch (mfcc_dtw.mfcc_batch, on device tensors; HTK-mel
    filterbank at 44.1 kHz and orthonormal DCT-II from mfcc_dtw).  mfcc_offsets [B+1] are row capacities, e.g.
    plan(offsets, frame_length, frame_shift).feat_offsets.  -> (mfcc f32 [total_frames, n_ceps], n_frames i32 [B]);
    rows of an utterance past its n_frames are zero."""
    if samples.dtype != torch.int16:
        raise ValueError("mfcc_batch takes 16-bit PCM")
    dev = samples.device
    # the tables at DEFAULTS["sample_rate"], which the op does not take (DeviceMFCC has a sample_rate parameter)
    p, fb, dct = _mfcc_setup(dict(DEFAULTS, frame_length=frame_length, frame_shift=frame_shift, n_fft=n_fft, n_mels=n_mels,
                                  n_ceps=n_ceps, pre_emphasis=pre_emphasis, log_floor=log_floor))
    p.window = window                             # an id; the C ABI rejects one outside 0..2
    # zero-filled, as documented above (DeviceMFCC.run leaves the rows past n_frames as they were)
    mfcc = torch.zeros(max(total_frames, 1), n_ceps, dtype=torch.float32, device=dev)
    n_frames = torch.zeros(offsets.numel() - 1, dtype=torch.int32, device=dev)
    _mfcc_device(_bind(dev), samples.contiguous(), offsets.contiguous(), None, start.contiguous(), end.contiguous(), p, fb,
                 dct, mfcc_offsets.contiguous(), mfcc, n_frames)
    return mfcc[:total_frames], n_frames


@mfcc_batch.register_fake
def _(samples, offsets, start, end, mfcc_offsets, total_frames, frame_length, frame_shift, n_fft, n_mels, n_ceps, window,
      pre_emphasis, log_floor):
    return (samples.new_empty((total_frames, n_ceps), dtype=torch.float32),
            samples.new_empty(offsets.shape[0] - 1, dtype=torch.int32))


def _dtw_handle(t_feats, t_offsets, t_labels, k):
    key = (t_feats.data_ptr(), tuple(t_feats.shape), t_feats._version, t_offsets.data_ptr(), t_offsets.numel(),
           t_offsets._version, t_labels.data_ptr(), t_labels._version, int(k), t_feats.device.index)
    return _fitted(_dtw_cache, key, lambda: DeviceDTW(k, device=t_feats.device).fit(
        t_feats.contiguous(), t_offsets.contiguous(), t_labels.contiguous()))


@torch.library.custom_op(f"{NS}::dtw_topk", mutates_args=(), device_types="cuda")
def dtw_topk(t_feats: torch.Tensor, t_offsets: torch.Tensor, t_labels: torch.Tensor, q_feats: torch.Tensor,
             q_offsets: torch.Tensor, k: int) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """k cheapest templates of each query under DTW (mfcc_dtw.DTWClassifier.kneighbors on device tensors): sequences
    are float32 [frames, dim] with int64 offsets [n+1] in frames; -> (cost f64 [nq,k], template index i64 [nq,k],
    label i32 [nq,k]), ties to the lower index, (inf, -1, -1) where fewer than k templates have a finite cost."""
    return _dtw_handle(t_feats, t_offsets, t_labels, k).topk(q_feats.contiguous(), q_offsets.contiguous())


@dtw_topk.register_fake
def _(t_feats, t_offsets, t_labels, q_feats, q_offsets, k):
    nq = q_offsets.shape[0] - 1
    return (q_feats.new_empty((nq, k), dtype=torch.float64), q_feats.new_empty((nq, k), dtype=torch.int64),
            q_feats.new_empty((nq, k), dtype=torch.int32))
