"""torch.library custom ops over the C ABI, for callers whose tensors are already torch CUDA tensors
(BASELINE.json north_star: "a thin ctypes/C-ABI layer, or torch custom ops where tensors are already torch").

    import dsp_audioreclabs_b200.torch_ops            # registers torch.ops.dsp_audioreclabs.*
    plan = torch_ops.plan(offsets, 256, 128)           # host arithmetic: ragged output layout of one batch shape
    start, end, n_frames, status, stats, energy, magnitude, zcr = torch.ops.dsp_audioreclabs.frontend_batch(
        samples, plan.offsets, plan.feat_offsets, plan.n_utts, plan.max_len, plan.total_frames, 256, 128, 1, True, 0.5, 0.1, 1.5)
    qn = torch.ops.dsp_audioreclabs.zscore_apply(stats, mean, std)
    labels = torch.ops.dsp_audioreclabs.knn_predict(train_norm, train_labels, qn, 3)

Each op enqueues libdspfront kernels on torch's CURRENT stream with the tensors' device pointers -- no host copies,
no torch arithmetic on the path -- and has a fake (meta) implementation, so the ops trace under torch.compile /
torch.export as opaque calls.  They are tensor-in / tensor-out mirrors of src/audio_processing.py:336-396 +
src/feature_extraction.py:91-112 (front end), :157-181 (z-score) and src/models.py:52-58 (KNN predict).
"""
import ctypes as C
from collections import OrderedDict
from typing import Tuple

import numpy as np
import torch

from . import _capi
from ._capi import FrontendOutputs, check
from .batch import _axis0_is_inner, default_context, make_params, plan as _host_plan

NS = "dsp_audioreclabs"
_WINDOWS = ("rectangular", "hamming", "hanning")
_TORCH_DTYPES = {torch.int16: _capi.DSP_S16, torch.uint8: _capi.DSP_U8, torch.float32: _capi.DSP_F32, torch.float64: _capi.DSP_F64}


def _dp(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _ctx_for(t):
    ctx = default_context(t.device.index or 0)
    ctx.set_stream(torch.cuda.current_stream(t.device).cuda_stream)
    return ctx


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
    dev = samples.device
    ctx = _ctx_for(samples)
    p = make_params(frame_length, frame_shift, _WINDOWS[window], do_endpoint_detection, energy_high_ratio, energy_low_ratio,
                    zcr_threshold_ratio)
    i32 = dict(dtype=torch.int32, device=dev)
    f32 = dict(dtype=torch.float32, device=dev)
    start, end, n_epd, n_frames, status = (torch.zeros(n_utts, **i32) for _ in range(5))
    stats = torch.zeros(n_utts, 15, **f32)
    energy, magnitude, zcr = (torch.zeros(max(total_frames, 1), **f32) for _ in range(3))
    out = FrontendOutputs(_dp(start), _dp(end), _dp(n_epd), _dp(n_frames), _dp(status), _dp(energy), _dp(magnitude), _dp(zcr),
                          _dp(stats), None, None)
    check(ctx.lib.dsp_frontend_batch_device(ctx.handle, _dp(samples.contiguous()), _TORCH_DTYPES[samples.dtype], _dp(offsets), None,
                                            _dp(feat_offsets), None, n_utts, max_len, C.byref(p), C.byref(out)))
    return start, end, n_frames, status, stats, energy[:total_frames], magnitude[:total_frames], zcr[:total_frames]


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
    ctx = _ctx_for(x)
    pairwise = _axis0_is_inner(x)
    x = x.contiguous()
    n, d = x.shape
    mean = torch.empty(d, dtype=torch.float64, device=x.device)
    std = torch.empty(d, dtype=torch.float64, device=x.device)
    check(ctx.lib.dsp_zscore_device(ctx.handle, _dp(x), n, d, 2 if pairwise else 1, _dp(mean), _dp(std), None))
    return mean, torch.where(std == 0, torch.ones_like(std), std)


@zscore_fit.register_fake
def _(x):
    return x.new_empty(x.shape[1]), x.new_empty(x.shape[1])


@torch.library.custom_op(f"{NS}::zscore_apply", mutates_args=(), device_types="cuda")
def zscore_apply(x: torch.Tensor, mean: torch.Tensor, std: torch.Tensor) -> torch.Tensor:
    """(x - mean) / std in float64 (feature_extraction.py:179); x is float64, or the float32 statistics of the front end."""
    assert x.dim() == 2 and mean.dtype == torch.float64 and std.dtype == torch.float64
    ctx = _ctx_for(x)
    x = x.contiguous()
    n, d = x.shape
    out = torch.empty(n, d, dtype=torch.float64, device=x.device)
    if x.dtype == torch.float32:
        check(ctx.lib.dsp_zscore_apply_f32_device(ctx.handle, _dp(x), n, d, _dp(mean.contiguous()), _dp(std.contiguous()), _dp(out)))
    else:
        assert x.dtype == torch.float64
        m, s = mean.clone(), std.clone()
        check(ctx.lib.dsp_zscore_device(ctx.handle, _dp(x), n, d, 0, _dp(m), _dp(s), _dp(out)))
    return out


@zscore_apply.register_fake
def _(x, mean, std):
    return x.new_empty(x.shape, dtype=torch.float64)


_knn_cache = OrderedDict()


def _knn_handle(train, labels, k):
    """Fitted handles are kept per (storage, version, k): a predict on the same train tensor does not re-pack it."""
    from .device import DeviceKNN
    key = (train.data_ptr(), tuple(train.shape), train._version, labels.data_ptr(), labels._version, int(k), train.device.index)
    knn = _knn_cache.get(key)
    if knn is None:
        knn = DeviceKNN(k, device=train.device).fit(train.contiguous(), labels.contiguous())
        _knn_cache[key] = knn
        while len(_knn_cache) > 4:
            _knn_cache.popitem(last=False)[1].free()
    return knn


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
