"""MFCC + DTW template matching on the GPU (BASELINE config 5; SURVEY.md section 8 rows a11 / f4).

The reference has no spectral features and no template matching (compare_feature_methods.py compares statistical
with zero-padded sequence features), so this variant is self-specified: same pre-processing, endpoints and framing
rule as the reference's front end, then the textbook MFCC chain and classic DTW.  The tables the kernel consumes
(mel filterbank, DCT matrix) are built here on the host; the arithmetic per sample runs in csrc/mfcc_dtw.cu.
"""
import ctypes as C
import functools

import numpy as np

from . import _capi
from .batch import _host_ctx, _ptr, _window_id, check

DEFAULTS = dict(frame_length=1102, frame_shift=441, n_fft=2048, n_mels=26, n_ceps=13, pre_emphasis=0.97,
                log_floor=1e-10, sample_rate=44100, window_type="hamming")


def mel_filterbank(n_mels, n_fft, sample_rate):
    """Triangular filters on the HTK mel scale 2595 log10(1 + f / 700) between 0 and sample_rate / 2, corner
    points at FFT bin floor((n_fft + 1) f / sample_rate): float32 [n_mels, n_fft // 2 + 1]."""
    mel_hi = 2595.0 * np.log10(1.0 + (sample_rate / 2.0) / 700.0)
    hz = 700.0 * (10.0 ** (np.linspace(0.0, mel_hi, n_mels + 2) / 2595.0) - 1.0)
    corner = np.floor((n_fft + 1) * hz / sample_rate).astype(np.int64)
    b = np.arange(n_fft // 2 + 1)[None, :]
    lo, ce, hi = corner[:-2, None], corner[1:-1, None], corner[2:, None]
    with np.errstate(divide="ignore", invalid="ignore"):
        up = (b - lo) / (ce - lo)
        down = (hi - b) / (hi - ce)
    fb = np.where((b >= lo) & (b < ce), up, 0.0) + np.where((b >= ce) & (b < hi), down, 0.0)
    return np.ascontiguousarray(fb, dtype=np.float32)


def dct_matrix(n_ceps, n_mels):
    """Rows of the orthonormal DCT-II: float32 [n_ceps, n_mels]."""
    k = np.arange(n_ceps)[:, None]
    m = np.arange(n_mels)[None, :]
    d = np.sqrt(2.0 / n_mels) * np.cos(np.pi * k * (2 * m + 1) / (2.0 * n_mels))
    d[0] /= np.sqrt(2.0)
    return np.ascontiguousarray(d, dtype=np.float32)


@functools.lru_cache(maxsize=8)
def _mfcc_tables(n_fft, n_mels, n_ceps, sample_rate):
    fb, dct = mel_filterbank(n_mels, n_fft, sample_rate), dct_matrix(n_ceps, n_mels)
    fb.flags.writeable = dct.flags.writeable = False          # shared by every caller with these parameters
    return fb, dct


def _mfcc_setup(p):
    """(MfccParams, filterbank, dct) of a parameter dict with the keys of DEFAULTS; an unknown window type raises
    ValueError.  The tables are built once per (n_fft, n_mels, n_ceps, sample_rate)."""
    cp = _capi.MfccParams(p["frame_length"], p["frame_shift"], p["n_fft"], p["n_mels"], p["n_ceps"],
                          _window_id(p["window_type"]), p["pre_emphasis"], p["log_floor"])
    return (cp,) + _mfcc_tables(p["n_fft"], p["n_mels"], p["n_ceps"], p["sample_rate"])


def mfcc_batch(samples, offsets, start, end, lengths=None, ctx=None, **params):
    """MFCC frames of the segments [start[b], end[b]) of a packed int16 batch (the endpoints come from
    batch.frontend_batch).  Returns (mfcc float32 [total_frames, n_ceps], mfcc_offsets int64 [B + 1])."""
    p = dict(DEFAULTS); p.update(params)
    ctx = _host_ctx(ctx)
    samples = np.ascontiguousarray(samples)
    if samples.dtype != np.int16:
        raise ValueError("mfcc_batch takes 16-bit PCM")
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    b = len(offsets) - 1
    start = np.ascontiguousarray(start, dtype=np.int32)
    end = np.ascontiguousarray(end, dtype=np.int32)
    if lengths is not None:
        lengths = np.ascontiguousarray(lengths, dtype=np.int32)
    cp, fb, dct = _mfcc_setup(p)
    lib = ctx.lib
    # frame_signal's frame count in closed form (dsp_frame_count; src/audio_processing.py:320-331), vectorised
    seg = np.maximum(end.astype(np.int64) - start.astype(np.int64), 0)
    fl_, fs_ = int(p["frame_length"]), int(p["frame_shift"])
    nfr = np.where(seg > 0, np.minimum(-(-seg // fs_), -(-np.maximum(seg - fl_, 0) // fs_) + 1), 0).astype(np.int64)
    mo = np.zeros(b + 1, dtype=np.int64)
    np.cumsum(nfr, out=mo[1:])
    out = np.zeros((int(mo[-1]), p["n_ceps"]), dtype=np.float32)
    got = np.zeros(b, dtype=np.int32)
    check(lib.dsp_mfcc_batch_host(ctx.handle, _ptr(samples), _ptr(offsets), _ptr(lengths), _ptr(start), _ptr(end), b,
                                  C.byref(cp), _ptr(fb), _ptr(dct), _ptr(mo), _ptr(out), _ptr(got)))
    assert np.array_equal(got, nfr)
    return out, mo


def pack_sequences(seqs, dim=None):
    """[(frames_i, dim)] -> (float32 [sum frames, dim], int64 offsets)."""
    if dim is None:
        dim = seqs[0].shape[1] if len(seqs) else 1
    off = np.zeros(len(seqs) + 1, dtype=np.int64)
    np.cumsum([len(s) for s in seqs], out=off[1:])
    flat = np.zeros((int(off[-1]), dim), dtype=np.float32)
    for s, o in zip(seqs, off[:-1]):
        flat[o:o + len(s)] = s
    return flat, off


class DTWClassifier:
    """k-nearest templates under the DTW cost, majority vote (ties to the smallest label), one CTA per pair."""

    def __init__(self, n_neighbors=1, ctx=None, index_base=0):
        self.k = int(n_neighbors)
        self.ctx = _host_ctx(ctx)
        self.index_base = int(index_base)

    def fit(self, template_seqs, labels):
        self.t_flat, self.t_off = pack_sequences(template_seqs)
        self.classes_, enc = np.unique(np.asarray(labels), return_inverse=True)
        self.t_lab = np.ascontiguousarray(enc, dtype=np.int32)
        return self

    def kneighbors(self, query_seqs, return_matrix=False):
        q_flat, q_off = pack_sequences(query_seqs, self.t_flat.shape[1])
        nq, nt, k = len(query_seqs), len(self.t_lab), self.k
        cost = np.zeros((nq, nt), dtype=np.float32) if return_matrix else None
        nc = np.zeros((nq, k), dtype=np.float64)
        ni = np.zeros((nq, k), dtype=np.int64)
        nl = np.zeros((nq, k), dtype=np.int32)
        check(self.ctx.lib.dsp_dtw_topk_host(self.ctx.handle, _ptr(q_flat), _ptr(q_off), nq, _ptr(self.t_flat), _ptr(self.t_off),
                                             _ptr(self.t_lab), nt, self.t_flat.shape[1], k, self.index_base, _ptr(cost),
                                             _ptr(nc), _ptr(ni), _ptr(nl)))
        return (nc, ni, nl, cost) if return_matrix else (nc, ni, nl)

    def predict(self, query_seqs):
        _, _, nl = self.kneighbors(query_seqs)
        out = np.empty(len(nl), dtype=np.int64)
        for i, row in enumerate(nl):
            cnt = np.bincount(row[row >= 0], minlength=len(self.classes_))
            out[i] = int(np.argmax(cnt))
        return self.classes_[out]
