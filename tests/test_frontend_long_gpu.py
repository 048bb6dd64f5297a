"""GPU parity of the front end on utterances longer than 65,535 samples, on every kernel route.

The pipelined kernel takes utterances up to 65,535 samples.  Above that, route_frontend (csrc/capi.cu) routes a batch by
its longest utterance and its layout: the shared-memory-resident build of frontend_pcm_kernel for packed (any alignment)
batches, a streaming build for batches whose utterances all start on 16-byte boundaries, and the float64 replay kernel
for everything longer than what those builds fit in shared memory (or longer than 2^20 samples, or not int16 mono).

Bars as in test_frontend_gpu.py: start / end / frame counts / zero-crossing counts exact, EPD energies to 1e-12,
energy and magnitude to 1e-5, statistics by assert_stats_close, float64 outputs bit-identical to NumPy.  The route an
utterance took is pinned with the DSP_UTT_EXACT status bit (0x100, set when the float64 replay produced the result).
"""
import os
import subprocess
import sys

import numpy as np
import pytest

from test_frontend_gpu import RTOL_EPD, RTOL_F32, assert_stats_close

pytestmark = pytest.mark.gpu

EXACT = 0x100
PIPE = 10                       # pcm_variant of the pipelined kernel (frontend_pcm.cu kVariants has 10 builds)
FAST_MAX_LEN = 1 << 20          # capi.cu kFastMaxLen
PIPE_MAX_LEN = 65535            # frontend_pipe.cu pipe_kernel_plan
STATIC_SMEM = 128               # frontend_pcm_kernel's static shared memory (s_prof[16]), ptxas -v
STREAM_MAIN_WARPS = {1: 3, 2: 3, 3: 3, 4: 6, 5: 6, 6: 4, 7: 4}      # frontend_pcm.cu kVariants: threads / 32 - stats warps
GEOMS = [(256, 128), (1102, 441)]
WINDOWS = ("rectangular", "hamming", "hanning")
SR = 44100
# EPD energies on DC-heavy content (mean code near +29,000 or -31,900): here the ORACLE is the inexact side.  NumPy
# subtracts a mean of ~0.9 from samples of ~0.9 in float64 and loses the leading bits, so its energies sit up to 2.0e-12
# from the exact rational value (near_min at 65,535 samples; 9e-13 for dc at 90 k; within 8e-16 on plain speech),
# while the fast kernels' integer formulation stays close to exact.  Every integer output is still compared exactly.
RTOL_EPD_DC = 5e-12


# ---- shared-memory limits of frontend_pcm_kernel ------------------------------------------------------------------
def _a16(x):
    return (x + 15) & ~15


def _frame_count(n, fl, fs):                     # kernels.cuh frame_count_host_device
    if n <= 0:
        return 0
    return min((n + fs - 1) // fs, (max(n - fl, 0) + fs - 1) // fs + 1)


def pcm_smem(n, fl, fs, resident):
    """Dynamic shared memory of frontend_pcm_kernel for a batch whose longest utterance has n samples: make_layout
    (csrc/frontend_pcm.cu:42) with cap_samples and cap_frames as route_frontend (csrc/capi.cu) derives them."""
    cs = (max(n, 1) + 63) // 64 * 64
    cf = max(_frame_count(n, fl, fs), 1)
    o = _a16(2 * cs + 32) if resident else 0
    o += _a16(4 * (cs // 32 + 4))
    o += _a16(max(12 * (cs // 64), 12 * cf))
    o += _a16(8 * cf) + _a16(4 * cf) + _a16(4 * fl)
    return o + 3 * 256 * 4 + 3 * 64 * 4 + 64 * 8 + 384


_LIMITS = {}


def pcm_limit(fl, fs, resident, static=STATIC_SMEM):
    """Longest utterance the resident / streaming build takes: dynamic + static shared memory within the device's
    opt-in per-block maximum (static=0: the dynamic layout alone fills it)."""
    key = (fl, fs, resident, static)
    if key not in _LIMITS:
        import torch
        cap = torch.cuda.get_device_properties(0).shared_memory_per_block_optin - static
        lo, hi = 1, FAST_MAX_LEN
        while lo < hi:
            m = (lo + hi + 1) // 2
            lo, hi = (m, hi) if pcm_smem(m, fl, fs, resident) <= cap else (lo, m - 1)
        _LIMITS[key] = lo
    return _LIMITS[key]


def replayed_route(n, fl, fs, aligned):
    """True when the automatic route sends a batch whose longest utterance has n samples to the float64 replay."""
    if n <= PIPE_MAX_LEN:
        return False
    return n > FAST_MAX_LEN or n > pcm_limit(fl, fs, resident=not aligned)


# ---- signals ------------------------------------------------------------------------------------------------------
def _gap(rng, n, level=20.0, dc=300.0):
    return rng.standard_normal(n) * level + dc


def speech_f(n, seed):
    """float64 PCM-scale signal: synth clips (0.3-1.0 s) separated by quiet gaps (0.1-0.4 s), quiet at both ends."""
    from oracle import synth
    rng = np.random.default_rng(seed)
    tail = min(int(0.12 * SR), n // 8)
    parts, tot, i = [], 0, 0
    while tot < n - tail:
        g = _gap(rng, int(rng.uniform(0.1, 0.4) * SR))
        c = synth.utterance_pcm(i, int(rng.uniform(0.3, 1.0) * SR), seed0=seed).astype(np.float64)
        parts += [g, c]
        tot += len(g) + len(c)
        i += 1
    body = np.concatenate(parts)[:n - tail]
    return np.concatenate([body, _gap(rng, tail)])


def to_pcm(x):
    return np.clip(np.round(x), -32768, 32767).astype(np.int16)


_SIG = {}


def signal(kind, n, seed=1):
    """int16 test signals (cached):
    speech      clips in quiet gaps
    dc          speech at ~5 % of full scale on a DC offset of 29,000: sum k ~ 2.9e4 n (32-bit partials wrap)
    near_min    content between -32,768 and ~-31,000: sum k within a few percent of INT32_MIN at 65,535 samples
    clipped     speech driven into both rails (+32767 / -32768)
    tail_burst  digital silence with a burst in the last 0.2 s (endpoints near the end, many equal EPD energies)"""
    key = (kind, n, seed)
    if key in _SIG:
        return _SIG[key]
    if kind == "speech":
        x = to_pcm(speech_f(n, seed))
    elif kind == "dc":
        x = to_pcm(speech_f(n, seed) * (1638.0 / 20000.0) + 29000.0)
    elif kind == "near_min":
        x = to_pcm(np.clip(speech_f(n, seed) * (900.0 / 20000.0) - 31900.0, -32768, -31000))
    elif kind == "clipped":
        x = to_pcm(speech_f(n, seed) * 4.0)
    elif kind == "tail_burst":
        from oracle import synth
        x = np.zeros(n, np.int16)
        m = min(int(0.2 * SR), n)
        x[n - m:] = synth.utterance_pcm(3, m, seed0=seed)
    else:
        raise ValueError(kind)
    _SIG[key] = x
    return x


_REF = {}


def oracle(kind, n, fl, fs, win, seed=1):
    """NumPy oracle per (signal, geometry, window), cached for the module."""
    from oracle import frontend_oracle as fo
    key = (kind, n, seed, fl, fs, win)
    if key not in _REF:
        _REF[key] = fo.frontend_utterance(signal(kind, n, seed), fl, fs, win)
    return _REF[key]


LEAD = ("speech", 4099, 7)      # a short first utterance: 4,099 = 8 * 512 + 3 puts the next start 3 samples past 16 bytes


def run_batch(ctx, items, fl, fs, win, aligned, variant=-1):
    """items: (kind, n, seed) triples.  Packed CSR (arbitrary starts) or pack_aligned (16-byte starts + lengths)."""
    from dsp_audioreclabs_b200 import batch
    utts = [signal(*it) for it in items]
    if aligned:
        s, o, l = batch.pack_aligned(utts)
        assert np.all(o % 8 == 0)
    else:
        l = None
        o = np.zeros(len(utts) + 1, np.int64)
        np.cumsum([len(u) for u in utts], out=o[1:])
        s = np.concatenate(utts)
    ctx.set_tuning("pcm_variant", variant)
    try:
        return batch.frontend_batch(s, o, fl, fs, win, emit_epd_lists=True, lengths=l, ctx=ctx)
    finally:
        ctx.set_tuning("pcm_variant", -1)


def check_utt(res, b, r, what, rtol_epd=RTOL_EPD):
    assert (int(res.status[b]) & 0xff) == 0, (what, int(res.status[b]))
    assert (int(res.start[b]), int(res.end[b])) == (r["start"], r["end"]), what
    assert int(res.n_frames[b]) == r["n_frames"] and int(res.n_epd_frames[b]) == r["n_epd_frames"], what
    el, zl = res.epd_lists(b)
    assert np.array_equal(zl.astype(np.float64), r["zcr_list"]), what
    assert np.allclose(el, r["energy_list"], rtol=rtol_epd, atol=0), (what, float(np.max(np.abs(el - r["energy_list"]) / np.maximum(r["energy_list"], 1e-300))))
    e, m, z = res.frames(b)
    assert np.array_equal(z.astype(np.float64), r["zcr"]), what
    assert np.allclose(e, r["energy"], rtol=RTOL_F32, atol=0), what
    assert np.allclose(m, r["magnitude"], rtol=RTOL_F32, atol=0), what
    assert_stats_close(res.stats[b], r["stats"], r)


def check_batch(res, items, fl, fs, win, what):
    for b, it in enumerate(items):
        check_utt(res, b, oracle(*it[:2], fl, fs, win, seed=it[2]), (what, it),
                  RTOL_EPD_DC if it[0] in ("dc", "near_min") else RTOL_EPD)


# ---- 1. length sweep across every route boundary ------------------------------------------------------------------
SWEEP = ["64k-1", "64k", "64k+1", "resident", "resident+1", "resident-dyn", "200k", "stream", "stream+1", "stream-dyn",
         "2^20", "2^20+1", "3M"]


def sweep_length(name, fl, fs):
    return {"64k-1": 65535, "64k": 65536, "64k+1": 65537, "resident": pcm_limit(fl, fs, True),
            "resident+1": pcm_limit(fl, fs, True) + 1, "resident-dyn": pcm_limit(fl, fs, True, static=0),
            "200k": 200_000, "stream": pcm_limit(fl, fs, False), "stream+1": pcm_limit(fl, fs, False) + 1,
            "stream-dyn": pcm_limit(fl, fs, False, static=0), "2^20": FAST_MAX_LEN, "2^20+1": FAST_MAX_LEN + 1,
            "3M": 3_000_000}[name]


@pytest.mark.parametrize("aligned", [False, True], ids=["packed", "aligned"])
@pytest.mark.parametrize("name", SWEEP)
@pytest.mark.parametrize("fl,fs", GEOMS)
def test_length_sweep_across_route_boundaries(ctx, fl, fs, name, aligned):
    """A short utterance then a long one.  Packed, the long one starts 3 samples past a 16-byte boundary; aligned, it
    starts on one.  Every result meets the oracle's bars, and the batch takes the route its longest utterance
    selects: a fast kernel (nothing replayed) up to and including each limit, the float64 replay above it.
    '-dyn' is the longest utterance whose dynamic layout alone fits the opt-in maximum: with the kernel's static
    shared memory on top it does not fit, and the call must still succeed (on the replay).  Where the static 128 B
    do not move the limit (1102/441 resident: 95,360 either way) '-dyn' is the same length as the limit itself."""
    n = sweep_length(name, fl, fs)
    win = WINDOWS[(SWEEP.index(name) + fl) % 3]
    items = [LEAD, ("speech", n, 11)]
    res = run_batch(ctx, items, fl, fs, win, aligned)
    replayed = (res.status & EXACT) != 0
    if replayed_route(n, fl, fs, aligned):
        assert replayed.all(), (n, res.status)
    else:
        assert not replayed.any(), (n, res.status)
    check_batch(res, items, fl, fs, win, (fl, fs, n, aligned))
    ref = oracle("speech", n, fl, fs, win, seed=11)
    assert 0 < ref["start"] and ref["end"] < n          # the endpoints really trim


# ---- 2. every build, forced ---------------------------------------------------------------------------------------
def dc_overflow_length(main_warps, dc=29000):
    """Length at which one main warp's share of sum k exceeds 2^31 by 20 % for the 'dc' signal."""
    return int(1.2 * main_warps * 2 ** 31 / dc)


SETS = {"90k": [("speech", 90_000, 21), ("dc", 90_000, 22), ("speech", 20_011, 23)],
        "300k": [("speech", 300_000, 24), ("dc", 300_000, 25), ("speech", 33_333, 26)]}


@pytest.mark.parametrize("size", ["90k", "300k", "dc_overflow"])
@pytest.mark.parametrize("variant", list(range(PIPE + 1)))
def test_every_build_forced(ctx, variant, size):
    """pcm_variant forces one build: 0, 8, 9 resident (packed input), 1-7 streaming (aligned input), 10 the pipelined
    kernel, which does not take these lengths and falls back to build 0.  A build runs a batch it fits (nothing
    replayed) and hands one it does not fit to the float64 replay (everything replayed).  dc_overflow: for every
    streaming build, a DC-heavy utterance long enough that one main warp's share of sum k exceeds 2^31."""
    fl, fs = 256, 128
    win = WINDOWS[variant % 3]
    stream = variant in STREAM_MAIN_WARPS
    if size == "dc_overflow":
        if not stream:
            pytest.skip("the resident builds hold at most ~95 k samples: their per-warp partials stay below 2^31")
        n = dc_overflow_length(STREAM_MAIN_WARPS[variant])
        assert n <= pcm_limit(fl, fs, False)
        items = [("dc", n, 30 + variant), ("speech", 12_345, 27)]
    else:
        items = SETS[size]
    n = max(it[1] for it in items)
    res = run_batch(ctx, items, fl, fs, win, aligned=stream, variant=variant)
    fits = n <= pcm_limit(fl, fs, resident=not stream)
    replayed = (res.status & EXACT) != 0
    assert (not replayed.any()) if fits else replayed.all(), (variant, size, res.status)
    check_batch(res, items, fl, fs, win, (variant, size))


# ---- 3. loud and DC-heavy long signals ----------------------------------------------------------------------------
LOUD = [("dc", 90_000), ("dc", 540_000), ("near_min", 65535), ("near_min", 65536), ("clipped", 65536),
        ("clipped", 200_000), ("tail_burst", 65536), ("tail_burst", 200_000)]


@pytest.mark.parametrize("aligned", [False, True], ids=["packed", "aligned"])
@pytest.mark.parametrize("kind,n", LOUD)
@pytest.mark.parametrize("fl,fs", GEOMS)
def test_loud_and_dc_heavy_signals(ctx, fl, fs, kind, n, aligned):
    win = WINDOWS[(n + fl) % 3]
    x = signal(kind, n, 5)
    if kind == "near_min":
        assert x.max() <= -31000 and x.min() == -32768
        assert abs(int(x.astype(np.int64).sum())) > 0.95 * 2 ** 31 * n / 65536
    if kind == "clipped":
        assert x.max() == 32767 and x.min() == -32768
    items = [LEAD, (kind, n, 5)]
    res = run_batch(ctx, items, fl, fs, win, aligned)
    if replayed_route(n, fl, fs, aligned):
        assert ((res.status & EXACT) != 0).all()
    check_batch(res, items, fl, fs, win, (kind, n, aligned))


# ---- 4. mixed batches ---------------------------------------------------------------------------------------------
def short_items(seed=40):
    from oracle import synth
    lens = synth.ragged_lengths(40, 0.3, 1.2, seed=seed)
    return [("speech", int(n), 100 + i) for i, n in enumerate(lens)]


def _same_ints(a, b, i, j, what):
    for name in ("start", "end", "n_frames", "n_epd_frames"):
        assert int(getattr(a, name)[i]) == int(getattr(b, name)[j]), (what, name)
    assert (int(a.status[i]) & 0xff) == (int(b.status[j]) & 0xff), what
    assert np.array_equal(a.frames(i)[2], b.frames(j)[2]), what
    assert np.array_equal(a.epd_lists(i)[1], b.epd_lists(j)[1]), what
    assert np.allclose(a.epd_lists(i)[0], b.epd_lists(j)[0], rtol=2 * RTOL_EPD, atol=0), what    # each within 1e-12 of exact
    for x, y in zip(a.frames(i)[:2], b.frames(j)[:2]):
        assert np.allclose(x, y, rtol=2e-6, atol=0), what
    for g in range(3):
        x, y = a.stats[i][5 * g:5 * g + 5], b.stats[j][5 * g:5 * g + 5]
        assert np.allclose(x, y, rtol=2e-6, atol=2e-6 * float(np.abs(y).max())), (what, g)


@pytest.mark.parametrize("aligned", [False, True], ids=["packed", "aligned"])
@pytest.mark.parametrize("long_n", [90_000, 200_000])
def test_mixed_batch_long_utterance_moves_the_short_ones(ctx, long_n, aligned):
    """40 short utterances alone run on the pipelined kernel; with one long utterance among them the whole batch runs
    on the resident, streaming or replay kernel.  The short results still meet the oracle's bars, their integer
    outputs equal those of the batch without the long one, and their fp32 outputs agree to 2e-6."""
    fl, fs, win = 1102, 441, "hamming"
    shorts = short_items()
    pos = 17
    items = shorts[:pos] + [("speech", long_n, 99)] + shorts[pos:]
    alone = run_batch(ctx, shorts, fl, fs, win, aligned)
    assert not ((alone.status & EXACT) != 0).any()
    mixed = run_batch(ctx, items, fl, fs, win, aligned)
    replayed = (mixed.status & EXACT) != 0
    assert replayed.all() if replayed_route(long_n, fl, fs, aligned) else not replayed.any()
    check_batch(mixed, items, fl, fs, win, ("mixed", long_n, aligned))
    for j in range(len(shorts)):
        _same_ints(mixed, alone, j + (j >= pos), j, ("mixed vs alone", long_n, aligned, j))


# ---- 5. host chunking ---------------------------------------------------------------------------------------------
def chunk_items():
    shorts = short_items()
    return shorts[:10] + [("speech", 600_000, 61)] + shorts[10:25] + [("speech", 200_000, 99), ("dc", 600_000, 62)] \
        + shorts[25:] + [("speech", 600_000, 63)]


_CHILD = """
import sys
import numpy as np
sys.path[:0] = [{tests!r}, {root!r}]
import test_frontend_long_gpu as t
from dsp_audioreclabs_b200 import batch
res = t.run_batch(batch.default_context(0), t.chunk_items(), 1102, 441, "hanning", aligned=False)
np.savez({out!r}, **{{k: getattr(res, k) for k in ("start", "end", "n_epd_frames", "n_frames", "status", "energy",
    "magnitude", "zcr", "stats", "feat_offsets", "epd_offsets", "epd_energy", "epd_zcr")}})
"""


def test_host_chunks_smaller_than_one_utterance(tmp_path):
    """DSP_HOST_CHUNK_MB=1 (read once per process, so in a child): every 600 k utterance exceeds a staging chunk and
    goes up alone; the short ones are grouped around them.  Every result meets the oracle's bars."""
    from dsp_audioreclabs_b200.batch import FrontendResult
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = str(tmp_path / "chunked.npz")
    code = _CHILD.format(tests=os.path.join(root, "tests"), root=root, out=out)
    r = subprocess.run([sys.executable, "-c", code], cwd=str(tmp_path), capture_output=True, text=True,
                       env=dict(os.environ, DSP_HOST_CHUNK_MB="1"), timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    with np.load(out) as z:
        res = FrontendResult(**{k: z[k] for k in z.files})
    items = chunk_items()
    assert len(res) == len(items)
    check_batch(res, items, 1102, 441, "hanning", "chunked")


# ---- 6. device API ------------------------------------------------------------------------------------------------
def test_device_api_long_aligned_batch_equals_host(ctx):
    """DeviceFrontend derives the 16-byte alignment from the tensor's pointer and runs the streaming build: its
    results equal the host API's on the same aligned layout.  A slot of the ragged per-frame buffers is sized for the
    untrimmed frame count and only its first n_frames entries are written, so the sequences compare per utterance."""
    import torch
    from dsp_audioreclabs_b200 import batch
    from dsp_audioreclabs_b200.device import DeviceFrontend
    fl, fs, win = 256, 128, "hanning"
    items = [("speech", 300_000, 71), LEAD, ("dc", dc_overflow_length(3), 72), ("speech", 70_001, 73)]
    s, o, l = batch.pack_aligned([signal(*it) for it in items])
    host = batch.frontend_batch(s, o, fl, fs, win, emit_epd_lists=True, lengths=l, ctx=ctx)
    assert not ((host.status & EXACT) != 0).any()
    check_batch(host, items, fl, fs, win, "host")
    dev = DeviceFrontend(o, fl, fs, win, emit_epd_lists=True, lengths=l, ctx=ctx)
    samples = torch.from_numpy(s).cuda()
    dev.run(samples)
    torch.cuda.synchronize()
    assert dev.params.aligned16 == 1
    got = batch.FrontendResult(**{k: getattr(dev, k).cpu().numpy() for k in (
        "start", "end", "n_epd_frames", "n_frames", "status", "stats", "energy", "magnitude", "zcr", "epd_energy",
        "epd_zcr")}, feat_offsets=dev.h_feat_offsets, epd_offsets=dev.h_epd_offsets)
    for name in ("start", "end", "n_epd_frames", "n_frames", "status", "stats"):
        assert np.array_equal(getattr(got, name), getattr(host, name)), name
    for b in range(len(items)):
        for x, y in zip(got.frames(b) + got.epd_lists(b), host.frames(b) + host.epd_lists(b)):
            assert np.array_equal(x, y), b
    check_batch(got, items, fl, fs, win, "device")


# ---- 7. long non-int16 inputs: the float64 replay ------------------------------------------------------------------
def float_signal(n, seed):
    """float64 signal that is not a PCM grid: NumPy's summation order decides the last bits of the mean."""
    rng = np.random.default_rng(seed)
    return speech_f(n, seed) * (0.7 / 32768.0) + 0.0123 + rng.standard_normal(n) * 1e-4


@pytest.mark.parametrize("n", [300_001, FAST_MAX_LEN])
def test_per_call_float64_long_signals(ctx, n):
    """preprocess (modes 0, 1, 2) and endpoint_detection of long float64 signals are bit-identical to NumPy: the mean
    is one pairwise tree over more than 2,048 leaves (frontend_exact.cu block_np_sum's single-thread branch)."""
    from dsp_audioreclabs_b200 import batch
    from oracle import frontend_oracle as fo
    assert n // 128 > 2048
    x = float_signal(n, 81)
    assert np.array_equal(batch.preprocess(x, 0, ctx=ctx), x - np.mean(x))
    assert np.array_equal(batch.preprocess(x, 1, ctx=ctx), fo.normalize_audio(x))
    z = batch.preprocess(x, 2, ctx=ctx)
    assert np.array_equal(z, fo.preprocess(x))
    for fl, fs in GEOMS:
        s, e, el, zl = batch.endpoint_detection(z, fl, fs, ctx=ctx)
        rs, re_, rel, rzl = fo.endpoint_detection(z, fl, fs)
        assert (s, e) == (rs, re_) and 0 < s and e < n
        assert np.array_equal(el, rel) and np.array_equal(zl, rzl)


def _check_f64(res, b, r, what):
    assert (int(res.status[b]) & 0xff) == 0 and (int(res.status[b]) & EXACT), what
    assert (int(res.start[b]), int(res.end[b]), int(res.n_frames[b])) == (r["start"], r["end"], r["n_frames"]), what
    el, zl = res.epd_lists(b)
    assert np.array_equal(el, r["energy_list"]) and np.array_equal(zl, r["zcr_list"]), what
    for got, key in zip(res.frames(b), ("energy", "magnitude", "zcr")):
        assert np.array_equal(got, r[key]), (what, key)
    assert np.array_equal(res.stats[b], r["stats"]), what


@pytest.mark.parametrize("kind", ["float32", "float64", "uint8", "stereo_int16"])
def test_long_non_int16_batches_bit_identical(ctx, kind):
    """Only the float64 replay serves these: frontend_batch(float64_outputs=True) equals the NumPy path bit for bit."""
    from dsp_audioreclabs_b200 import batch
    from oracle import frontend_oracle as fo
    fl, fs, win = 1102, 441, "hamming"
    lens = [210_000, 700_001, 333_333]
    utts, refs = [], []
    for i, n in enumerate(lens):
        f = float_signal(n, 90 + i)
        if kind == "float32":
            u = f.astype(np.float32)
            x = u.astype(np.float64)
        elif kind == "float64":
            u = x = f
        elif kind == "uint8":
            u = np.clip(np.round(f * 128.0 / 0.72 + 128.0), 0, 255).astype(np.uint8)
            x = fo.pcm_to_float(u)
        else:
            other = to_pcm(speech_f(n, 190 + i))
            u = np.stack([to_pcm(f * 32768.0), other], axis=1).ravel()
            x = fo.stereo_to_mono(fo.pcm_to_float(u))
        utts.append(u)
        refs.append(fo.frontend_utterance(x, fl, fs, win))
    off = np.zeros(len(utts) + 1, np.int64)
    np.cumsum([len(u) for u in utts], out=off[1:])
    res = batch.frontend_batch(np.concatenate(utts), off, fl, fs, win, emit_epd_lists=True, float64_outputs=True,
                               channels=2 if kind == "stereo_int16" else 1, ctx=ctx)
    for b, r in enumerate(refs):
        _check_f64(res, b, r, (kind, b))
