"""Host dispatch (csrc/capi.cu): the kernel route one call takes and the launches it counts.

Front end: every route of DESIGN §3.1b -- the pipelined kernel, the automatic builds 0 (packed) and 2 (16-byte aligned),
every build forced with pcm_variant, a forced 10 that does not fit the pipelined kernel, and the float64 replay for
batches no fast kernel takes.  A fast kernel counts two launches (itself and the replay of the utterances it flagged)
and replays nothing on these signals; the replay alone counts one and sets DSP_UTT_EXACT (0x100) on every utterance.

KNN: every scan kind (knn.last_stats()[1]) and each form of the tensor-core filter call (tile pruning off / automatic /
always, bounded), with the launches one top-k call counts: bench.py reports them as gpu_launches."""
import numpy as np
import pytest

from test_frontend_long_gpu import EXACT, PIPE, signal
from test_knn_routes_gpu import Env

pytestmark = pytest.mark.gpu

FL, FS = 256, 128
# Packed, LEAD puts the next start 3 samples past a 16-byte boundary: the host API then sees a batch that is not aligned16.
LEAD = ("speech", 4099, 7)
SHORT = [LEAD, ("speech", 20_011, 1), ("speech", 16_000, 2)]
LONG = [LEAD, ("speech", 90_000, 21), ("speech", 20_011, 23)]     # above the pipelined kernel, within build 0 (94,080)
LONGER = [LEAD, ("speech", 300_000, 24)]                          # beyond build 0, within build 2 (557,632)
RESIDENT_MISS = [LEAD, ("speech", 100_000, 4)]                    # packed, beyond build 0's shared memory
OVERSIZE = [LEAD, ("speech", (1 << 20) + 1, 6)]                   # beyond the fast kernels' exact-integer bounds
STREAM_BUILDS = range(1, 8)


def front(ctx, items, aligned=False, variant=-1, dtype=np.int16, **kw):
    """One frontend_batch call -> (launches it counted, replay bit of every utterance)."""
    from dsp_audioreclabs_b200 import batch
    utts = [signal(*it).astype(dtype) for it in items]
    if aligned:
        s, o, l = batch.pack_aligned(utts)
    else:
        l = None
        o = np.zeros(len(utts) + 1, np.int64)
        np.cumsum([len(u) for u in utts], out=o[1:])
        s = np.concatenate(utts)
    ctx.set_tuning("pcm_variant", variant)
    try:
        before = ctx.launch_count
        res = batch.frontend_batch(s, o, FL, FS, "hamming", lengths=l, ctx=ctx, **kw)
        return ctx.launch_count - before, (res.status & EXACT) != 0
    finally:
        ctx.set_tuning("pcm_variant", -1)


FAST = [("pipe", SHORT, False, -1), ("pipe aligned", SHORT, True, -1), ("build 0", LONG, False, -1),
        ("build 2", LONGER, True, -1), ("forced 10", SHORT, False, PIPE), ("forced 10 falls back to build 0", LONG, False, PIPE),
        ("forced 10 falls back to build 0, aligned", LONG, True, PIPE)]
FAST += [(f"forced {v}", LONG, v in STREAM_BUILDS, v) for v in range(PIPE)]


@pytest.mark.parametrize("name,items,aligned,variant", FAST, ids=[f[0] for f in FAST])
def test_frontend_fast_routes(ctx, name, items, aligned, variant):
    launches, replayed = front(ctx, items, aligned, variant)
    assert launches == 2, name
    assert not replayed.any(), (name, replayed)


REPLAY = [("beyond build 0's shared memory", RESIDENT_MISS, {}), ("over 2^20 samples", OVERSIZE, {}),
          ("force_exact", SHORT, {"force_exact": True}), ("float64 outputs", SHORT, {"float64_outputs": True}),
          ("float32 input", SHORT, {"dtype": np.float32}), ("float64 input", SHORT, {"dtype": np.float64}),
          ("forced build 0 beyond its shared memory", RESIDENT_MISS, {"variant": 0})]


@pytest.mark.parametrize("name,items,kw", REPLAY, ids=[r[0] for r in REPLAY])
def test_frontend_replay_routes(ctx, name, items, kw):
    launches, replayed = front(ctx, items, **kw)
    assert launches == 1, name
    assert replayed.all(), (name, replayed)


def test_frontend_stereo_takes_the_replay(ctx):
    from dsp_audioreclabs_b200 import batch
    x = np.stack([signal("speech", 20_011, 1), signal("speech", 20_011, 2)], axis=1).ravel()
    before = ctx.launch_count
    res = batch.frontend_batch(x, np.array([0, x.size]), FL, FS, "hamming", channels=2, ctx=ctx)
    assert ctx.launch_count - before == 1
    assert (res.status & EXACT).all()


# ---- KNN -----------------------------------------------------------------------------------------------------------
# (d, n, k, env, knn_prune, scan kind, launches of one top-k call)
KNN = [
    ("tc16 pruned", 15, 2000, 3, None, 1, 3, 18),        # prune pass 12 + filter 2 + rerank 1 + refine 2 + rescan 1
    ("tc16 always pruned", 15, 2000, 3, None, 2, 3, 18),
    ("tc16 unpruned", 15, 2000, 3, None, 0, 3, 6),       # filter 2 + rerank 1 + refine 2 + rescan 1
    ("fp32 with refine", 15, 2000, 3, {"DSP_KNN_NO_TC16": "1"}, 1, 1, 5),
    ("fp32 under 64 train rows", 15, 63, 3, None, 1, 1, 5),
    ("fp32 k = 8", 15, 2000, 8, None, 1, 1, 3),          # k >= 8: no filter and no refine
    ("fp32 d = 40", 40, 2000, 3, None, 1, 1, 3),
    ("dense", 100, 2000, 3, None, 1, 2, 4),              # pack + scan per query chunk, rerank, rescan
    ("float64 only", 100, 2000, 3, {"DSP_KNN_NO_DENSE": "1"}, 1, 0, 2),
    ("float64 only, d > 16384", 16385, 70, 3, None, 1, 0, 2),
]


def knn_case(d, n, m, seed=0):
    rng = np.random.default_rng(seed + d)
    train = rng.standard_normal((n, d))
    near = train[rng.integers(0, n, m // 2)] + rng.standard_normal((m // 2, d)) * 1e-3
    q = np.concatenate([near, rng.standard_normal((m - m // 2, d))])
    return train, rng.integers(0, 4, n), q


@pytest.mark.parametrize("name,d,n,k,env,prune,kind,launches", KNN, ids=[c[0] for c in KNN])
def test_knn_scan_kinds(ctx, name, d, n, k, env, prune, kind, launches):
    from dsp_audioreclabs_b200 import batch
    train, y, q = knn_case(d, n, 300)
    ctx.set_tuning("knn_prune", prune)
    try:
        with Env(**(env or {})):
            knn = batch.KNN(k, ctx=ctx).fit(train, y)
            assert knn.last_stats()[1] == kind, name
            before = ctx.launch_count
            knn.kneighbors(q)
            assert ctx.launch_count - before == launches, name
            assert knn.last_stats()[1] == kind, name
    finally:
        ctx.set_tuning("knn_prune", 1)


def test_knn_dense_query_chunks_count_per_chunk(ctx):
    from dsp_audioreclabs_b200 import batch
    train, y, q = knn_case(64, 300, 32_769)
    knn = batch.KNN(3, ctx=ctx).fit(train, y)
    before = ctx.launch_count
    knn.kneighbors(q)
    assert ctx.launch_count - before == 2 * 2 + 2
    assert knn.last_stats()[1] == 2


@pytest.mark.parametrize("prune,launches", [(0, 7), (1, 18)])       # unpruned: + the start thresholds of the bound
def test_knn_bounded_filter_call(ctx, prune, launches):
    import torch
    from dsp_audioreclabs_b200.device import DeviceKNN
    train, y, q = knn_case(15, 2000, 300)
    tt = torch.from_numpy(train).cuda()
    qt = torch.from_numpy(q).cuda()
    ctx.set_tuning("knn_prune", prune)
    try:
        knn = DeviceKNN(3, ctx=ctx).fit(tt, torch.from_numpy(y.astype(np.int32)).cuda())
        ref = knn.topk(qt)
        bound = torch.full((len(q),), float("inf"), dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        before = ctx.launch_count
        got = knn.topk(qt, bound)
        torch.cuda.synchronize()
        assert ctx.launch_count - before == launches
        assert knn.last_stats()[1] == 3
        assert torch.equal(got[1], ref[1]) and torch.equal(got[0], ref[0])
        knn.free()
    finally:
        ctx.set_tuning("knn_prune", 1)
