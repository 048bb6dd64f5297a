"""KNN against the float64 oracle on every route the dispatch can take (csrc/capi.cu, csrc/knn.cu).

Routes: the scan kind chosen at fit (3 tensor-core filter, d <= 15 and k < 8; 1 fp32 tiled scan, d <= 63; 2 tensor-core
dense scan, 64 <= d <= 16,384; 0 float64 only), the refine pass and its 65,536-query cap, the exhaustive rescan split over
`parts` slices of the train rows, the dense scan's 32,768-query chunks, the vote and the sharded merge.  Every case
asserts the route it meant to reach (knn.last_stats(), the DSP_KNN_DEBUG line), then compares with the oracle:
neighbour indices, squared distances (np.array_equal: every kernel sums (q_j - t_j)^2 in feature order in float64
without FMA) and labels, exactly."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from oracle import knn_oracle as ko

pytestmark = pytest.mark.gpu

KNN_CAND = 8                # kKnnCand: the filter's certificate only for k below it
MAX_K = 16                  # kKnnMaxK
DENSE_MAX_DIM = 16384       # kKnnDenseMaxDim
DENSE_CHUNK = 32768         # kKnnDenseQueryChunk
REFINE_CAP = 65536


# ---- reference --------------------------------------------------------------------------------
def ref_topk(train, q, k):
    """knn_oracle.knn_topk over blocks of queries: the same per-feature float64 accumulation, ties by (distance, index);
    ranks beyond n are (-1, inf)."""
    train = np.asarray(train, np.float64)
    q = np.asarray(q, np.float64)
    n, m = len(train), len(q)
    kk = min(k, n)
    idx = np.full((m, k), -1, np.int64)
    dist = np.full((m, k), np.inf)
    block = max(1, min(m, (1 << 22) // max(n, 1)))
    tt = np.ascontiguousarray(train.T)
    for b0 in range(0, m, block):
        qb = q[b0:b0 + block]
        d = np.zeros((len(qb), n))
        for j in range(train.shape[1]):
            t = qb[:, j:j + 1] - tt[j][None, :]
            d += t * t
        # the kk smallest by (distance, index): everything below the kk-th value, then the lowest indices equal to it
        vk = np.partition(d, kk - 1, axis=1)[:, kk - 1:kk]
        lt = d < vk
        eq = d == vk
        sel = lt | (eq & (np.cumsum(eq, axis=1) <= kk - lt.sum(axis=1, keepdims=True)))
        cols = np.nonzero(sel)[1].reshape(len(qb), kk)
        dv = np.take_along_axis(d, cols, axis=1)
        order = np.lexsort((cols, dv), axis=-1)
        idx[b0:b0 + len(qb), :kk] = np.take_along_axis(cols, order, axis=1)
        dist[b0:b0 + len(qb), :kk] = np.take_along_axis(dv, order, axis=1)
    return idx, dist


def ref_vote(nbr_labels, classes):
    """Majority over the ranks present (label index >= 0), ties to the smallest class."""
    counts = np.stack([(nbr_labels == c).sum(axis=1) for c in range(len(classes))], axis=1)
    return classes[np.argmax(counts, axis=1)]


def test_reference_copy_matches_oracle():
    rng = np.random.default_rng(0)
    train = rng.integers(-2, 3, (300, 7)).astype(np.float64)          # many exact ties
    q = rng.integers(-2, 3, (50, 7)) + rng.choice([0.0, 0.5], (50, 7))
    for k in (1, 3, 8, 16):
        i, d = ref_topk(train, q, k)
        ri, rd = ko.knn_topk(train, q, k)
        assert np.array_equal(i, ri) and np.array_equal(d, rd)
        y = rng.integers(0, 4, 300)
        assert np.array_equal(ref_vote(y[i], np.unique(y)), ko.knn_predict(train, y, q, k))
    i, d = ref_topk(train[:5], q, 9)
    assert np.all(i[:, 5:] == -1) and np.all(np.isinf(d[:, 5:])) and np.array_equal(i[:, :5], ko.knn_topk(train[:5], q, 5)[0])


# ---- running the library ----------------------------------------------------------------------
class Env:
    """Sets the DSP_KNN_* switches the library reads at fit / per call (getenv), restores them after."""

    def __init__(self, **kw):
        self.kw = {k: v for k, v in kw.items() if v is not None}

    def __enter__(self):
        self.old = {k: os.environ.get(k) for k in self.kw}
        os.environ.update(self.kw)

    def __exit__(self, *a):
        for k, v in self.old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def run(ctx, train, y, q, k, env=None, prune=None):
    """fit + top-k (raw squared distances) + predict through the host API -> (idx, d2, labels, pred, (rescanned, kind))."""
    from dsp_audioreclabs_b200 import batch
    from dsp_audioreclabs_b200._capi import check
    env = env or {}
    if prune is not None:
        ctx.set_tuning("knn_prune", prune)
    try:
        with Env(**env):
            knn = batch.KNN(k, ctx=ctx).fit(train, y)
            q = np.ascontiguousarray(q, np.float64)
            m = len(q)
            idx = np.empty((m, k), np.int64)
            d2 = np.empty((m, k), np.float64)
            lab = np.empty((m, k), np.int32)
            check(ctx.lib.dsp_knn_topk_host(knn.handle, q.ctypes.data_as(C.c_void_p), m, idx.ctypes.data_as(C.c_void_p),
                                            d2.ctypes.data_as(C.c_void_p), lab.ctypes.data_as(C.c_void_p)))
            stats = knn.last_stats()
            pred = knn.predict(q)
            assert knn.last_stats() == stats
    finally:
        if prune is not None:
            ctx.set_tuning("knn_prune", 1)
    return idx, d2, lab, pred, knn.classes_, stats


def expected_kind(d, n, k, env=None):
    env = env or {}
    if d <= 15 and n >= 64 and k < KNN_CAND and "DSP_KNN_NO_TC16" not in env:
        return 3
    if d <= 63:
        return 1
    if d <= DENSE_MAX_DIM and "DSP_KNN_NO_DENSE" not in env:
        return 2
    return 0


def check(ctx, train, y, q, k, kind, env=None, prune=None, rescanned=None, ref=None):
    """Runs one case; asserts its route, then exact equality with the oracle.  Returns last_stats()."""
    idx, d2, lab, pred, classes, stats = run(ctx, train, y, q, k, env, prune)
    assert stats[1] == kind, (stats, kind)
    if rescanned is not None:
        assert stats[0] == rescanned, (stats, rescanned)
    ri, rd = ref if ref is not None else ref_topk(train, q, k)
    assert np.array_equal(idx, ri)
    assert np.array_equal(d2, rd)
    enc = np.searchsorted(classes, np.asarray(y))
    rl = np.where(ri >= 0, enc[np.maximum(ri, 0)], -1)
    assert np.array_equal(lab, rl)
    assert np.array_equal(pred, ref_vote(rl, classes))
    return stats


def gauss(rng, n, d, scale=1.0):
    return rng.standard_normal((n, d)) * scale


def debug_counts(capfd, fn):
    """Runs fn with DSP_KNN_DEBUG set; -> (exhaustive, refined, refined->exhaustive) of the last [knn] line."""
    capfd.readouterr()
    with Env(DSP_KNN_DEBUG="1"):
        out = fn()
    err = capfd.readouterr().err
    hits = re.findall(r"\[knn\] m=\d+ n=\d+ exhaustive=(\d+) refined=(\d+) refined->exhaustive=(\d+)", err)
    assert hits, err
    return out, tuple(int(v) for v in hits[-1])


# ---- feature width --------------------------------------------------------------------------------
WIDTHS = [(1, 127, 257), (15, 129, 256), (16, 255, 255), (17, 256, 1), (31, 257, 256), (32, 128, 257), (33, 129, 255),
          (63, 256, 256), (64, 255, 257), (65, 257, 1), (127, 128, 256), (128, 129, 255), (16384, 129, 257),
          (16385, 127, 256)]


@pytest.mark.parametrize("d,n,m", WIDTHS)
def test_width_sweep(ctx, d, n, m):
    rng = np.random.default_rng(d * 7 + n)
    train = gauss(rng, n, d)
    q = np.concatenate([train[:m // 3] + gauss(rng, m // 3, d, 1e-3), gauss(rng, m - m // 3, d)])
    y = rng.integers(0, 5, n)
    kind = expected_kind(d, n, 3)
    check(ctx, train, y, q, 3, kind, rescanned=m if kind == 0 else None)


@pytest.mark.parametrize("d,env", [(15, {"DSP_KNN_NO_TC16": "1"}), (200, {"DSP_KNN_NO_DENSE": "1"})])
def test_forced_scans(ctx, d, env):
    rng = np.random.default_rng(d)
    train, q = gauss(rng, 1000, d), gauss(rng, 300, d)
    y = rng.integers(0, 4, 1000)
    kind = expected_kind(d, 1000, 3, env)
    assert kind in (1, 0)
    check(ctx, train, y, q, 3, kind, env=env, rescanned=300 if kind == 0 else None)


@pytest.mark.parametrize("d", [64, 100])
def test_train_value_beyond_fp16_takes_float64_scan(ctx, d):
    rng = np.random.default_rng(d + 1)
    train, q = gauss(rng, 257, d), gauss(rng, 256, d)
    train[100, d // 2] = 1e5                                 # above 65504: the dense scan cannot hold it
    q[:10] = train[100] + gauss(rng, 10, d, 1e-2)
    check(ctx, train, rng.integers(0, 3, 257), q, 3, 0, rescanned=256)


# ---- k --------------------------------------------------------------------------------------------
K_ROUTES = [(15, None), (40, None), (100, None), (100, {"DSP_KNN_NO_DENSE": "1"})]


@pytest.mark.parametrize("d,env", K_ROUTES)
def test_k_sweep(ctx, d, env):
    rng = np.random.default_rng(d)
    n, m = 300, 200
    train = gauss(rng, n, d)
    q = np.concatenate([train[::3][:100] + gauss(rng, 100, d, 0.05), gauss(rng, 100, d)])
    y = rng.integers(0, 4, n)
    full = ref_topk(train, q, MAX_K)
    for k in range(1, MAX_K + 1):
        kind = expected_kind(d, n, k, env)
        # k >= kKnnCand: the candidate list cannot certify k neighbours, every query takes the exhaustive scan
        every = kind == 0 or k >= KNN_CAND
        check(ctx, train, y, q, k, kind, env=env, rescanned=m if every else None, ref=(full[0][:, :k], full[1][:, :k]))


@pytest.mark.parametrize("k", [4, 7])
@pytest.mark.parametrize("prune", [0, 1, 2])
def test_filter_k_prune_modes(ctx, k, prune):
    rng = np.random.default_rng(k * 10 + prune)
    centers = gauss(rng, 12, 15, 3.0)
    lab = rng.integers(0, 12, 4000)
    train = centers[lab] + gauss(rng, 4000, 15, 0.3)
    q = centers[rng.integers(0, 12, 1500)] + gauss(rng, 1500, 15, 0.3)
    check(ctx, train, lab, q, k, 3, prune=prune)


@pytest.mark.parametrize("d,env", [(15, None), (40, None), (100, None), (100, {"DSP_KNN_NO_DENSE": "1"})])
def test_k_above_n(ctx, d, env):
    """n = 5 rows, k = 9 or 16: ranks beyond n are (-1, inf, label -1), the vote counts the ranks present."""
    rng = np.random.default_rng(d + 5)
    train, q = gauss(rng, 5, d), gauss(rng, 40, d)
    y = np.array([3, 1, 3, 1, 2])
    for k in (9, 16):
        idx, d2, lab, pred, classes, stats = run(ctx, train, y, q, k, env)
        assert stats[1] == expected_kind(d, 5, k, env)
        assert np.all(idx[:, 5:] == -1) and np.all(np.isinf(d2[:, 5:])) and np.all(lab[:, 5:] == -1)
        check(ctx, train, y, q, k, stats[1], env=env)
        assert np.all(pred == 1)                            # 2 x 1, 2 x 3, 1 x 2: the tie goes to the smallest label


def test_k_above_limit_is_refused_before_any_launch(ctx):
    import torch
    from dsp_audioreclabs_b200 import batch, device
    rng = np.random.default_rng(17)
    train = gauss(rng, 300, 15)
    before = ctx.launch_count
    with pytest.raises(ValueError, match="n_neighbors"):
        batch.KNN(MAX_K + 1, ctx=ctx).fit(train, np.zeros(300, int))
    dev = torch.device("cuda", 0)
    with pytest.raises(ValueError, match="n_neighbors"):
        device.DeviceKNN(MAX_K + 1, ctx=ctx, device=dev).fit(torch.from_numpy(train).to(dev),
                                                             torch.zeros(300, dtype=torch.int32, device=dev))
    assert ctx.launch_count == before


# ---- ties -----------------------------------------------------------------------------------------
def rescan_geometry(ctx, n, d, total):
    """(parts, rows_per) of the exhaustive rescan for `total` rejected queries, as knn.cu computes them: 16 warps
    (d <= 64) or 16 CTAs (d > 64) per SM, parts = clamp(workers / total, 1, 64), slices rounded to 32 / 128 rows."""
    workers = 16 * ctx.sm_count
    parts = min(64, max(1, workers // max(total, 1)))
    unit = 32 if d <= 64 else 128
    return parts, ((n + parts - 1) // parts + unit - 1) // unit * unit


def lattice_case(ctx, d, n, m, seed):
    """Integer-lattice rows (exact float64 distances, many exact ties) in the first 3 features of d, plus copies of rows
    placed one filter tile (128 rows) and one rescan slice apart."""
    rng = np.random.default_rng(seed)
    train = np.zeros((n, d))
    train[:, :3] = rng.integers(0, 6, (n, 3))
    if d > 3:
        train[:, 3] = rng.integers(0, 2, n)
    offsets = {128} | {rescan_geometry(ctx, n, d, t)[1] for t in (m, 1, 16 * ctx.sm_count // 2)}
    for o in sorted(offsets):
        for i in range(0, n - o, max(1, (n - o) // 12)):
            train[i + o] = train[i]
    q = np.zeros((m, d))
    q[:, :3] = rng.integers(0, 6, (m, 3)) + rng.choice([0.0, 0.5], (m, 3))
    return train, q


LABELS = {"str": np.array(["cat", "dog", "eel"]), "neg": np.array([-7, -1, 0]), "float": np.array([0.5, -2.25, 3.0])}


@pytest.mark.parametrize("d", [15, 20, 70])
@pytest.mark.parametrize("labels", list(LABELS))
def test_lattice_ties(ctx, d, labels):
    n, m = 1500, 600
    train, q = lattice_case(ctx, d, n, m, d)
    rng = np.random.default_rng(d + len(labels))
    y = LABELS[labels][rng.integers(0, 3, n)]
    full = ref_topk(train, q, MAX_K)
    for k in (1, 2, 3, 4, 8, 16):
        kind = expected_kind(d, n, k)
        check(ctx, train, y, q, k, kind, rescanned=m if k >= KNN_CAND else None, ref=(full[0][:, :k], full[1][:, :k]))


# ---- exhaustive rescan: slices and their merge ---------------------------------------------------------
RESCAN_ROUTES = [(20, None, 1000), (33, None, 33), (64, {"DSP_KNN_NO_DENSE": "1"}, 1000), (64, {"DSP_KNN_NO_DENSE": "1"}, 5),
                 (70, None, 1000), (70, None, 33), (70, {"DSP_KNN_NO_DENSE": "1"}, 5)]


@pytest.mark.parametrize("d,env,n", RESCAN_ROUTES)
def test_rescan_split_boundaries(ctx, d, env, n):
    """k >= 8: every query is rescanned, so the number of queries sets the number of rejected ones and with it `parts`:
    64 (1 and W/64 queries), 2 (W/2), 1 (W/2 + 1, W, W + 1), with W = 16 x SMs.  Narrow kernel for d <= 64, wide above."""
    W = 16 * ctx.sm_count
    totals = [1, W // 64, W // 2, W // 2 + 1, W, W + 1]
    train, q = lattice_case(ctx, d, n, W + 1, d + n)
    y = np.random.default_rng(n).integers(0, 4, n)
    for k in (8, 16):
        full = ref_topk(train, q, k)
        for t in totals:
            kind = expected_kind(d, n, k, env)
            parts = rescan_geometry(ctx, n, d, t)[0]
            assert parts == (64 if t <= W // 64 else 2 if t == W // 2 else 1)
            check(ctx, train, y, q[:t], k, kind, env=env, rescanned=t, ref=(full[0][:t], full[1][:t]))


# ---- dense scan: query chunks ---------------------------------------------------------------------------
@pytest.mark.parametrize("d", [64, 200])
def test_dense_query_chunks(ctx, d):
    rng = np.random.default_rng(d)
    n, mmax = 129, DENSE_CHUNK + 500
    train = gauss(rng, n, d)
    q = train[rng.integers(0, n, mmax)] + gauss(rng, mmax, d, 0.3)
    y = rng.integers(0, 6, n)
    full = ref_topk(train, q, 3)
    for m in (DENSE_CHUNK - 1, DENSE_CHUNK, DENSE_CHUNK + 1, mmax):
        check(ctx, train, y, q[:m], 3, 2, ref=(full[0][:m], full[1][:m]))
    # one query beyond the fp16 range, only in the second chunk: the whole call takes the float64 scan, still exact
    far = DENSE_CHUNK + 123
    q[far, d - 1] = 7e4
    ri, rd = ref_topk(train, q[far:far + 1], 3)
    full[0][far], full[1][far] = ri[0], rd[0]
    check(ctx, train, y, q, 3, 2, rescanned=mmax, ref=full)


# ---- refine pass and its cap ----------------------------------------------------------------------
def test_refine_cap(ctx, capfd):
    """Tight clusters of 20 rows within 1e-6 of each other: the filter's certificate rejects every query, the refine
    pass resolves the first 65,536 of them, the rest take the exhaustive scan."""
    rng = np.random.default_rng(5)
    centers = gauss(rng, 64, 15, 2.0)
    member = np.repeat(np.arange(64), 20)
    train = centers[member] + gauss(rng, len(member), 15, 1e-6)
    y = member % 5
    m = REFINE_CAP + 2000
    q = centers[rng.integers(0, 64, m)] + gauss(rng, m, 15, 5e-7)
    stats, counts = debug_counts(capfd, lambda: check(ctx, train, y, q, 3, 3))
    assert counts == (m - REFINE_CAP, REFINE_CAP, 0), counts
    assert stats[0] == m


# ---- sharded merge ----------------------------------------------------------------------------------
@pytest.mark.parametrize("bounds", [(0, 700, 2000), (0, 300, 1100, 2000)])
@pytest.mark.parametrize("k", [1, 7, 16])
@pytest.mark.parametrize("bounded", [False, True])
def test_sharded_merge(ctx, bounds, k, bounded):
    """Row shards (DeviceKNN index_base) + merge_vote, unbounded or with the owner shard's k-th distance as the bound."""
    import torch
    from dsp_audioreclabs_b200 import device
    rng = np.random.default_rng(k + len(bounds))
    centers = gauss(rng, 10, 15, 3.0)
    lab = rng.integers(0, 10, 2000)
    train = centers[lab] + gauss(rng, 2000, 15, 0.4)
    train[1500:1510] = train[100:110]                        # exact duplicates in other shards
    q = np.concatenate([centers[rng.integers(0, 10, 700)] + gauss(rng, 700, 15, 0.4), train[95:115]])
    dev = torch.device("cuda", 0)
    xt = torch.from_numpy(train).to(dev)
    yt = torch.from_numpy(lab.astype(np.int32)).to(dev)
    qt = torch.from_numpy(q).to(dev)
    r = len(bounds) - 1
    knns = [device.DeviceKNN(k, ctx=ctx, device=dev, index_base=bounds[s]).fit(xt[bounds[s]:bounds[s + 1]].contiguous(),
                                                                               yt[bounds[s]:bounds[s + 1]].contiguous())
            for s in range(r)]
    bound = None
    if bounded:
        owner = torch.arange(len(q), device=dev) % r
        own_kth = torch.stack([kn.topk(qt)[0][:, k - 1] for kn in knns])
        bound = own_kth.gather(0, owner[None, :])[0].contiguous()
    cd, ci, cl = zip(*[kn.topk(qt, bound) for kn in knns])
    labels, idx, d2 = knns[0].merge_vote(torch.stack(cd), torch.stack(ci), torch.stack(cl))
    torch.cuda.synchronize()
    ri, rd = ref_topk(train, q, k)
    assert np.array_equal(idx.cpu().numpy(), ri)
    assert np.array_equal(d2.cpu().numpy(), rd)
    assert np.array_equal(labels.cpu().numpy(), ref_vote(lab[ri], np.arange(10)))
    for kn in knns:
        kn.free()
