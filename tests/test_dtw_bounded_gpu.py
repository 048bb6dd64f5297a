"""DTW top-k with a per-query cost bound (DeviceDTW.topk(bound=), dsp_dtw_topk_bounded_device) and row-sharded DTW on
device tensors (dist.ShardedDeviceDTW).

The expected answers come from the host path's fp32 cost matrix (mfcc_dtw.DTWClassifier.kneighbors(return_matrix=True)):
for each query the first min(k, #{finite cost <= U}) templates of its (cost, index)-sorted costs <= U, compared in
float64, then (inf, -1, -1)."""
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


# ---- helpers ---------------------------------------------------------------------------------------------------------
def _seq_maker(dim, seed):
    rng = np.random.default_rng(seed)

    def seq(n, c):
        return (rng.standard_normal((n, dim)) * 0.3 + np.sin(np.arange(n)[:, None] * (0.1 + 0.05 * c)) * 2).astype(np.float32)
    return seq, rng


def _device_seqs(seqs, dim):
    from dsp_audioreclabs_b200 import mfcc_dtw
    flat, off = mfcc_dtw.pack_sequences(seqs, dim)
    return torch.from_numpy(flat).cuda(), torch.from_numpy(off).cuda()


def _cost_matrix(temps, labels, quers, ctx):
    """The host path's fp32 cost matrix [nq, nt]."""
    from dsp_audioreclabs_b200 import mfcc_dtw
    return mfcc_dtw.DTWClassifier(1, ctx=ctx).fit(temps, labels).kneighbors(quers, return_matrix=True)[3]


def _expected(cost, labels, k, bound, index_base=0):
    """(cost f64, index i64, label i32) [nq, k] of the bounded contract, from the cost matrix."""
    nq = cost.shape[0]
    c = np.full((nq, k), np.inf)
    i = np.full((nq, k), -1, dtype=np.int64)
    l = np.full((nq, k), -1, dtype=np.int32)
    for q in range(nq):
        row = cost[q].astype(np.float64)
        keep = np.nonzero(np.isfinite(row) & (row <= bound[q]))[0]
        order = keep[np.lexsort((keep, row[keep]))][:k]
        c[q, :len(order)], i[q, :len(order)], l[q, :len(order)] = row[order], order + index_base, labels[order]
    return c, i, l


def _fit(temps, labels, k, dim, index_base=0):
    from dsp_audioreclabs_b200 import device
    tf, to = _device_seqs(temps, dim)
    return device.DeviceDTW(k, index_base=index_base).fit(tf, to, torch.tensor(np.asarray(labels), dtype=torch.int32).cuda())


def _np(ts):
    return [t.cpu().numpy() for t in ts]


def _assert_same(got, want):
    for a, b, name in zip(got, want, ("cost", "index", "label")):
        assert a.shape == b.shape and np.array_equal(a, b), (name, a, b)


def _vote(lab):
    out = []
    for row in lab:
        row = row[row >= 0]
        out.append(int(np.bincount(row).argmax()) if len(row) else -1)
    return np.array(out, dtype=np.int32)


def _cuda_bound(b):
    return torch.tensor(np.asarray(b, dtype=np.float64)).cuda()


T_LENS = [1, 2, 31, 32, 33, 64, 65, 100, 128, 129, 200, 256, 40, 57, 90, 7, 300, 513]
Q_LENS = [1, 5, 32, 33, 64, 97, 128, 130, 255, 256, 77, 257, 300, 511, 512, 513, 700]


# ---- single handle ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [1, 3, 16])
@pytest.mark.parametrize("dim", [1, 13, 16, 24, 40, 128])
def test_bound_inf_and_exact_kth_change_nothing(ctx, dim, k):
    """bound = +inf for every query, and bound = the unbounded call's k-th cost: bit-identical to the unbounded call,
    which equals the host path.  Queries cross strip boundaries; the max_q_frames hints pick every (R, DMAX) build of
    the feature dimension (1 x 16 .. 8 x 16 for dim <= 16, 4 x 32, 2 x 64, 1 x 128)."""
    seq, _ = _seq_maker(dim, 100 + dim)
    t_lens = [n for n in T_LENS if dim < 128 or n <= 300]
    labels = np.array([i % 4 for i in range(len(t_lens))])
    temps = [seq(n, labels[i]) for i, n in enumerate(t_lens)]
    quers = [seq(n, i % 4) for i, n in enumerate(Q_LENS)]
    cost = _cost_matrix(temps, labels, quers, ctx)
    want = _expected(cost, labels, k, np.full(len(quers), np.inf))
    dtw = _fit(temps, labels, k, dim)
    qf, qo = _device_seqs(quers, dim)
    for hint in ((32, 64, 128, 700) if dim <= 16 else (None,)):
        free = dtw.topk(qf, qo, max_q_frames=hint)
        _assert_same(_np(free), want)
        inf = dtw.topk(qf, qo, max_q_frames=hint, bound=_cuda_bound(np.full(len(quers), np.inf)))
        _assert_same(_np(inf), want)
        kth = dtw.topk(qf, qo, max_q_frames=hint, bound=free[0][:, k - 1].contiguous())
        _assert_same(_np(kth), want)


def _prev32(x):
    return float(np.nextafter(np.float32(x), np.float32(-np.inf)))


@pytest.mark.parametrize("k", [1, 3, 16])
def test_mixed_bounds_in_one_call(ctx, k):
    """One call, one kind of bound per query: 0, negative, NaN, +inf, exactly a neighbour's cost (tie at the radius),
    between two costs, and a value in (prev fp32 of c, c) for a neighbour cost c: rounded up to fp32 it is c, so only
    the float64 comparison keeps c out."""
    seq, _ = _seq_maker(13, 7)
    labels = np.arange(60) % 5
    temps = [seq(int(n), labels[i]) for i, n in enumerate(np.random.default_rng(1).integers(5, 80, 60))]
    temps[41] = temps[3].copy()
    quers = [seq(int(n), i % 5) for i, n in enumerate(np.random.default_rng(2).integers(5, 80, 16))]
    quers[0] = temps[3].copy()
    cost = _cost_matrix(temps, labels, quers, ctx)
    s = np.sort(cost.astype(np.float64), axis=1)
    bound = np.array([0.0, -1.0, np.nan, np.inf, s[4, 1], (s[5, 0] + s[5, 1]) / 2, (_prev32(s[6, 1]) + s[6, 1]) / 2,
                      (_prev32(s[7, 0]) + s[7, 0]) / 2, s[8, 0], s[9, 2], -0.0, s[11, 5], np.inf, 1e300, s[14, 0] * 0.99,
                      s[15, 3]])
    assert _prev32(s[6, 1]) < bound[6] < s[6, 1]
    want = _expected(cost, labels, k, bound)
    assert list(want[1][0][:2]) == [3, 41][:k] and np.all(want[1][1:3] == -1)
    assert np.all(want[1][7] == -1) and np.all(want[1][14] == -1)
    dtw = _fit(temps, labels, k, 13)
    qf, qo = _device_seqs(quers, 13)
    got = _np(dtw.topk(qf, qo, bound=_cuda_bound(bound)))
    _assert_same(got, want)
    pred = dtw.predict(qf, qo, bound=_cuda_bound(bound)).cpu().numpy()
    assert np.array_equal(pred, _vote(want[2]))
    assert np.all(pred[[1, 2, 7, 10, 14]] == -1)


def test_ties_at_the_radius_across_slices(ctx):
    """Few queries, many templates: the fused kernel cuts the templates into several slices.  Template 5 reappears as
    600 and 1000 (other slices); with the bound at the duplicated cost the kept indices follow the lower-index rule,
    and a bound just below it (rounding up to it in fp32) keeps none of the three."""
    seq, rng = _seq_maker(13, 9)
    nt = 1024
    labels = np.arange(nt) % 4
    temps = [seq(20 + i % 17, labels[i]) for i in range(nt)]
    temps[600] = temps[5].copy()
    temps[1000] = temps[5].copy()
    near = temps[5] + 0.01 * rng.standard_normal(temps[5].shape).astype(np.float32)
    quers = [temps[5].copy(), near, seq(25, 1), near.copy()]
    cost = _cost_matrix(temps, labels, quers, ctx)
    assert cost[1, 5] == cost[1, 600] == cost[1, 1000] > 0
    c = float(cost[3, 5])
    bound = np.array([0.0, float(cost[1, 5]), float(cost[2].min()), (_prev32(c) + c) / 2])
    for k in (1, 2, 3, 16):
        want = _expected(cost, labels, k, bound)
        assert list(want[1][0][:3]) == [5, 600, 1000][:k] and list(want[1][1][:3]) == [5, 600, 1000][:k]
        assert not np.any(np.isin(want[1][3], [5, 600, 1000]))
        dtw = _fit(temps, labels, k, 13)
        qf, qo = _device_seqs(quers, 13)
        _assert_same(_np(dtw.topk(qf, qo, bound=_cuda_bound(bound))), want)


def test_edge_cases_with_bounds(ctx):
    """Fewer templates than k, an empty query, an empty template, index_base != 0, no queries at all."""
    seq, _ = _seq_maker(13, 5)
    temps = [seq(n, i) for i, n in enumerate([12, 0, 30, 5, 40])]
    labels = np.array([3, 1, 2, 3, 0])
    quers = [seq(n, i) for i, n in enumerate([20, 0, 1, 45, 33])]
    cost = _cost_matrix(temps, labels, quers, ctx)
    s = np.sort(cost.astype(np.float64), axis=1)
    for bound in (np.full(5, np.inf), np.array([s[0, 1], np.inf, 0.0, s[3, 0], s[4, 3]])):
        for k in (1, 3, 16):
            want = _expected(cost, labels, k, bound, index_base=1000)
            dtw = _fit(temps, labels, k, 13, index_base=1000)
            qf, qo = _device_seqs(quers, 13)
            _assert_same(_np(dtw.topk(qf, qo, bound=_cuda_bound(bound))), want)
            assert np.all(want[1][1] == -1) and not np.any(want[1] == 1001)
            qf0, qo0 = _device_seqs([], 13)
            c0, i0, l0 = dtw.topk(qf0, qo0, bound=_cuda_bound([]))
            assert tuple(c0.shape) == (0, k) and tuple(i0.shape) == (0, k)
            assert dtw.last_stats() == (0, 0)
            assert tuple(dtw.predict(qf0, qo0, bound=_cuda_bound([])).shape) == (0,)


def test_bound_is_checked(ctx):
    seq, _ = _seq_maker(13, 4)
    temps = [seq(10, 0), seq(12, 1)]
    dtw = _fit(temps, [0, 1], 1, 13)
    qf, qo = _device_seqs([seq(9, 0), seq(8, 1)], 13)
    for bad in (torch.zeros(2, dtype=torch.float32, device="cuda"), torch.zeros(3, dtype=torch.float64, device="cuda"),
                torch.zeros(2, dtype=torch.float64), torch.zeros(4, dtype=torch.float64, device="cuda")[::2]):
        with pytest.raises(ValueError):
            dtw.topk(qf, qo, bound=bad)


def test_stats_with_a_tight_bound(ctx):
    """Eight well-separated clusters: a bound at each query's nearest cost abandons at least as many pairs as the
    unbounded call, and scored + abandoned is the pair count (a query with a negative bound counts as abandoned)."""
    rng = np.random.default_rng(3)
    centres = rng.standard_normal((8, 13)).astype(np.float32) * 20

    def member(c, n):
        return (centres[c] + rng.standard_normal((n, 13)) * 0.5).astype(np.float32)
    temps = [member(i % 8, int(rng.integers(10, 60))) for i in range(1024)]
    labels = np.arange(1024) % 8
    quers = [member(i % 8, int(rng.integers(10, 60))) for i in range(64)]
    cost = _cost_matrix(temps, labels, quers, ctx)
    dtw = _fit(temps, labels, 3, 13)
    qf, qo = _device_seqs(quers, 13)
    free = dtw.topk(qf, qo)
    s_free, a_free = dtw.last_stats()
    bound = free[0][:, 0].contiguous()
    bound[5] = -1.0
    got = _np(dtw.topk(qf, qo, bound=bound))
    s_b, a_b = dtw.last_stats()
    _assert_same(got, _expected(cost, labels, 3, bound.cpu().numpy()))
    assert s_free + a_free == 64 * 1024 and s_b + a_b == 64 * 1024
    assert a_b >= a_free, (a_b, a_free)


@pytest.mark.parametrize("shards", [2, 3, 8])
def test_emulated_shards_merge_to_the_single_handle(ctx, shards):
    """R template shards on one GPU (with 19 templates, eight shards hold fewer than k = 3 each): per-shard topk,
    unbounded and bounded by the whole set's k-th cost, merged with dsp_knn_merge_vote_device (DeviceKNN.merge_vote)
    and with dist.merge_topk, equal the single handle's answer."""
    from dsp_audioreclabs_b200 import device, dist as ddist
    seq, rng = _seq_maker(13, 40 + shards)
    nt, k = 19, 3
    labels = np.arange(nt) % 3
    temps = [seq(int(n), labels[i]) for i, n in enumerate(rng.integers(8, 70, nt))]
    temps[15] = temps[2].copy()
    quers = [seq(int(n), i % 3) for i, n in enumerate(rng.integers(8, 70, 30))]
    quers[0] = temps[2].copy()
    qf, qo = _device_seqs(quers, 13)
    whole = _fit(temps, labels, k, 13)
    ref = whole.topk(qf, qo)
    ref_pred = whole.predict(qf, qo)
    tb = ddist.balanced_bounds(nt, shards)
    assert min(np.diff(tb)) < k or shards < 8
    parts = [_fit(temps[tb[r]:tb[r + 1]], labels[tb[r]:tb[r + 1]], k, 13, index_base=int(tb[r])) for r in range(shards)]
    for bound in (None, ref[0][:, k - 1].contiguous()):
        cand = [torch.stack(t) for t in zip(*[p.topk(qf, qo, bound=bound) for p in parts])]
        lab, idx, d = device.DeviceKNN(k).merge_vote(*cand)
        assert torch.equal(idx, ref[1]) and torch.equal(d, ref[0]) and torch.equal(lab, ref_pred)
        for a, b in zip(ddist.merge_topk(*cand, k), ref):
            assert torch.equal(a, b)


def test_bounded_call_captures_in_a_cuda_graph(ctx):
    """Once warm, the bounded call captures in a CUDA graph (the capture fails on any synchronisation or allocation),
    and a replay with new bounds written in place gives the eager results for them."""
    seq, rng = _seq_maker(13, 12)
    labels = np.arange(200) % 5
    temps = [seq(int(n), labels[i]) for i, n in enumerate(rng.integers(5, 60, 200))]
    quers = [seq(int(n), i % 5) for i, n in enumerate(rng.integers(5, 60, 40))]
    dtw = _fit(temps, labels, 3, 13)
    qf, qo = _device_seqs(quers, 13)
    free = dtw.topk(qf, qo)
    b1 = free[0][:, 1].contiguous()
    b2 = free[0][:, 0].contiguous() * 0.5
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    bound = b1.clone()
    with torch.cuda.stream(stream):
        warm = [t.clone() for t in dtw.topk(qf, qo, max_q_frames=60, bound=bound)]
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=stream):
        outs = dtw.topk(qf, qo, max_q_frames=60, bound=bound)
    for t in outs:
        t.fill_(0)
    g.replay()
    torch.cuda.synchronize()
    for a, b in zip(outs, warm):
        assert torch.equal(a, b)
    bound.copy_(b2)
    g.replay()
    torch.cuda.synchronize()
    ctx.use_own_stream()
    for a, b in zip(outs, dtw.topk(qf, qo, bound=b2)):
        assert torch.equal(a, b)
    assert torch.all(outs[1][:, 0] == -1)


# ---- process groups --------------------------------------------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _sharded_data():
    seq, rng = _seq_maker(13, 77)
    nt = 301
    labels = (np.arange(nt) % 6).astype(np.int32)
    temps = [seq(int(n), labels[i]) for i, n in enumerate(rng.integers(10, 64, nt))]
    temps[250] = temps[17].copy()
    quers = [seq(int(n), i % 6) for i, n in enumerate(rng.integers(10, 64, 90))]
    quers[3] = temps[17].copy()
    return temps, labels, quers


def _sharded_run(rank, world, dev):
    """kneighbors / predict of ShardedDeviceDTW (default CUDA scoring) on this rank's shard, without and with a bound
    (the single-handle 2nd cost, and -1 for every 7th query); returns them with the single-handle answers."""
    from dsp_audioreclabs_b200 import device, dist as ddist
    temps, labels, quers = _sharded_data()
    tb = ddist.balanced_bounds(len(temps), world)
    with torch.cuda.device(dev):
        tf, to = _device_seqs(temps[tb[rank]:tb[rank + 1]], 13)
        qf, qo = _device_seqs(quers, 13)
        whole_tf, whole_to = _device_seqs(temps, 13)
        whole = device.DeviceDTW(3, device=dev).fit(whole_tf, whole_to, torch.from_numpy(labels).to(dev))
        bound = whole.topk(qf, qo)[0][:, 1].contiguous()
        bound[::7] = -1.0
        sd = ddist.ShardedDeviceDTW(3).fit(tf, to, torch.from_numpy(labels[tb[rank]:tb[rank + 1]]).to(dev))
        out = {}
        for name, b in (("free", None), ("bounded", bound)):
            got = sd.kneighbors(qf, qo, bound=b, max_q_frames=64)
            want = whole.topk(qf, qo, bound=b)
            out[name] = ([t.cpu() for t in got], [t.cpu() for t in want],
                         sd.predict(qf, qo, bound=b).cpu(), whole.predict(qf, qo, bound=b).cpu())
        return out


def _check_sharded(out):
    for name, (got, want, pred, want_pred) in out.items():
        for a, b in zip(got, want):
            assert torch.equal(a, b), name
        assert torch.equal(pred, want_pred), name
    assert torch.all(out["bounded"][2][::7] == -1)


def test_sharded_device_dtw_one_rank_nccl(ctx):
    import torch.distributed as dist
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{_free_port()}", rank=0, world_size=1,
                            device_id=torch.device("cuda", 0))
    try:
        _check_sharded(_sharded_run(0, 1, torch.device("cuda", 0)))
    finally:
        dist.destroy_process_group()


def _nccl_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world, device_id=dev)
    try:
        torch.save(_sharded_run(rank, world, dev), os.path.join(out_dir, f"r{rank}.pt"))
    finally:
        dist.destroy_process_group()


def test_sharded_device_dtw_two_ranks_nccl(tmp_path):
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("two-rank NCCL test: needs 2 visible GPUs, %d visible" % torch.cuda.device_count())
    mp.spawn(_nccl_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    for r in range(2):
        _check_sharded(torch.load(tmp_path / f"r{r}.pt"))
