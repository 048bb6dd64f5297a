"""MFCC + DTW template matching on device tensors (device.DeviceMFCC / DeviceDTW, torch ops mfcc_batch / dtw_topk).

The device path must give the host path's bits: MFCC rows equal to mfcc_dtw.mfcc_batch, DTW costs equal to the cost
matrix entries of mfcc_dtw.DTWClassifier (the same cell arithmetic), the same neighbours with ties to the lower index.
On top of that it keeps its promises: no cost matrix, early exit that changes nothing, no synchronisation or allocation
on the hot path (CUDA graph capture)."""
import numpy as np
import pytest
import torch


# ---- helpers ---------------------------------------------------------------------------------------------------------
def _sixteen_utterances():
    """The utterances of test_mfcc_dtw_gpu.py::test_mfcc_matches_the_self_oracle."""
    from oracle import synth
    lens = synth.ragged_lengths(14, 0.25, 1.0, seed=8)
    utts = [synth.utterance_pcm(i, int(n), seed0=321) for i, n in enumerate(lens)]
    utts.append(np.full(3000, 1234, dtype=np.int16))              # constant signal: every mel energy on the log floor
    utts.append(utts[0][:700].copy())                             # shorter than one frame
    return utts


def _seq_maker(dim, seed):
    rng = np.random.default_rng(seed)

    def seq(n, c):
        return (rng.standard_normal((n, dim)) * 0.3 + np.sin(np.arange(n)[:, None] * (0.1 + 0.05 * c)) * 2).astype(np.float32)
    return seq, rng


def _device_seqs(seqs, dim):
    from dsp_audioreclabs_b200 import mfcc_dtw
    flat, off = mfcc_dtw.pack_sequences(seqs, dim)
    return torch.from_numpy(flat).cuda(), torch.from_numpy(off).cuda()


def _host_topk(temps, labels, quers, k, index_base=0, ctx=None):
    from dsp_audioreclabs_b200 import mfcc_dtw
    return mfcc_dtw.DTWClassifier(k, ctx=ctx, index_base=index_base).fit(temps, labels).kneighbors(quers)


def _device_topk(temps, labels, quers, k, dim, index_base=0, max_q_frames=None):
    from dsp_audioreclabs_b200 import device
    tf, to = _device_seqs(temps, dim)
    qf, qo = _device_seqs(quers, dim)
    dtw = device.DeviceDTW(k, index_base=index_base).fit(tf, to, torch.tensor(np.asarray(labels), dtype=torch.int32).cuda())
    out = [t.cpu().numpy() for t in dtw.topk(qf, qo, max_q_frames=max_q_frames)]
    return out, dtw


def _assert_same(dev, host):
    for a, b, name in zip(dev, host, ("cost", "index", "label")):
        assert a.shape == b.shape and np.array_equal(a, b), name


# ---- CPU -------------------------------------------------------------------------------------------------------------
def test_ops_are_registered_with_fake_implementations():
    import dsp_audioreclabs_b200.torch_ops  # noqa: F401
    from torch._subclasses.fake_tensor import FakeTensorMode
    ns = torch.ops.dsp_audioreclabs
    assert hasattr(ns, "mfcc_batch") and hasattr(ns, "dtw_topk")
    with FakeTensorMode():
        s = torch.empty(5000, dtype=torch.int16)
        off = torch.empty(4, dtype=torch.int64)
        se = torch.empty(3, dtype=torch.int32)
        mfcc, nf = ns.mfcc_batch(s, off, se, se, off, 17, 1102, 441, 2048, 26, 13, 1, 0.97, 1e-10)
        assert tuple(mfcc.shape) == (17, 13) and mfcc.dtype == torch.float32
        assert tuple(nf.shape) == (3,) and nf.dtype == torch.int32
        tf = torch.empty(50, 13, dtype=torch.float32)
        cost, idx, lab = ns.dtw_topk(tf, off, se, tf, torch.empty(6, dtype=torch.int64), 3)
        assert [tuple(t.shape) for t in (cost, idx, lab)] == [(5, 3)] * 3
        assert (cost.dtype, idx.dtype, lab.dtype) == (torch.float64, torch.int64, torch.int32)


def test_plan_capacities_bound_every_segment():
    """The rows DeviceMFCC plans per utterance (dsp_frontend_plan's untrimmed frame counts) hold the frames of any
    segment [start, end) inside the utterance (frame count of the oracle's frame_signal rule)."""
    from dsp_audioreclabs_b200 import batch
    from oracle import frontend_oracle as fo
    rng = np.random.default_rng(11)
    for fl, fs in ((1102, 441), (256, 128), (400, 160), (7, 3)):
        lens = rng.integers(0, 20000, 200)
        lens[:3] = (0, 1, fl)
        off = np.concatenate([[0], np.cumsum(lens)])
        cap = np.diff(batch.plan(off, batch.make_params(fl, fs))[0])
        for n, c in zip(lens, cap):
            for _ in range(5):
                a = int(rng.integers(0, n + 1))
                b = int(rng.integers(a, n + 1))
                assert fo.feature_frame_count(b - a, fl, fs) <= c
            assert fo.feature_frame_count(int(n), fl, fs) == c


# ---- GPU: MFCC -------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_device_mfcc_equals_the_host_call(ctx):
    from dsp_audioreclabs_b200 import batch, device, mfcc_dtw
    utts = _sixteen_utterances()
    s, o, l = batch.pack_aligned(utts)
    res = batch.frontend_batch(s, o, 1102, 441, "hamming", lengths=l, emit_frames=False, ctx=ctx)
    mf, off = mfcc_dtw.mfcc_batch(s, o, res.start, res.end, lengths=l, ctx=ctx)
    dm = device.DeviceMFCC(o, lengths=l)
    out = torch.full((max(dm.total_frames, 1), 13), float("nan"), dtype=torch.float32, device="cuda")
    got, cap, nf = dm.run(torch.from_numpy(s).cuda(), torch.from_numpy(res.start).cuda(), torch.from_numpy(res.end).cuda(),
                          out=out)
    got, cap, nf = got.cpu().numpy(), cap.cpu().numpy(), nf.cpu().numpy()
    assert np.array_equal(nf, np.diff(off))
    for b in range(len(utts)):
        assert np.array_equal(got[cap[b]:cap[b] + nf[b]], mf[off[b]:off[b + 1]]), b
        assert np.all(np.isnan(got[cap[b] + nf[b]:cap[b + 1]])), b


@pytest.mark.gpu
def test_front_end_to_mfcc_stays_on_the_device(ctx):
    from dsp_audioreclabs_b200 import batch, device, mfcc_dtw
    utts = _sixteen_utterances()
    s, o, l = batch.pack_aligned(utts)
    d_s = torch.from_numpy(s).cuda()
    fe = device.DeviceFrontend(o, 1102, 441, "hamming", lengths=l).run(d_s)
    dm = device.DeviceMFCC(o, lengths=l)
    got, cap, nf = dm.run(d_s, fe.start, fe.end)
    res = batch.frontend_batch(s, o, 1102, 441, "hamming", lengths=l, emit_frames=False, ctx=ctx)
    mf, off = mfcc_dtw.mfcc_batch(s, o, res.start, res.end, lengths=l, ctx=ctx)
    assert np.array_equal(fe.start.cpu().numpy(), res.start) and np.array_equal(fe.end.cpu().numpy(), res.end)
    got, cap, nf = got.cpu().numpy(), cap.cpu().numpy(), nf.cpu().numpy()
    assert np.array_equal(nf, np.diff(off))
    for b in range(len(utts)):
        assert np.array_equal(got[cap[b]:cap[b] + nf[b]], mf[off[b]:off[b + 1]]), b


# ---- GPU: DTW --------------------------------------------------------------------------------------------------------
T_LENS = [1, 2, 31, 32, 33, 64, 65, 100, 128, 129, 200, 256, 40, 57, 90, 7, 300, 513]
Q_LENS = [1, 5, 32, 33, 64, 97, 128, 130, 255, 256, 77, 257, 300, 511, 512, 513, 700]


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 3, 16])
@pytest.mark.parametrize("dim", [1, 13, 16, 17, 39, 64, 100, 128])
def test_dtw_topk_equals_the_host_path(ctx, dim, k):
    """The lengths of test_dtw_costs_and_neighbours (strip boundaries of every build); at dim 128 without the 513-frame
    template, which the host path cannot hold in shared memory."""
    seq, _ = _seq_maker(dim, dim)
    t_lens = [n for n in T_LENS if dim < 128 or n <= 300]
    labels = np.array([i % 4 for i in range(len(t_lens))])
    temps = [seq(n, labels[i]) for i, n in enumerate(t_lens)]
    quers = [seq(n, i % 4) for i, n in enumerate(Q_LENS)]
    host = _host_topk(temps, labels, quers, k, ctx=ctx)
    dev, _ = _device_topk(temps, labels, quers, k, dim, max_q_frames=max(Q_LENS) if k == 3 else None)
    _assert_same(dev, host)
    assert np.all(np.isinf(dev[0][:, len(t_lens):])) and np.all(dev[1][:, len(t_lens):] == -1)


@pytest.mark.gpu
def test_dtw_topk_edge_cases(ctx):
    """Fewer templates than k, an empty query, an empty template, index_base != 0, no queries at all."""
    seq, _ = _seq_maker(13, 5)
    temps = [seq(n, i) for i, n in enumerate([12, 0, 30, 5, 40])]
    labels = np.array([3, 1, 2, 3, 0])
    quers = [seq(n, i) for i, n in enumerate([20, 0, 1, 45, 33])]
    for k in (1, 3, 16):
        host = _host_topk(temps, labels, quers, k, index_base=1000, ctx=ctx)
        dev, dtw = _device_topk(temps, labels, quers, k, 13, index_base=1000)
        _assert_same(dev, host)
        assert np.all(dev[1][1] == -1) and np.all(np.isinf(dev[0][1]))       # the empty query
        assert not np.any(dev[1] == 1001)                                    # the empty template
        qf, qo = _device_seqs([], 13)
        cost, idx, lab = dtw.topk(qf, qo)
        assert tuple(cost.shape) == (0, k) and tuple(idx.shape) == (0, k)
        assert dtw.last_stats() == (0, 0)
        assert tuple(dtw.predict(qf, qo).shape) == (0,)


@pytest.mark.gpu
def test_dtw_topk_beyond_the_host_query_slab(ctx):
    """70,000 short queries against 64 short templates: more queries than one 65,535-query slab of the host grid."""
    seq, rng = _seq_maker(13, 70)
    temps = [seq(int(n), i % 5) for i, n in enumerate(rng.integers(1, 9, 64))]
    labels = np.arange(64) % 5
    quers = [seq(int(n), i % 5) for i, n in enumerate(rng.integers(1, 9, 70000))]
    host = _host_topk(temps, labels, quers, 3, ctx=ctx)
    dev, dtw = _device_topk(temps, labels, quers, 3, 13)
    _assert_same(dev, host)
    scored, abandoned = dtw.last_stats()
    assert scored + abandoned == 70000 * 64


@pytest.mark.gpu
def test_dtw_duplicate_templates_in_different_slices_tie_to_the_lower_index(ctx):
    """256 templates are cut into several slices; template 5 reappears as 200 and 250 (other slices): a query equal to
    it costs 0 against all three, and the lower indices win."""
    seq, _ = _seq_maker(13, 9)
    temps = [seq(20 + i % 17, i % 4) for i in range(256)]
    temps[200] = temps[5].copy()
    temps[250] = temps[5].copy()
    labels = np.arange(256) % 4
    quers = [temps[5].copy(), seq(25, 1), temps[5].copy(), seq(3, 2)]
    for k in (1, 2, 3):
        host = _host_topk(temps, labels, quers, k, ctx=ctx)
        dev, _ = _device_topk(temps, labels, quers, k, 13)
        _assert_same(dev, host)
        assert list(dev[1][0]) == [5, 200, 250][:k] and np.all(dev[0][0] == 0.0)


@pytest.mark.gpu
def test_dtw_early_exit_runs_and_changes_nothing(ctx):
    """Eight well-separated clusters: most (query, template) pairs are far apart and are abandoned early."""
    rng = np.random.default_rng(3)
    centres = rng.standard_normal((8, 13)).astype(np.float32) * 20

    def member(c, n):
        return (centres[c] + rng.standard_normal((n, 13)) * 0.5).astype(np.float32)
    temps = [member(i % 8, int(rng.integers(10, 60))) for i in range(1024)]
    labels = np.arange(1024) % 8
    quers = [member(i % 8, int(rng.integers(10, 60))) for i in range(64)]
    for k in (1, 3):
        host = _host_topk(temps, labels, quers, k, ctx=ctx)
        dev, dtw = _device_topk(temps, labels, quers, k, 13)
        _assert_same(dev, host)
        scored, abandoned = dtw.last_stats()
        assert abandoned > 0 and scored + abandoned == 64 * 1024, (scored, abandoned)


@pytest.mark.gpu
def test_dtw_topk_needs_no_cost_matrix(ctx):
    """70,000 x 4,096 pairs: a float32 cost matrix would take 1.07 GiB; the call may take less than 256 MB."""
    from dsp_audioreclabs_b200 import device
    seq, rng = _seq_maker(13, 4096)
    nq, nt = 70000, 4096
    assert nq * nt * 4 >= 1 << 30
    temps = [seq(int(n), i % 6) for i, n in enumerate(rng.integers(2, 9, nt))]
    labels = np.arange(nt) % 6
    quers = [seq(int(n), i % 6) for i, n in enumerate(rng.integers(2, 9, nq))]
    tf, to = _device_seqs(temps, 13)
    qf, qo = _device_seqs(quers, 13)
    dtw = device.DeviceDTW(3).fit(tf, to, torch.from_numpy(labels.astype(np.int32)).cuda())
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    cost, idx, lab = dtw.topk(qf, qo, max_q_frames=8)
    torch.cuda.synchronize()
    drop = free0 - torch.cuda.mem_get_info()[0]
    assert drop < 256 << 20, drop
    scored, abandoned = dtw.last_stats()
    assert scored + abandoned == nq * nt
    sel = np.arange(0, nq, 997)
    host = _host_topk(temps, labels, [quers[i] for i in sel], 3, ctx=ctx)
    _assert_same([cost.cpu().numpy()[sel], idx.cpu().numpy()[sel], lab.cpu().numpy()[sel]], host)


@pytest.mark.gpu
def test_mfcc_and_dtw_capture_in_a_cuda_graph(ctx):
    """DeviceMFCC.run -> DeviceDTW.topk (on the MFCC rows in place: capacities as offsets, n_frames as lengths) captured
    after one warm-up: the capture fails on any synchronisation, allocation or pageable copy, and a replay gives the
    warm-up results."""
    from dsp_audioreclabs_b200 import batch, device, mfcc_dtw
    utts = _sixteen_utterances()
    s, o, l = batch.pack_aligned(utts)
    res = batch.frontend_batch(s, o, 1102, 441, "hamming", lengths=l, emit_frames=False, ctx=ctx)
    mf, off = mfcc_dtw.mfcc_batch(s, o, res.start, res.end, lengths=l, ctx=ctx)
    temps = [mf[off[b]:off[b + 1]] for b in range(len(utts))]
    d_s, d_st, d_en = (torch.from_numpy(a).cuda() for a in (s, res.start, res.end))
    tf, to = _device_seqs(temps, 13)
    dm = device.DeviceMFCC(o, lengths=l)
    dtw = device.DeviceDTW(3).fit(tf, to, torch.arange(len(utts), dtype=torch.int32).cuda())
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())

    def step():
        mfcc, cap, nf = dm.run(d_s, d_st, d_en)
        return (mfcc, nf) + dtw.topk(mfcc, cap, lengths=nf, max_q_frames=200)
    with torch.cuda.stream(stream):
        warm = [t.clone() for t in step()]
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=stream):
        outs = step()
    for t in outs:
        t.fill_(0)
    g.replay()
    torch.cuda.synchronize()
    for a, b in zip(outs, warm):
        assert torch.equal(a, b)
    found = warm[1].cpu() > 0
    assert torch.equal(warm[3][:, 0].cpu()[found], torch.arange(len(utts))[found])   # every utterance finds itself
    ctx.use_own_stream()


@pytest.mark.gpu
def test_torch_ops_match_the_device_classes(ctx):
    from dsp_audioreclabs_b200 import batch, device, torch_ops
    ns = torch.ops.dsp_audioreclabs
    utts = _sixteen_utterances()
    s, o = np.concatenate(utts), np.concatenate([[0], np.cumsum([len(u) for u in utts])])
    res = batch.frontend_batch(s, o, 1102, 441, "hamming", emit_frames=False, ctx=ctx)
    pl = torch_ops.plan(o, 1102, 441)
    d_s, d_st, d_en = (torch.from_numpy(a).cuda() for a in (s, res.start, res.end))
    args = (d_s, pl.offsets, d_st, d_en, pl.feat_offsets, pl.total_frames, 1102, 441, 2048, 26, 13, 1, 0.97, 1e-10)
    mfcc, nf = ns.mfcc_batch(*args)
    ref, cap, rnf = device.DeviceMFCC(o).run(d_s, d_st, d_en)
    assert torch.equal(nf, rnf)
    for b in range(len(utts)):
        c0, n = int(cap[b]), int(nf[b])
        assert torch.equal(mfcc[c0:c0 + n], ref[c0:c0 + n]), b
    torch.library.opcheck(ns.mfcc_batch, args, test_utils=("test_schema", "test_faketensor"))
    seq, _ = _seq_maker(13, 1)
    temps = [seq(n, i % 3) for i, n in enumerate([10, 40, 3, 25, 60, 33, 17, 8])]
    quers = [seq(n, i % 3) for i, n in enumerate([12, 0, 50, 31, 7])]
    tf, to = _device_seqs(temps, 13)
    qf, qo = _device_seqs(quers, 13)
    tl = torch.tensor([2, 0, 1, 2, 0, 1, 2, 0], dtype=torch.int32).cuda()
    got = ns.dtw_topk(tf, to, tl, qf, qo, 3)
    want = device.DeviceDTW(3).fit(tf, to, tl).topk(qf, qo)
    for a, b in zip(got, want):
        assert torch.equal(a, b)
    torch.library.opcheck(ns.dtw_topk, (tf, to, tl, qf, qo, 3), test_utils=("test_schema", "test_faketensor"))
    pred = device.DeviceDTW(3).fit(tf, to, tl).predict(qf, qo).cpu().numpy()
    assert np.array_equal(pred, _vote(want[2].cpu().numpy()))


def _vote(lab):
    """Majority label per row (ties to the smallest label; -1 entries ignored, -1 when there are none)."""
    out = []
    for row in lab:
        row = row[row >= 0]
        out.append(int(np.bincount(row).argmax()) if len(row) else -1)
    return out
