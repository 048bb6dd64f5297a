"""CPU, worlds 2 and 3 over gloo: the exchange logic of dist.ShardedDeviceDTW (template shards, one candidate
all-gather, the k-way merge, the vote), with and without a per-query cost bound.  The compute callbacks are the
(self-)oracle here -- the product has no CPU path."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

K = 3


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _data():
    rng = np.random.default_rng(33)

    def seq(n, c):
        return (rng.standard_normal((n, 4)) * 0.2 + np.cos(np.arange(n)[:, None] * (0.2 + 0.1 * c))).astype(np.float32)
    labels = np.arange(13) % 4
    temps = [seq(int(rng.integers(4, 25)), c) for c in labels]
    temps[9] = temps[1].copy()            # the same template in two shards: ties go to the lower index
    labels[9] = 3
    quers = [seq(int(rng.integers(4, 25)), c) for c in (0, 1, 2, 3, 1, 0, 2)]
    quers[1] = temps[1].copy()            # cost 0 against templates 1 and 9
    return temps, labels, quers


def _bounds(cost):
    """Per-query bounds over the full cost matrix: none (inf), exactly 0 for the query equal to templates 1 and 9 (a
    tie at the radius across shards), below every cost (empty), negative, NaN, between the 1st and 2nd cost, and
    exactly the 3rd cost."""
    s = np.sort(cost, axis=1)
    return np.array([np.inf, 0.0, s[2, 0] * 0.5, -1.0, np.nan, (s[5, 0] + s[5, 1]) / 2, s[6, 2]])


def _select(cost_row, labels, k, bound, index_base=0):
    """The first min(k, #{cost <= bound}) templates by (cost, index) with cost <= bound, then (inf, -1, -1)."""
    keep = np.nonzero(cost_row <= bound)[0]
    order = keep[np.lexsort((keep, cost_row[keep]))][:k]
    c = np.full(k, np.inf)
    i = np.full(k, -1, dtype=np.int64)
    l = np.full(k, -1, dtype=np.int32)
    c[:len(order)], i[:len(order)], l[:len(order)] = cost_row[order], order + index_base, labels[order]
    return c, i, l


def _expected(bound):
    from oracle import mfcc_dtw_oracle as mo
    temps, labels, quers = _data()
    cost = mo.dtw_matrix(quers, temps)
    b = np.full(len(quers), np.inf) if bound is None else bound
    rows = [_select(cost[q], labels, K, b[q]) for q in range(len(quers))]
    return tuple(np.stack(a) for a in zip(*rows))


def _vote(lab):
    out = []
    for row in lab:
        row = row[row >= 0]
        out.append(int(np.bincount(row).argmax()) if len(row) else -1)
    return np.array(out, dtype=np.int32)


def _unpack(feats, offsets, lengths):
    off = offsets.numpy()
    n = np.diff(off) if lengths is None else lengths.numpy()
    return [feats.numpy()[off[i]:off[i] + n[i]] for i in range(len(off) - 1)]


def _oracle_topk(t_feats, t_offsets, t_labels, q_feats, q_offsets, k, index_base, bound=None, t_lengths=None,
                 q_lengths=None, max_q_frames=None):
    """local_topk honouring the bound: the shard's templates with cost <= bound, sorted by (cost, index)."""
    from oracle import mfcc_dtw_oracle as mo
    temps, quers = _unpack(t_feats, t_offsets, t_lengths), _unpack(q_feats, q_offsets, q_lengths)
    labels = t_labels.numpy()
    cost = mo.dtw_matrix(quers, temps).reshape(len(quers), len(temps))
    b = np.full(len(quers), np.inf) if bound is None else bound.numpy()
    rows = [_select(cost[q], labels, k, b[q], index_base) for q in range(len(quers))]
    c, i, l = (np.stack(a) for a in zip(*rows))
    return torch.from_numpy(c), torch.from_numpy(i), torch.from_numpy(l.astype(np.int32))


def _oracle_merge_vote(cost, idx, lab):
    """merge_vote: the k best of the R lists by (cost, index), empty slots ignored, then the majority label."""
    r, m, k = cost.shape
    c, i, l = (a.permute(1, 0, 2).reshape(m, -1).numpy() for a in (cost, idx, lab))
    out = []
    for q in range(m):
        ok = np.nonzero(i[q] >= 0)[0]
        order = ok[np.lexsort((i[q][ok], c[q][ok]))][:k]
        out.append(l[q][order])
    return torch.from_numpy(_vote(out))


def _pack(seqs, pad=0):
    """Packed float32 feats and int64 offsets, with `pad` unused rows after each sequence; lengths int32."""
    off = np.concatenate([[0], np.cumsum([len(s) + pad for s in seqs])]).astype(np.int64)
    flat = np.zeros((max(int(off[-1]), 1), 4), np.float32)
    for s, o in zip(seqs, off):
        flat[o:o + len(s)] = s
    return torch.from_numpy(flat), torch.from_numpy(off), torch.tensor([len(s) for s in seqs], dtype=torch.int32)


def _worker(rank, world, port, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from dsp_audioreclabs_b200 import dist as ddist
    from oracle import mfcc_dtw_oracle as mo
    temps, labels, quers = _data()
    tb = ddist.balanced_bounds(len(temps), world)
    # world 3 passes template lengths (rows padded between templates), world 2 the offsets alone
    tf, to, tl = _pack(temps[tb[rank]:tb[rank + 1]], pad=2 if world == 3 else 0)
    qf, qo, _ = _pack(quers)
    sd = ddist.ShardedDeviceDTW(K, local_topk=_oracle_topk, merge_vote=_oracle_merge_vote)
    sd.fit(tf, to, torch.from_numpy(labels[tb[rank]:tb[rank + 1]].astype(np.int32)), tl if world == 3 else None)
    assert sd.index_base == tb[rank] and sd.n_total == len(temps)
    bound = _bounds(mo.dtw_matrix(quers, temps))
    res = {}
    for name, b in (("free", None), ("bounded", torch.from_numpy(bound))):
        c, i, l = sd.kneighbors(qf, qo, bound=b)
        res[name + "_cost"], res[name + "_idx"], res[name + "_lab"] = c.numpy(), i.numpy(), l.numpy()
        res[name + "_pred"] = sd.predict(qf, qo, bound=b).numpy()
    np.savez(os.path.join(out_dir, f"w{world}r{rank}.npz"), **res)
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_device_dtw_matches_single_rank(tmp_path, world):
    """Merged neighbours and votes on every rank equal the single-rank oracle, with no bound and with per-query
    bounds that keep everything, cut at a tie, empty a query (below every cost, negative, NaN) or cut between costs."""
    from oracle import mfcc_dtw_oracle as mo
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    temps, _, quers = _data()
    bound = _bounds(mo.dtw_matrix(quers, temps))
    for name, b in (("free", None), ("bounded", bound)):
        cost, idx, lab = _expected(b)
        if b is not None:
            assert np.all(idx[2:5] == -1)                                          # emptied
            assert list(idx[1]) == [1, 9, -1] and list(cost[1][:2]) == [0.0, 0.0]     # the tie at the radius
            assert np.sum(idx[5] >= 0) == 1 and np.all(idx[6] >= 0)
        for r in range(world):
            o = np.load(tmp_path / f"w{world}r{r}.npz")
            assert np.array_equal(o[name + "_idx"], idx), (name, r)
            assert np.array_equal(o[name + "_cost"], cost), (name, r)
            assert np.array_equal(o[name + "_lab"], lab), (name, r)
            assert np.array_equal(o[name + "_pred"], _vote(lab)), (name, r)
