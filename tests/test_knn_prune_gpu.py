"""Tile pruning of the D <= 15 tensor-core filter (csrc/knn_tc16.cu, tuning key knn_prune: 0 off, 1 automatic, 2 always).
Pruning changes which train tiles the filter visits, never the answer: neighbour indices and labels stay bit-exact."""
import contextlib
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MODES = (0, 1, 2)


@contextlib.contextmanager
def prune_mode(ctx, mode):
    ctx.set_tuning("knn_prune", mode)
    try:
        yield
    finally:
        ctx.set_tuning("knn_prune", 1)


def topk(ctx, mode, train, labels, q, k=3):
    from dsp_audioreclabs_b200 import batch
    with prune_mode(ctx, mode):
        knn = batch.KNN(k, ctx=ctx).fit(train, labels)
        _, idx, _ = knn.kneighbors(q)
        return idx, knn.predict(q)


def test_tuning_key_range(ctx):
    for bad in (-1, 3):
        with pytest.raises(ValueError):
            ctx.set_tuning("knn_prune", bad)


@pytest.mark.parametrize("mode", MODES)
def test_sklearn_fixture(ctx, golden_knn, mode):
    k = golden_knn
    idx, pred = topk(ctx, mode, k["d15/train_norm"], k["d15/train_labels"], k["d15/query_norm"])
    assert np.array_equal(idx, k["d15/nbr_idx"])
    assert np.array_equal(pred, k["d15/pred"])


@pytest.mark.parametrize("mode", MODES)
def test_config3_fixture(ctx, mode):
    from conftest import GOLDEN
    from dsp_audioreclabs_b200 import batch
    from oracle.gen_golden_knn3 import checksum, config3_data
    g = np.load(os.path.join(GOLDEN, "knn_config3_golden.npz"))
    xtr, ytr, xq, _ = config3_data()
    if not np.array_equal(checksum(xtr, xq), g["checksum"]):
        pytest.skip("numpy's random stream differs from the one the fixture was generated with")
    tn, mu, sd = batch.zscore(xtr, ctx=ctx)
    qn, _, _ = batch.zscore(xq, mu, sd, ctx=ctx)
    idx, pred = topk(ctx, mode, tn, ytr, qn)
    assert np.array_equal(idx, g["nbr_idx"])
    assert np.array_equal(pred, g["pred"])


def clustered(rng, n, d=15, centers=12, spread=0.3):
    """Features shaped like the statistical ones: a few dominant directions, tight clusters."""
    c = rng.standard_normal((centers, d)) * np.linspace(3.0, 0.2, d)
    lab = rng.integers(0, centers, n)
    return c[lab] + rng.standard_normal((n, d)) * spread * np.linspace(1.0, 0.1, d), lab


def check_forced(ctx, train, labels, q):
    from oracle import knn_oracle as ko
    idx, pred = topk(ctx, 2, train, labels, q)
    assert np.array_equal(idx, ko.knn_topk(train, q, 3)[0])
    assert np.array_equal(pred, ko.knn_predict(train, labels, q, 3))


def test_duplicate_rows_split_across_tiles(ctx):
    rng = np.random.default_rng(11)
    base, lab = clustered(rng, 3000)
    train = np.concatenate([base, base[::7], base[::13]])         # copies land in other tiles of the median splits
    labels = np.concatenate([lab, (lab[::7] + 1) % 12, (lab[::13] + 2) % 12])
    q = np.concatenate([base[::5], base[::5] + 1e-9, clustered(rng, 500)[0]])
    check_forced(ctx, train, labels, q)


def test_neighbours_tied_at_the_radius(ctx):
    """Integer lattice: exact float64 distances, many rows at exactly the k-th distance, in different tiles."""
    rng = np.random.default_rng(12)
    g = np.stack(np.meshgrid(np.arange(16), np.arange(16), np.arange(12), indexing="ij"), -1).reshape(-1, 3).astype(np.float64)
    train = np.zeros((len(g), 15))
    train[:, :3] = g
    labels = rng.integers(0, 5, len(train))
    q = np.zeros((1000, 15))
    q[:, :3] = rng.integers(0, 16, (1000, 3)) + rng.choice([0.0, 0.5], (1000, 3))
    check_forced(ctx, train, labels, q)


def test_queries_far_outside_the_train_cloud(ctx):
    rng = np.random.default_rng(13)
    train, labels = clustered(rng, 5000)
    q = clustered(rng, 600)[0]
    q[:200, 0] += 60.0                                            # far away, still inside the filter's range
    q[200:210] *= 40.0                                            # outside the filter's range: float64 rescan
    check_forced(ctx, train, labels, q)


def test_all_queries_identical(ctx):
    rng = np.random.default_rng(14)
    train, labels = clustered(rng, 4000)
    check_forced(ctx, train, labels, np.repeat(train[17:18] + 0.01, 777, axis=0))


@pytest.mark.parametrize("n,m", [(1000 + 37, 1000 + 3), (128 * 9, 256 * 3), (64, 300), (5000, 1)])
def test_ragged_sizes(ctx, n, m):
    rng = np.random.default_rng(n + m)
    train, labels = clustered(rng, n)
    check_forced(ctx, train, labels, clustered(rng, m)[0])


def test_isotropic_data_takes_the_fallback(ctx, capfd):
    """An isotropic Gaussian in 15 dimensions: the lists keep most tiles, the automatic mode walks every tile; same answer."""
    rng = np.random.default_rng(15)
    ytr = rng.integers(0, 10, 20000)
    train = rng.standard_normal((20000, 15))
    q = rng.standard_normal((4000, 15))
    ref = topk(ctx, 0, train, ytr, q)
    os.environ["DSP_KNN_DEBUG"] = "1"
    try:
        capfd.readouterr()
        got = topk(ctx, 1, train, ytr, q)
        err = capfd.readouterr().err
    finally:
        del os.environ["DSP_KNN_DEBUG"]
    assert "every tile walked" in err, err
    assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1])
    assert np.array_equal(topk(ctx, 2, train, ytr, q)[0], ref[0])


@pytest.mark.parametrize("shards", [2, 8])
def test_row_sharded_hints_with_pruning(ctx, golden_knn, shards):
    """Bounded calls (dsp_knn_topk_bounded_device) with tile pruning forced: the bound is min(seed radius, hint)."""
    import torch
    from dsp_audioreclabs_b200 import device
    k = golden_knn
    dev = torch.device("cuda", 0)
    xn = torch.from_numpy(k["d15/train_norm"]).to(dev)
    y = torch.from_numpy(k["d15/train_labels"].astype(np.int32)).to(dev)
    q = torch.from_numpy(k["d15/query_norm"]).to(dev)
    m = q.shape[0]
    with prune_mode(ctx, 2):
        bounds = np.linspace(0, xn.shape[0], shards + 1).astype(int)
        knns = [device.DeviceKNN(3, ctx=ctx, device=dev, index_base=int(bounds[r])).fit(
            xn[bounds[r]:bounds[r + 1]].contiguous(), y[bounds[r]:bounds[r + 1]].contiguous()) for r in range(shards)]
        owner = torch.arange(m, device=dev) % shards
        own_kth = torch.stack([kn.topk(q)[0][:, 2] for kn in knns])
        bound = own_kth.gather(0, owner[None, :])[0].contiguous()
        cd, ci, cl = [], [], []
        for kn in knns:
            d2, idx, lab = kn.topk(q, bound)
            cd.append(d2); ci.append(idx); cl.append(lab)
        labels, idx, _ = knns[0].merge_vote(torch.stack(cd), torch.stack(ci), torch.stack(cl))
        torch.cuda.synchronize()
    assert np.array_equal(idx.cpu().numpy(), k["d15/nbr_idx"])
    assert np.array_equal(labels.cpu().numpy(), k["d15/pred"])
