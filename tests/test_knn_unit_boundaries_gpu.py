"""Work units of the D <= 15 tensor-core filter (csrc/knn_tc16.cu): a pruned call uses 128-query units when it has few
units per SM and 256-query units otherwise (knn_prune_unit_queries); unpruned calls use 256.  Query counts around the unit
boundaries, with tile pruning off, automatic and forced (tuning key knn_prune), must give the float64 oracle's neighbours
and labels, and a call large enough for 256-query pruned units must give the unpruned call's."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def clustered(rng, n, d=15, centers=12, spread=0.3):
    c = rng.standard_normal((centers, d)) * np.linspace(3.0, 0.2, d)
    lab = rng.integers(0, centers, n)
    return c[lab] + rng.standard_normal((n, d)) * spread * np.linspace(1.0, 0.1, d), lab


@pytest.mark.parametrize("mode", (0, 1, 2))
@pytest.mark.parametrize("m", (127, 128, 129, 255, 257))
def test_query_counts_at_unit_boundaries(ctx, m, mode):
    from dsp_audioreclabs_b200 import batch
    from oracle import knn_oracle as ko
    rng = np.random.default_rng(m)
    train, labels = clustered(rng, 3000 + m)
    q = clustered(rng, m)[0]
    ctx.set_tuning("knn_prune", mode)
    try:
        knn = batch.KNN(3, ctx=ctx).fit(train, labels)
        _, idx, _ = knn.kneighbors(q)
        pred = knn.predict(q)
    finally:
        ctx.set_tuning("knn_prune", 1)
    assert np.array_equal(idx, ko.knn_topk(train, q, 3)[0])
    assert np.array_equal(pred, ko.knn_predict(train, labels, q, 3))


def test_pruned_256_query_units_match_unpruned(ctx):
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    m = 8 * sms * 256 + 129                      # kPruneUnitsPerSm units of 256 per SM, and a ragged last unit
    rng = np.random.default_rng(21)
    train, labels = clustered(rng, 20000)
    q = clustered(rng, m)[0]
    from dsp_audioreclabs_b200 import batch
    got = {}
    for mode in (0, 2):
        ctx.set_tuning("knn_prune", mode)
        try:
            knn = batch.KNN(3, ctx=ctx).fit(train, labels)
            got[mode] = knn.kneighbors(q)[1], knn.predict(q)
        finally:
            ctx.set_tuning("knn_prune", 1)
    assert np.array_equal(got[0][0], got[2][0])
    assert np.array_equal(got[0][1], got[2][1])
