"""normalize_features on the GPU against the NumPy oracle for every memory layout the caller may hand in.

NumPy sums axis 0 row by row or column by column pairwise depending on the layout (tests/test_zscore_rule.py), so the
oracle is applied to the very same array object: mean, std and z-scores must be bit-identical (np.array_equal)."""
import numpy as np
import pytest

from oracle import frontend_oracle as fo

pytestmark = pytest.mark.gpu

NS = (1, 2, 8, 9, 127, 128, 129, 1000, 100003)


def _data(shape, seed):
    rng = np.random.default_rng(seed)
    return rng.standard_normal(shape) * 1e3 + 0.1 * rng.standard_normal(shape[1:] or ())


def layouts(n, seed=0):
    """name -> array of n rows, every layout whose axis-0 sum order NumPy chooses differently or could."""
    c = _data((n, 15), seed)
    return {
        "C": c,
        "F": np.asfortranarray(_data((n, 15), seed + 1)),
        "transposed": np.ascontiguousarray(_data((15, n), seed + 2)).T,
        "C rows strided": _data((2 * n, 15), seed + 3)[::2],
        "C columns strided": _data((n, 30), seed + 4)[:, ::2],
        "C reversed": _data((n, 15), seed + 5)[::-1],
        "F rows strided": np.asfortranarray(_data((2 * n, 15), seed + 6))[::2],
        "F reversed": np.asfortranarray(_data((n, 15), seed + 7))[::-1],
        "(n,)": _data((n,), seed + 8),
        "(n, 1)": _data((n, 1), seed + 9),
        "(n, 1) column of C": c[:, 4:5],
        "(n, 1, 1)": _data((n, 1, 1), seed + 10),
        "(n, 3, 5)": _data((n, 3, 5), seed + 11),
        "(n, 3, 5) F": np.asfortranarray(_data((n, 3, 5), seed + 12)),
    }


def check_same(got, ref, what):
    for g, r, name in zip(got, ref, ("z", "mean", "std")):
        assert np.shape(g) == np.shape(r) and np.array_equal(g, r), (what, name)


@pytest.mark.parametrize("name", list(layouts(1)))
@pytest.mark.parametrize("n", NS)
def test_fit_every_layout(ctx, n, name):
    from dsp_audioreclabs_b200 import batch
    x = layouts(n, seed=n)[name]
    check_same(batch.zscore(x, ctx=ctx), fo.zscore(x), (n, name))


def test_fit_deep_pairwise_tree(ctx):
    """1,000,000 rows, Fortran order: each column is a 1-D pairwise sum many levels deep."""
    from dsp_audioreclabs_b200 import batch
    x = np.asfortranarray(_data((1_000_000, 2), 7))
    check_same(batch.zscore(x, ctx=ctx), fo.zscore(x), "1e6 x 2 F")


def test_given_mean_and_std(ctx):
    from dsp_audioreclabs_b200 import batch
    for name, x in layouts(129, seed=50).items():
        _, mu, sd = fo.zscore(x[::-1].copy())
        # fitted statistics handed back, as arrays of one row's shape
        check_same(batch.zscore(x, mu, sd, ctx=ctx), fo.zscore(x, mu, sd), (name, "arrays"))
        # scalars, one of them zero (std 0 -> 1)
        for m, s in ((0.25, 3.0), (-1.5, 0.0)):
            z, gm, gs = batch.zscore(x, m, s, ctx=ctx)
            rz, rm, rs = fo.zscore(x, m, s)
            assert np.array_equal(z, rz), (name, m, s)
            assert np.array_equal(np.broadcast_to(gm, np.shape(rz)[1:]), np.broadcast_to(rm, np.shape(rz)[1:])), (name, m)
            assert np.array_equal(np.broadcast_to(gs, np.shape(rz)[1:]), np.broadcast_to(rs, np.shape(rz)[1:])), (name, s)


@pytest.mark.parametrize("order", ["C", "F"])
def test_constant_columns(ctx, order):
    from dsp_audioreclabs_b200 import batch
    x = _data((1000, 6), 60)
    x[:, 1] = 0.0
    x[:, 4] = 0.1                           # constant, but its mean is not exact: std may come out as a tiny non-zero
    x = np.asarray(x, order=order)
    z, mu, sd = batch.zscore(x, ctx=ctx)
    check_same((z, mu, sd), fo.zscore(x), order)
    assert sd[1] == 1.0 and np.all(z[:, 1] == 0.0)


def test_device_and_torch_ops(ctx):
    """device.zscore_device and torch_ops.zscore_fit / zscore_apply: normalize_features(t.cpu().numpy())."""
    import torch
    from dsp_audioreclabs_b200 import device, torch_ops  # noqa: F401  (registers torch.ops.dsp_audioreclabs)
    ops = torch.ops.dsp_audioreclabs
    dev = torch.device("cuda", 0)
    for n in (1, 9, 129, 1000, 100003):
        base = torch.from_numpy(_data((n, 15), n + 70)).to(dev)
        wide = torch.from_numpy(_data((15, n), n + 71)).to(dev)
        views = {"C": base, "transposed": wide.T, "C rows strided": base[::2], "C columns strided": base[:, ::3],
                 "(n, 1) of transposed": wide.T[:, 2:3], "(n, 1)": base[:, 5:6], "F rows strided": wide.T[::2]}
        for name, t in views.items():
            x = t.cpu().numpy()
            ref = fo.zscore(x)
            out, mu, sd = device.zscore_device(t, ctx=ctx)
            torch.cuda.synchronize()
            check_same((out.cpu().numpy(), mu.cpu().numpy(), sd.cpu().numpy()), ref, ("zscore_device", n, name))
            mu2, sd2 = ops.zscore_fit(t)
            z2 = ops.zscore_apply(t, mu2, sd2)
            check_same((z2.cpu().numpy(), mu2.cpu().numpy(), sd2.cpu().numpy()), ref, ("torch_ops", n, name))
            # apply with given statistics
            q = t.flip(0)
            out, _, _ = device.zscore_device(q, mu2, sd2, ctx=ctx)
            rq = fo.zscore(q.cpu().numpy(), ref[1], ref[2])[0]
            assert np.array_equal(out.cpu().numpy(), rq) and np.array_equal(ops.zscore_apply(q, mu2, sd2).cpu().numpy(), rq), (n, name)


@pytest.mark.parametrize("d", [1, 15, 40])
def test_apply_f32(ctx, d):
    """zscore_apply_f32 (the benchmark's path): float32 statistics widened exactly, then (x - mean) / std in float64,
    a zero std counting as 1."""
    import torch
    from dsp_audioreclabs_b200 import device
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(d)
    stats = (rng.standard_normal((70001, d)) * 50 + 3).astype(np.float32)
    mean = rng.standard_normal(d) * 10
    std = np.abs(rng.standard_normal(d)) + 0.01
    std[d // 2] = 0.0
    out = device.zscore_apply_f32(torch.from_numpy(stats).to(dev), torch.from_numpy(mean).to(dev),
                                  torch.from_numpy(std).to(dev), ctx=ctx)
    torch.cuda.synchronize()
    ref = (stats.astype(np.float64) - mean) / np.where(std == 0, 1.0, std)
    assert np.array_equal(out.cpu().numpy(), ref)
