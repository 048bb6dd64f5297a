"""The summation order of normalize_features' fit, checked against NumPy on the CPU.

np.mean / np.std over axis 0 add the rows one after another for some layouts and sum each column pairwise for
others.  batch._axis0_is_inner decides which from the caller's strides; the GPU fit then runs the matching mode
(tests/test_zscore_layouts_gpu.py).  Here the rule itself is compared with what NumPy does, so a NumPy whose
iterator chose differently would fail on every machine, not only on one with a GPU."""
import numpy as np
import pytest

from dsp_audioreclabs_b200.batch import _axis0_is_inner

N = 1001


def _data(shape, seed):
    # a large offset and a wide spread: the two summation orders differ in the last bits of nearly every column
    rng = np.random.default_rng(seed)
    return rng.standard_normal(shape) * 1e3 + 0.1


def layouts():
    c = _data((N, 15), 1)
    f = np.asfortranarray(_data((N, 15), 2))
    return {
        "C": c,
        "F": f,
        "transposed": np.ascontiguousarray(_data((15, N), 3)).T,
        "C rows strided": _data((2 * N, 15), 4)[::2],
        "C columns strided": _data((N, 30), 5)[:, ::2],
        "C reversed": _data((N, 15), 6)[::-1],
        "C both reversed": _data((N, 15), 7)[::-1, ::-1],
        "F rows strided": np.asfortranarray(_data((2 * N, 15), 8))[::2],
        "F reversed": np.asfortranarray(_data((N, 15), 9))[::-1],
        "F columns reversed": np.asfortranarray(_data((N, 15), 10))[:, ::-1],
        "(n,)": _data((N,), 11),
        "(n, 1)": _data((N, 1), 12),
        "(n, 1) column of C": c[:, 3:4],
        "(n, 1) column of F": f[:, 3:4],
        "(n, 1, 1)": _data((N, 1, 1), 13),
        "(n, 3, 5)": _data((N, 3, 5), 14),
        "(n, 3, 5) F": np.asfortranarray(_data((N, 3, 5), 15)),
        "(n, 3, 5) axes moved": np.moveaxis(_data((3, N, 5), 16), 1, 0),
        "(n, 2, 1) F": np.asfortranarray(_data((N, 2, 1), 17)),
        "(n, 1, 2)": _data((N, 1, 2), 18),
        "broadcast column": np.broadcast_to(_data((N, 1), 19), (N, 7)),
        "broadcast row": np.broadcast_to(_data((7,), 20), (N, 7)),
        "equal strides": np.lib.stride_tricks.as_strided(np.asfortranarray(_data((N, 7), 21)), (N, 7), (8, 8)),
    }


def rowwise(fn, x):
    """fn over axis 0 with the rows added one after another (the row-order fit)."""
    x2 = np.ascontiguousarray(x).reshape(len(x), -1)
    s = np.zeros(x2.shape[1])
    for r in x2:
        s = s + r
    mu = s / len(x2)
    if fn is np.mean:
        return mu
    s2 = np.zeros(x2.shape[1])
    for r in x2:
        v = r - mu
        s2 = s2 + v * v
    return np.sqrt(s2 / len(x2))


def columnwise(fn, x):
    """fn of each column as a 1-D array (NumPy's pairwise sum: the pairwise fit)."""
    x2 = np.ascontiguousarray(x).reshape(len(x), -1)
    return np.array([fn(np.ascontiguousarray(x2[:, j])) for j in range(x2.shape[1])])


@pytest.mark.parametrize("name", list(layouts()))
def test_rule_matches_numpy(name):
    x = layouts()[name]
    pairwise = _axis0_is_inner(x)
    for fn in (np.mean, np.std):
        got = np.asarray(fn(x, axis=0)).reshape(-1)
        row, col = rowwise(fn, x), columnwise(fn, x)
        if pairwise:
            assert np.array_equal(got, col), (name, fn.__name__)
        else:
            assert np.array_equal(got, row), (name, fn.__name__)
        # the layout tells the two orders apart: the other order gives other bits
        if not name.startswith("broadcast"):
            assert not np.array_equal(got, row if pairwise else col), (name, fn.__name__)


def test_rule_on_torch_tensors():
    """torch_ops / device.zscore_device decide on the tensor; x.numpy() has the same layout."""
    torch = pytest.importorskip("torch")
    t = torch.from_numpy(_data((15, N), 30))
    for view in (t, t.T, t.T[::2], t[:, ::2], t[:1].T, t.T.unsqueeze(-1)):
        assert _axis0_is_inner(view) == _axis0_is_inner(view.numpy()), tuple(view.stride())
    assert _axis0_is_inner(t.T) and not _axis0_is_inner(t)


def test_single_row_and_short_columns():
    for x in (_data((1, 15), 40), _data((1,), 41), _data((5, 15), 42), np.asfortranarray(_data((7, 3), 43))):
        assert np.array_equal(np.mean(x, axis=0).reshape(-1), columnwise(np.mean, x))
        if not _axis0_is_inner(x):
            assert np.array_equal(np.mean(x, axis=0).reshape(-1), rowwise(np.mean, x))
