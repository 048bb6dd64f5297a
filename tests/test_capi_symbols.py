"""CPU: the C-ABI library builds, loads and exports every symbol include/dspfront.h declares
(no compute without a GPU), and the host-only arithmetic entry points agree with the oracle."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    text = open(os.path.join(ROOT, "include", "dspfront.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(dsp_[a-z0-9_]+)\s*\(", text)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    from dsp_audioreclabs_b200 import _capi
    if not os.path.exists(_capi.LIB_PATH):
        g.build()
    return _capi.load_library()


def test_every_declared_symbol_is_exported_and_bound(lib):
    from dsp_audioreclabs_b200 import _capi
    declared = header_functions()
    assert len(declared) >= 25
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in dspfront.h but not exported"
    assert sorted(_capi.SIGNATURES) == declared      # the ctypes stub binds exactly the header
    assert lib.dsp_abi_version() == 2


def test_no_cpu_fallback(lib):
    """Without a CUDA device the context cannot be created and says why.  On a machine with a GPU this test runs
    itself again in a child process that is shown no device."""
    import torch
    if torch.cuda.is_available():
        r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", f"{__file__}::test_no_cpu_fallback"],
                           cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True, text=True)
        assert r.returncode == 0 and "1 passed" in r.stdout, r.stdout[-3000:]
        return
    from dsp_audioreclabs_b200 import _capi
    h = C.c_void_p()
    rc = lib.dsp_create(0, C.byref(h))
    assert rc == _capi.DSP_ERR_NO_DEVICE and not h.value
    assert b"no CPU path" in lib.dsp_last_error()
    from dsp_audioreclabs_b200 import batch
    with pytest.raises(_capi.DspError):
        batch.frontend_batch(np.zeros(1000, np.int16), np.array([0, 1000]), 256, 128)


def test_plan_and_frame_count_match_the_oracle(lib):
    from dsp_audioreclabs_b200 import batch
    from oracle import frontend_oracle as fo
    rng = np.random.default_rng(0)
    for _ in range(300):
        n, fl, fs = int(rng.integers(0, 5000)), int(rng.integers(1, 600)), int(rng.integers(1, 600))
        assert lib.dsp_frame_count(n, fl, fs) == fo.feature_frame_count(n, fl, fs)
        x = np.zeros(n)
        assert len(fo.frame_signal(x, fl, fs, "rectangular")) == fo.feature_frame_count(n, fl, fs)
    lens = rng.integers(0, 3000, 50)
    off = np.concatenate([[0], np.cumsum(lens)])
    p = batch.make_params(256, 128)
    fo_, eo, mx = batch.plan(off, p)
    assert mx == lens.max()
    assert np.array_equal(np.diff(fo_), [fo.feature_frame_count(int(n), 256, 128) for n in lens])
    assert np.array_equal(np.diff(eo), [((n - 256) // 128 + 1) if n >= 256 else 0 for n in lens])
    with pytest.raises(ValueError):
        batch.plan(np.array([0, 10, 5]), p)
    with pytest.raises(ValueError):
        batch.make_params(256, 128, "blackman")


def test_windows_match_numpy(lib):
    from dsp_audioreclabs_b200 import batch
    for n in (1, 2, 3, 64, 255, 256, 1102, 2205):
        assert np.array_equal(batch.window("rectangular", n), np.ones(n))
        assert np.allclose(batch.window("hamming", n), np.hamming(n), rtol=1e-14, atol=1e-16)
        w = batch.window("hanning", n)
        assert np.allclose(w, np.hanning(n), rtol=1e-14, atol=1e-16)
        if n > 1:
            assert w[0] == 0.0 and w[-1] == 0.0          # exact zeros: they decide ZCR signs
