"""bench.py --dump-outputs: the arrays of the last timed step land in DIR/<name>.npy (float32 / float64, at most 64 MB),
and two runs with the same arguments write the same values (the inputs are generated from fixed seeds)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

SMALL = ["--utts", "3000", "--train-utts", "3000", "--steps", "4", "--warmup", "3", "--no-e2e", "--no-cpu-baseline", "--no-knn"]


def run_bench(args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, cwd=ROOT, capture_output=True, text=True)


def test_steps_must_be_positive():
    r = run_bench(["--steps", "0"])
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr


@pytest.mark.gpu
def test_dumped_outputs_are_complete_and_repeatable(tmp_path):
    dumps = []
    for run in ("a", "b"):
        out = tmp_path / run
        r = run_bench(SMALL + ["--dump-outputs", str(out)])
        assert r.returncode == 0, r.stderr[-3000:]
        line = json.loads(r.stdout.strip().splitlines()[-1])
        assert line["steps"] == 4 and line["value"] > 0
        dumps.append({f[:-4]: np.load(out / f) for f in sorted(os.listdir(out))})
    a, b = dumps
    assert sorted(a) == sorted(b) == sorted(["utterances", "labels", "zscores", "stats", "start", "end", "n_epd_frames",
                                             "n_frames", "status", "frame_utterances", "frame_offsets", "frame_energy",
                                             "frame_magnitude", "frame_zcr"])
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    for name in a:
        assert a[name].dtype in (np.float32, np.float64), name
        assert np.array_equal(a[name], b[name]), name
    n = 3000
    assert a["labels"].shape == (n,) and a["zscores"].shape == (n, 15) and a["stats"].shape == (n, 15)
    assert np.array_equal(a["utterances"], np.arange(n))
    assert set(np.unique(a["labels"])) <= set(range(10))
    assert np.all(a["start"] < a["end"]) and np.all(a["n_frames"] > 0)
    nf = a["n_frames"][a["frame_utterances"].astype(np.int64)]
    assert np.array_equal(np.diff(a["frame_offsets"]), nf)
    assert len(a["frame_energy"]) == len(a["frame_zcr"]) == a["frame_offsets"][-1]
