"""GPU: the reference's driver scripts run UNCHANGED on the CUDA drop-in modules (BASELINE configs[0] and the
ablation sweep of configs[3]; SURVEY.md section 4 item 5).

The scripts come from oracle/_ref -- an unmodified copy of the reference made by oracle/make_ref.py in the build
container (git-ignored, shipped with the snapshot).  Each script runs twice on the SAME data directory, as a
subprocess: once as the reference itself (CPU, stub plotting modules) and once through
`python -m dsp_audioreclabs_b200.run <script>` (drop-in `config` / `src.*`, CUDA).  Outputs must be identical:
the drop-in serves the float64 replay kernel's values, which are the reference's own bit for bit.  The run
report proves the CUDA path ran (kernel launches > 0, modules resolved to the drop-in) and that a whole data
tree costs ONE front-end launch per configuration (SURVEY.md 8 f2).  Without that copy those tests skip;
test_config1_feature_matrix_matches_the_stored_reference_matrix still holds the CUDA path to the matrix the reference
built (tests/golden/scripts_golden.npz).
"""
import json
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu
REF = os.path.join(ROOT, "oracle", "_ref")
STUBS = os.path.join(ROOT, "tests", "stubs")
GOLD = os.path.join(ROOT, "tests", "golden", "scripts_golden.npz")
DROPIN = os.path.join(ROOT, "dsp_audioreclabs_b200", "dropin")
needs_ref = pytest.mark.skipif(not os.path.isfile(os.path.join(REF, "run.py")),
                               reason="oracle/_ref (copy of the reference's scripts, oracle/make_ref.py) is not present")


@pytest.fixture(scope="module")
def work(tmp_path_factory):
    from oracle import synth
    base = tmp_path_factory.mktemp("scripts")
    data = base / "data"
    assert synth.write_config1_dataset(data) == 200
    ref = base / "ref"
    shutil.copytree(REF, ref)                      # the reference writes results/ next to its config.py
    return {"base": base, "data": str(data), "ref": str(ref)}


def run_reference(work, script, args):
    env = dict(os.environ, PYTHONPATH=STUBS, SPEECH_DATA_DIR=work["data"], OMP_NUM_THREADS="1")
    subprocess.run([sys.executable, script] + args, cwd=work["ref"], env=env, check=True, stdout=subprocess.DEVNULL)
    return os.path.join(work["ref"], "results")


def run_dropin(work, script, args, tag):
    results = str(work["base"] / f"results_{tag}")
    report = str(work["base"] / f"report_{tag}.jsonl")
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([ROOT, STUBS]), SPEECH_DATA_DIR=work["data"],
               DSP_RESULTS_DIR=results, DSP_RUN_REPORT=report)
    # the script file is the reference's own, started from ITS directory like a user would
    subprocess.run([sys.executable, "-m", "dsp_audioreclabs_b200.run", os.path.join(work["ref"], script)] + args,
                   cwd=work["ref"], env=env, check=True, stdout=subprocess.DEVNULL)
    rep = json.loads(open(report).read().strip().splitlines()[-1])
    assert "error" not in rep, rep
    assert rep["gpu_launches"] > 0
    assert rep["src.audio_processing"].startswith(DROPIN) and rep["config"].startswith(DROPIN)
    return results, rep


@needs_ref
def test_run_py_feature_experiment_unchanged(work):
    """BASELINE configs[0]: python run.py --experiment feature --window-type hamming (run.py:46-53,84-130)."""
    args = ["--experiment", "feature", "--window-type", "hamming"]
    ours, rep = run_dropin(work, "run.py", args, "feature")
    text = open(os.path.join(ours, "exp3_feature_analysis", "feature_analysis.txt"), encoding="utf-8").read()
    theirs = run_reference(work, "run.py", args)
    assert text == open(os.path.join(theirs, "exp3_feature_analysis", "feature_analysis.txt"), encoding="utf-8").read()
    assert text == str(np.load(GOLD)["feature_analysis"])        # captured from /root/reference by oracle/gen_golden_scripts.py
    assert os.path.exists(os.path.join(ours, "exp3_feature_analysis", "feature_distribution.png"))
    # 200 files, one configuration: ONE front-end launch
    assert rep["frontend_launches"] == [["tree", 200]]


@needs_ref
def test_ablation_frame_length_knn_unchanged(work):
    """python ablation_study.py --experiment frame_length --classifier knn (ablation_study.py:146-163 ->
    train_model.py:21-110,113-207): 12 frame lengths, the whole tree re-processed per value, z-score + KNN."""
    args = ["--experiment", "frame_length", "--classifier", "knn"]
    ours, rep = run_dropin(work, "ablation_study.py", args, "ablation")
    got = json.load(open(os.path.join(ours, "ablation_frame_length", "results.json"), encoding="utf-8"))
    theirs = run_reference(work, "ablation_study.py", args)
    want = json.load(open(os.path.join(theirs, "ablation_frame_length", "results.json"), encoding="utf-8"))
    assert list(got["results"]) == list(want["results"]) == [str(v) for v in (8, 10, 12, 15, 18, 20, 25, 30, 35, 40, 45, 50)]
    for k in want["results"]:
        assert got["results"][k] == want["results"][k], k          # accuracy, train accuracy, confusion matrix
    assert {k: got[k] for k in ("experiment", "dataset", "param_name")} == {k: want[k] for k in ("experiment", "dataset", "param_name")}
    # one launch per sweep value, decoded once
    assert rep["frontend_launches"] == [["tree", 200]] * 12


@needs_ref
def test_load_dataset_matrix_matches_the_reference(work):
    """X (200, 15) of SpeechRecognitionExperiment.load_dataset('hamming') (experiments/run_experiments.py:45-126)
    equals the matrix the reference built in the build container -- bit for bit, rows compared per class."""
    harness = work["base"] / "harness.py"
    out = work["base"] / "x.npz"
    harness.write_text(
        "import sys, numpy as np\n"
        f"sys.path.append({work['ref']!r})\n"
        "import config\n"
        "from experiments.run_experiments import SpeechRecognitionExperiment as E\n"
        f"e = E(config.DATA_DIR, {str(work['base'] / 'res_h')!r})\n"
        "X, y, names = e.load_dataset('hamming')\n"
        f"np.savez({str(out)!r}, X=X, y=y, names=np.array(names))\n")
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([ROOT, STUBS]), SPEECH_DATA_DIR=work["data"],
               DSP_RESULTS_DIR=str(work["base"] / "res_h"))
    subprocess.run([sys.executable, "-m", "dsp_audioreclabs_b200.run", str(harness)], cwd=str(work["base"]), env=env, check=True,
                   stdout=subprocess.DEVNULL)
    z, g = np.load(out), np.load(GOLD)
    X, y = z["X"], z["y"]
    order = np.lexsort(tuple(X[:, j] for j in range(X.shape[1] - 1, -1, -1)) + (y,))
    assert X.shape == (200, 15) and X.dtype == np.float64
    assert np.array_equal(y[order], g["y_sorted"])
    assert np.array_equal(X[order], g["X_sorted"])
    assert list(z["names"]) == list(g["names"])


def test_config1_feature_matrix_matches_the_stored_reference_matrix(tmp_path):
    """The same comparison without a copy of the reference: the per-file loop of load_dataset('hamming') (sorted class
    folders, glob('*.wav') per class, process_audio_file + extract_features_from_frames with config's constants) over
    the drop-in modules reproduces the stored (200, 15) matrix bit for bit, and the whole tree costs ONE launch."""
    from oracle import synth
    data = tmp_path / "data"
    assert synth.write_config1_dataset(data) == 200
    harness = tmp_path / "harness.py"
    out = tmp_path / "x.npz"
    harness.write_text(
        "import glob, os, numpy as np\n"
        "import config\n"
        "from src.audio_processing import process_audio_file\n"
        "from src.feature_extraction import extract_features_from_frames\n"
        "X, y, names = [], [], None\n"
        "classes = sorted(c for c in os.listdir(config.DATA_DIR) if os.path.isdir(os.path.join(config.DATA_DIR, c)) and not c.startswith('.'))\n"
        "for label, c in enumerate(classes):\n"
        "    for p in glob.glob(os.path.join(config.DATA_DIR, c, '*.wav')):\n"
        "        frames, _, _ = process_audio_file(p, config.FRAME_LENGTH, config.FRAME_SHIFT, 'hamming', True,\n"
        "                                          config.ENERGY_HIGH_RATIO, config.ENERGY_LOW_RATIO, config.ZCR_THRESHOLD_RATIO)\n"
        "        vec, names = extract_features_from_frames(frames, method='statistical')\n"
        "        X.append(vec)\n"
        "        y.append(label)\n"
        f"np.savez({str(out)!r}, X=np.array(X), y=np.array(y), names=np.array(names))\n")
    report = str(tmp_path / "report.jsonl")
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([ROOT, STUBS]), SPEECH_DATA_DIR=str(data),
               DSP_RESULTS_DIR=str(tmp_path / "results"), DSP_RUN_REPORT=report)
    subprocess.run([sys.executable, "-m", "dsp_audioreclabs_b200.run", str(harness)], cwd=str(tmp_path), env=env, check=True,
                   stdout=subprocess.DEVNULL)
    rep = json.loads(open(report).read().strip().splitlines()[-1])
    assert "error" not in rep, rep
    assert rep["src.audio_processing"].startswith(DROPIN) and rep["config"].startswith(DROPIN)
    assert rep["gpu_launches"] > 0 and rep["frontend_launches"] == [["tree", 200]]
    z, g = np.load(out), np.load(GOLD)
    X, y = z["X"], z["y"]
    order = np.lexsort(tuple(X[:, j] for j in range(X.shape[1] - 1, -1, -1)) + (y,))
    assert X.shape == (200, 15) and X.dtype == np.float64
    assert np.array_equal(y[order], g["y_sorted"])
    assert np.array_equal(X[order], g["X_sorted"])
    assert list(z["names"]) == list(g["names"])


@needs_ref
def test_compare_feature_methods_unchanged(work):
    """compare_feature_methods.py (module-level script: statistical vs zero-padded sequence features, KNN / SVM /
    decision tree on both, compare_feature_methods.py:43-176): every accuracy it prints is the reference's.  KNN runs
    on the CUDA path (D = 15: tensor-core filter; D = 2 max_len: tensor-core scan); SVM / tree are delegated to the
    reference's own src/models.py.  Both passes over the tree share ONE front-end launch."""
    env = dict(os.environ, PYTHONPATH=STUBS, SPEECH_DATA_DIR=work["data"], OMP_NUM_THREADS="1")
    ref_out = subprocess.run([sys.executable, "compare_feature_methods.py"], cwd=work["ref"], env=env, check=True,
                             capture_output=True, text=True).stdout
    report = str(work["base"] / "report_cmp.jsonl")
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([ROOT, STUBS]), SPEECH_DATA_DIR=work["data"],
               DSP_RESULTS_DIR=str(work["base"] / "results_cmp"), DSP_RUN_REPORT=report, OMP_NUM_THREADS="1")
    our_out = subprocess.run([sys.executable, "-m", "dsp_audioreclabs_b200.run", os.path.join(work["ref"], "compare_feature_methods.py")],
                             cwd=work["ref"], env=env, check=True, capture_output=True, text=True).stdout
    keep = lambda text: [ln for ln in text.splitlines() if any(ch.isdigit() for ch in ln)]
    assert keep(our_out) == keep(ref_out)
    assert len(keep(our_out)) > 15
    rep = json.loads(open(report).read().strip().splitlines()[-1])
    assert rep["gpu_launches"] > 0 and rep["frontend_launches"] == [["tree", 200]]
