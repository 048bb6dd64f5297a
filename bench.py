#!/usr/bin/env python3
"""Headline benchmark: audio-seconds processed per second by the full pipeline --
features + endpoints + KNN classify (BASELINE.json `metric`).

Workload per GPU and step (BASELINE.json configs[1] batch through the pipeline of configs[2]): 100,000 synthetic
1 s utterances (44.1 kHz int16 PCM, SURVEY.md 8(d) recipe generated on the device), frame 256 / shift 128, the three
window types cycled across steps -> fused front end (DC removal, peak normalisation, endpoint detection, framing +
window, energy / magnitude / ZCR, 15 statistics) -> z-score with the train set's mean / std -> KNN (k = 3) against a
100,000-utterance train set whose features were extracted by the same front end, with the same window type (one fitted
classifier per window, as a reference run uses one --window-type for train and test), before the timed region.
N = 1: the whole train set lives on the GPU.  N > 1 (one rank per GPU, weak scaling: 100,000 query utterances per
GPU): the train rows are sharded over the ranks; every step all-gathers the ranks' query features, scores ALL of them
against the local rows, exchanges the packed top-k candidates in ONE NCCL all-gather and merges + votes
(SURVEY.md 8(e), `dist.ShardedKNN.predict_sharded`).

  python bench.py [--gpus N] [--steps K] [--warmup W]           # our CUDA path
  python bench.py ... --dump-outputs DIR                        # + what the last timed step computed, DIR/<name>.npy
  python bench.py --impl reference ...                          # the reference's own code on the host cores
  torchrun --nproc-per-node N ... bench.py --gpus N ...         # N>1

Rank 0 prints ONE JSON line.  `value` is device-resident throughput of the whole pipeline (CUDA events, max over
ranks); `roofline` is the dominant kernel (the fused front end) from CUDA events around its launches inside the same
timed region; `frontend_only` is configs[1] by itself; `e2e` is the same pipeline through the host-buffer API with
the H2D / D2H copies inside the timed region.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SR = 44100
FL, FS = 256, 128
WINDOWS = ("rectangular", "hamming", "hanning")
UTT_LEN = 44100        # samples per utterance: exactly 1 s, packed CSR (every other utterance starts 8 bytes off a
                       # 16-byte boundary: the kernel streams from the boundary below and carries the offset)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=12)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--utts", type=int, default=100000, help="utterances per GPU")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-knn", action="store_true", help="skip the secondary KNN numbers")
    ap.add_argument("--cpu-utts", type=int, default=600, help="utterances in the cpu_baseline sample")
    ap.add_argument("--train-utts", type=int, default=100000, help="utterances of the KNN train set (whole job)")
    ap.add_argument("--knn-path", default="sharded", choices=["sharded", "replicated"],
                    help="N>1: row-sharded train set with the candidate all-gather (north star), or train rows replicated")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (rank 0) to DIR/<name>.npy, for comparing two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# --------------------------------------------------------------------------------------------
def synth_batch_device(n_utts, device, seed, chunk=2048, first_index=0, lengths=None):
    """SURVEY.md 8(d) generator on the GPU: noise floor, 50 ms unvoiced onset, Hann-enveloped
    two-partial burst, DC offset, truncation to int16.  Utterance i has class (first_index + i) mod 10.
    lengths (optional int64 [n_utts], each <= 1.2 s): ragged batch -- every utterance is generated at ITS length (burst
    at the same fractions of it) and the batch is packed back to back.  Returns (samples, CSR offsets[n+1])."""
    import torch
    gen = torch.Generator(device=device)
    gen.manual_seed(seed)
    n = UTT_LEN if lengths is None else int(max(lengths))
    if lengths is None:
        out = torch.zeros(n_utts * n + 64, dtype=torch.int16, device=device)
        view = out[: n_utts * n].view(n_utts, n)
        offsets = np.arange(n_utts + 1, dtype=np.int64) * n
    else:
        offsets = np.concatenate([[0], np.cumsum(np.asarray(lengths, dtype=np.int64))])
        out = torch.zeros(int(offsets[-1]) + 64, dtype=torch.int16, device=device)
        d_len = torch.from_numpy(np.asarray(lengths, dtype=np.int64)).to(device)
    pos = torch.arange(n, device=device, dtype=torch.float32)[None, :]
    t = pos / SR
    on = int(0.050 * SR)
    for c0 in range(0, n_utts, chunk):
        c = min(chunk, n_utts - c0)
        cls = (torch.arange(first_index + c0, first_index + c0 + c, device=device) % 10).float()[:, None]
        u = torch.rand(c, 3, device=device, generator=gen)
        ln = float(n) if lengths is None else d_len[c0:c0 + c, None].float()
        b0 = torch.floor((0.15 + 0.15 * u[:, 0:1]) * ln)
        b1 = torch.floor((0.60 + 0.25 * u[:, 1:2]) * ln)
        f0 = 150.0 + 90.0 * cls + (20.0 * u[:, 2:3] - 10.0)
        x = torch.randn(c, n, device=device, generator=gen) * 0.005
        inb = (pos >= b0) & (pos < b1)
        env = 0.5 - 0.5 * torch.cos(2 * np.pi * (pos - b0) / (b1 - b0 - 1).clamp(min=1))
        burst = 0.6 * (torch.sin(2 * np.pi * f0 * t) + 0.3 * torch.sin(2 * np.pi * (2 * f0 + 5 * cls) * t))
        x += inb * env * burst
        onset = (pos >= b0 - on) & (pos < b0)
        x += onset * torch.randn(c, n, device=device, generator=gen) * 0.03
        x += 0.01
        x.clamp_(-1.0, 32767.0 / 32768.0)
        pcm = torch.trunc(x * 32768.0).to(torch.int16)
        if lengths is None:
            view[c0:c0 + c] = pcm
        else:
            keep = pos < d_len[c0:c0 + c, None].float()            # row-major: rows packed back to back
            out[int(offsets[c0]): int(offsets[c0 + c])] = pcm[keep]
        del x, inb, env, burst, onset, pcm
    return out, offsets


class ClockSampler:
    """nvidia-smi SM clock / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [s.strip() for s in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nme, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# --------------------------------------------------------------------------------------------
# CPU legs: the reference's own code (oracle/_ref, an unmodified copy made by oracle/make_ref.py) when it travelled
# with the snapshot, else the oracle port.  Test/bench infrastructure only -- never on the product path.
REF_DIR = os.path.join(ROOT, "oracle", "_ref")
N_TRAIN_CPU = 100000
_cpu = {}


def _cpu_setup():
    """-> dict(kind, fe(pcm, window) -> 15 stats, zscore(X, mu, sd), clf with predict): the reference's modules when
    oracle/_ref exists (kind 'reference'), else the oracle port (kind 'port')."""
    if _cpu:
        return _cpu
    if os.path.isfile(os.path.join(REF_DIR, "src", "audio_processing.py")):
        sys.path.insert(0, REF_DIR)
        import src.audio_processing as ap
        import src.feature_extraction as fe
        import src.models as mo

        def front(pcm, window):
            # process_audio_file minus the WAV decode (src/audio_processing.py:364-394) + the 'statistical' features
            x = ap.preprocess(pcm / 32768.0)
            s, e, _, _ = ap.endpoint_detection(x, FL, FS, 0.5, 0.1, 1.5)
            frames = ap.frame_signal(x[s:e], FL, FS, window)
            return fe.extract_features_from_frames(frames, method="statistical")[0]

        _cpu.update(kind="reference", front=front, zscore=fe.normalize_features,
                    make_clf=lambda: mo.create_classifier("knn", n_neighbors=3),
                    what="oracle/_ref: the reference's own src.audio_processing / src.feature_extraction / src.models (sklearn KNN)")
    else:
        from oracle import frontend_oracle as fo, knn_oracle as ko

        class _Clf:
            def fit(self, X, y):
                self.X, self.y = X, y

            def predict(self, Q):
                return ko.knn_predict(self.X, self.y, Q, 3)

        _cpu.update(kind="port", front=lambda pcm, window: fo.frontend_utterance(pcm, FL, FS, window)["stats"],
                    zscore=fo.zscore, make_clf=_Clf,
                    what="oracle/frontend_oracle.py + oracle/knn_oracle.py (oracle/_ref is absent)")
    return _cpu


def _cpu_train_set(n_base=512):
    """A 100,000 x 15 train matrix for the CPU KNN: the reference front end on `n_base` generated utterances, resampled
    with 5 % per-feature jitter (running the CPU front end on 100,000 utterances would take ~7 CPU-minutes per core)."""
    from oracle import synth
    c = _cpu_setup()
    base = np.stack([c["front"](synth.utterance_pcm(900000 + i, UTT_LEN, 4242), "hamming") for i in range(n_base)])
    rng = np.random.default_rng(7)
    pick = rng.integers(0, n_base, N_TRAIN_CPU)
    X = base[pick] + rng.standard_normal((N_TRAIN_CPU, 15)) * 0.05 * base.std(axis=0)
    y = (900000 + pick) % 10
    Xn, mu, sd = c["zscore"](X)
    clf = c["make_clf"]()
    clf.fit(Xn, y)
    c.update(clf=clf, mu=mu, sd=sd)


_UTTS = []          # the CPU sample, generated before the timed region (and before the fork: shared copy-on-write)


def _cpu_sample(n):
    from oracle import synth
    while len(_UTTS) < n:
        _UTTS.append(synth.utterance_pcm(len(_UTTS), UTT_LEN, 777))


def _cpu_worker(args):
    """The whole pipeline for a slice of the resident sample on one core: front end per utterance, z-score, KNN predict."""
    first, count = args
    c = _cpu_setup()
    utts = _UTTS[first:first + count]
    t0 = time.perf_counter()
    X = np.stack([c["front"](pcm, WINDOWS[i % 3]) for i, pcm in enumerate(utts)])
    t1 = time.perf_counter()
    c["clf"].predict(c["zscore"](X, c["mu"], c["sd"])[0])
    t2 = time.perf_counter()
    return t2 - t0, t1 - t0


def cpu_baseline_single(n_utts):
    c = _cpu_setup()
    _cpu_train_set()
    _cpu_sample(n_utts)
    dt, dt_fe = _cpu_worker((0, n_utts))
    return {"value": n_utts * (UTT_LEN / SR) / dt, "unit": "audio-s/s", "cores": 1, "kind": c["kind"],
            "frontend_only_value": n_utts * (UTT_LEN / SR) / dt_fe,
            "sample": f"{n_utts} utterances of the same generator/config (1 s, 256/128, windows cycled) through {c['what']}: "
                      f"front end {dt_fe:.1f} s + z-score + KNN(3) predict against a {N_TRAIN_CPU}-row train set {dt - dt_fe:.1f} s"}


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the pipeline on all host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    for v in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS"):
        os.environ[v] = "1"
    c = _cpu_setup()
    _cpu_train_set()                    # before the fork: the workers share the fitted classifier copy-on-write
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    per_worker = 24
    _cpu_sample(cores * per_worker)     # inputs resident before the timed region, the same sample every step (as on the GPU arm)
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        def step(s):
            jobs = [(w * per_worker, per_worker) for w in range(cores)]
            t0 = time.perf_counter()
            pool.map(_cpu_worker, jobs)
            return time.perf_counter() - t0
        for s in range(args.warmup):
            step(s)
        total = sum(step(args.warmup + s) for s in range(args.steps))
    n = cores * per_worker * args.steps
    val = n * (UTT_LEN / SR) / total
    line = {
        "impl": "reference", "metric": METRIC, "value": val,
        "unit": "audio-s/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000.0 * total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": bench_config(args, int(os.environ.get("WORLD_SIZE", "1"))),
        "cpu_baseline": {"value": val, "unit": "audio-s/s", "cores": cores, "kind": c["kind"],
                         "sample": f"{cores * per_worker} utterances per step (a bounded sample of the 100k-utterance batch: per-utterance cost is constant) x {args.steps} steps, multiprocessing.Pool({cores}), {c['what']}; "
                                   f"KNN against a {N_TRAIN_CPU}-row train set fitted before the timed region"},
        "e2e": {"value": val, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


METRIC = "audio-seconds processed/sec (features+endpoints+KNN)"
WORKLOAD = ("configs[1] batch through the configs[2] pipeline: 100k synthetic 1 s utterances per GPU, frame 256 / shift 128, three windows "
            "cycled over steps -> fused front end -> z-score -> KNN(3) vs a 100k-utterance train set framed with the same window")


def bench_config(args, world):
    """The workload both arms are quoted on (the reference arm times a bounded sample of it per step: its
    cpu_baseline.sample says which)."""
    return {"workload": WORKLOAD,
            "utterances_per_gpu": args.utts, "samples_per_utterance": UTT_LEN, "frame_length": FL, "frame_shift": FS,
            "windows": list(WINDOWS), "train_utterances": args.train_utts, "knn_k": 3,
            "parallelism": f"utterance shards x{world}" + ("" if world == 1 else f", KNN train rows {args.knn_path} x{world} (NCCL)"),
            "layout": "packed CSR, no padding between utterances",
            "l2_policy": f"input {args.utts * UTT_LEN * 2 / 1e9:.2f} GB per pass >> 126 MB L2 (no flush needed)"}


def knn_section(dev, ctx):
    """Secondary numbers of the same run (not part of `value`): the classify step alone at BASELINE configs[2] size on one GPU
    (1 M queries x 100 k train rows, D = 15, k = 3: tcgen05 K = 16 candidate filter + float64 certificate) and the
    sequence-feature variant (D = 1024: tcgen05 tensor-core scan), device-resident, CUDA events."""
    import torch
    from dsp_audioreclabs_b200 import device as devapi
    out = {}
    try:
        for tag, (m, n, d) in {"statistical_d15": (1000000, 100000, 15), "sequence_d1024": (131072, 50000, 1024)}.items():
            g = torch.Generator(device=dev).manual_seed(5)
            centers = torch.randn(10, d, device=dev, generator=g, dtype=torch.float64) * 1.5
            ytr = torch.randint(0, 10, (n,), device=dev, generator=g)
            xtr = centers[ytr] + torch.randn(n, d, device=dev, generator=g, dtype=torch.float64)
            yq = torch.randint(0, 10, (m,), device=dev, generator=g)
            xq = centers[yq] + torch.randn(m, d, device=dev, generator=g, dtype=torch.float64)
            knn = devapi.DeviceKNN(3, ctx=ctx, device=dev).fit(xtr.contiguous(), ytr.to(torch.int32))
            knn.predict(xq)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            knn.predict(xq)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            rescanned, kind = knn.last_stats()
            out[tag] = {"queries": m, "train_rows": n, "dim": d, "ms": ms, "queries_per_s": m / (ms / 1e3),
                        "algorithmic_TFLOPs": 2.0 * d * m * n / (ms / 1e3) / 1e12,
                        "scan": {1: "fp32 tiled", 2: "tcgen05 split-fp16 (3 MMA passes)",
                                 3: "tcgen05 K=16 filter, split-fp16 (3 MMA passes), |t|^2 as 16th feature"}.get(kind, "float64"),
                        "rescanned_in_float64": rescanned}
            del xtr, xq, knn
            torch.cuda.empty_cache()
    except Exception as exc:      # secondary numbers must never break the bench line
        out["error"] = repr(exc)
    return out


def traffic_of_record(kernel_src):
    """dram bytes per launch of the front-end kernel from the committed ncu capture of THIS source file (profiles/
    traffic_r02.json carries the sha of csrc/frontend_pipe.cu it was taken on); None when the kernel changed since."""
    import hashlib
    tp = os.path.join(ROOT, "profiles", "traffic_r02.json")
    try:
        rec = json.load(open(tp))
        sha = hashlib.sha256(open(kernel_src, "rb").read()).hexdigest()[:16]
        return rec.get("dram_bytes_per_launch") if rec.get("source_sha16") == sha else None
    except Exception:
        return None


DUMP_MAX_UTTS = 200000      # per-utterance arrays: 236 B an utterance in float64 / float32 -> at most 47 MB
DUMP_FRAME_UTTS = 512       # per-frame arrays for a fixed sample of utterances (<= 343 frames each at 256 / 128)


def dump_outputs(out_dir, fe, qn, labels):
    """What one step of the timed path hands its caller -- KNN labels, z-scored features, the front end's statistics,
    endpoints, frame counts and status per utterance, per-frame energy / magnitude / ZCR -- as out_dir/<name>.npy.
    Integer outputs are stored as float64 (exact).  Batches above DUMP_MAX_UTTS utterances keep a fixed, seeded sample
    of utterances (`utterances` lists which); the per-frame arrays cover a fixed, seeded sample of DUMP_FRAME_UTTS
    utterances (`frame_utterances`), packed back to back at `frame_offsets`."""
    import torch
    n = fe.n_utts
    rows = np.arange(n) if n <= DUMP_MAX_UTTS else np.sort(np.random.default_rng(0).choice(n, DUMP_MAX_UTTS, replace=False))
    f64 = lambda t: t.cpu().numpy().astype(np.float64)
    out = {"utterances": rows.astype(np.float64), "labels": f64(labels)[rows], "zscores": f64(qn)[rows],
           "stats": fe.stats.cpu().numpy()[rows]}
    for name in ("start", "end", "n_epd_frames", "n_frames", "status"):
        out[name] = f64(getattr(fe, name))[rows]
    picked = np.sort(np.random.default_rng(1).choice(n, min(n, DUMP_FRAME_UTTS), replace=False))
    nf = fe.n_frames.cpu().numpy()[picked].astype(np.int64)
    idx = np.concatenate([np.arange(fe.h_feat_offsets[b], fe.h_feat_offsets[b] + k) for b, k in zip(picked, nf)] + [[]])
    idx = torch.from_numpy(idx.astype(np.int64)).to(fe.device)
    out["frame_utterances"] = picked.astype(np.float64)
    out["frame_offsets"] = np.concatenate([[0], np.cumsum(nf)]).astype(np.float64)
    for name in ("energy", "magnitude", "zcr"):
        out[f"frame_{name}"] = getattr(fe, name)[idx].cpu().numpy()
    total = sum(a.nbytes for a in out.values())
    assert total <= 64 << 20 and all(a.dtype in (np.float32, np.float64) for a in out.values()), total
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)
    return total


# --------------------------------------------------------------------------------------------
def run_ours(args):
    import faulthandler
    import torch
    import torch.distributed as dist
    # a rank that waits forever (a collective its peers never enter) must end the run with a stack trace, not hang the box
    faulthandler.dump_traceback_later(int(os.environ.get("BENCH_WATCHDOG_S", "420")), exit=True)
    from dsp_audioreclabs_b200 import batch, device as devapi, dist as ddist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = ddist.bind_to_gpu_numa(local)         # before any pinned allocation: first touch places the staging buffers
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    n_utts = args.utts
    ctx = batch.default_context(local)
    stream = torch.cuda.Stream(device=dev)
    audio_s_per_step = n_utts * (UTT_LEN / SR)

    # ---- train set (outside the timed region, like model weights): rank r owns rows [tb[r], tb[r+1]) -----------------
    tb = ddist.balanced_bounds(args.train_utts, world)
    n_tr = int(tb[rank + 1] - tb[rank])
    # one classifier per window type, as in the reference (a run extracts train AND test features with the same
    # --window-type, run.py:84-130): the step that frames its queries with window w classifies them against models[w]
    models = {}
    with torch.cuda.stream(stream):
        tr_samples, tr_offsets = synth_batch_device(n_tr, dev, seed=990000 + rank, first_index=int(tb[rank]))
        y_tr = (torch.arange(int(tb[rank]), int(tb[rank + 1]), device=dev) % 10).to(torch.int32)
        for w in WINDOWS:
            tr_fe = devapi.DeviceFrontend(tr_offsets, FL, FS, w, ctx=ctx, device=dev)
            tr_fe.run(tr_samples, stream=stream)
            x_tr = tr_fe.stats.double().contiguous()
            if world > 1:
                mean, std = ddist.zscore_stats_allreduce(x_tr)          # one tiny all-reduce (fit time)
                std = torch.where(std == 0, torch.ones_like(std), std)
                x_tr_n, _, _ = devapi.zscore_device(x_tr, mean, std, ctx=ctx)
                knn = ddist.ShardedKNN(3, replicate_below=(0 if args.knn_path == "sharded" else 1 << 62)).fit(x_tr_n.contiguous(), y_tr)
            else:
                x_tr_n, mean, std = devapi.zscore_device(x_tr, ctx=ctx)
                knn = devapi.DeviceKNN(3, ctx=ctx, device=dev).fit(x_tr_n.contiguous(), y_tr)
            models[w] = (mean, std, knn, x_tr_n)
            stream.synchronize()
            del tr_fe
    stream.synchronize()
    del tr_samples
    torch.cuda.empty_cache()

    # ---- query utterances: rank r owns utterances [r*n_utts, (r+1)*n_utts) of the global batch ------------------------
    samples, row_offsets = synth_batch_device(n_utts, dev, seed=1234 + rank, first_index=rank * n_utts)
    y_q = (torch.arange(rank * n_utts, (rank + 1) * n_utts, device=dev) % 10).to(torch.int32)
    frontends = {w: devapi.DeviceFrontend(row_offsets, FL, FS, w, ctx=ctx, device=dev) for w in WINDOWS}
    qn = torch.empty(n_utts, 15, dtype=torch.float64, device=dev)
    ev_fe = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    labels = [None]

    def step(i, timed=None):
        """One pass of the hot path over the rank's batch; everything is enqueued on `stream`."""
        fe = frontends[WINDOWS[i % 3]]
        if timed is not None:
            ev_fe[timed][0].record(stream)
        fe.run(samples, stream=stream)
        if timed is not None:
            ev_fe[timed][1].record(stream)
        mean, std, knn, _ = models[WINDOWS[i % 3]]
        devapi.zscore_apply_f32(fe.stats, mean, std, out=qn, ctx=ctx)
        labels[0] = knn.predict(qn, [n_utts] * world) if world > 1 else knn.predict(qn)

    with torch.cuda.stream(stream):
        for i in range(max(args.warmup, 3)):
            step(i)
    barrier()
    # ---- timed region: K steps, CUDA events on the launching stream ---------------------------------------------------
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    launches0 = ctx.launch_count
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    torch.cuda.cudart().cudaProfilerStart()      # `ncu --profile-from-start off` lists exactly the timed region's launches
    with torch.cuda.stream(stream):
        ev[0].record(stream)
        for i in range(args.steps):
            step(i, timed=i)
            ev[i + 1].record(stream)
    stream.synchronize()
    torch.cuda.cudart().cudaProfilerStop()
    if args.dump_outputs and rank == 0:
        # before anything below reruns the front end or the classifier on these buffers
        nbytes = dump_outputs(args.dump_outputs, frontends[WINDOWS[(args.steps - 1) % 3]], qn, labels[0])
        print(f"bench: outputs of timed step {args.steps} ({WINDOWS[(args.steps - 1) % 3]} window, {nbytes / 1e6:.1f} MB) "
              f"-> {args.dump_outputs}", file=sys.stderr, flush=True)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    launches = ctx.launch_count - launches0
    total_ms = ev[0].elapsed_time(ev[-1])
    step_ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(args.steps)]
    fe_ms = [a.elapsed_time(b) for a, b in ev_fe]
    tmax = torch.tensor([total_ms, float(np.mean(fe_ms))], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    total_ms_max, fe_ms_max = float(tmax[0].item()), float(tmax[1].item())
    value = world * audio_s_per_step * args.steps / (total_ms_max / 1000.0)

    # ---- roofline of the dominant kernel (frontend_pipe_kernel, csrc/frontend_pipe.cu): CUDA events around its
    # launches inside the timed region --------------------------------------------------------------------------------
    per_window = {}
    for wi, w in enumerate(WINDOWS):
        ms = [fe_ms[i] for i in range(args.steps) if i % 3 == wi]
        if ms:
            per_window[w] = {"ms": float(np.mean(ms)), "algorithmic_bytes": frontends[w].algorithmic_bytes()}
    alg_bytes = float(np.mean([v["algorithmic_bytes"] for v in per_window.values()]))
    avg_fe_ms = float(np.mean(fe_ms))
    avg_step_ms = float(np.mean(step_ms))
    peak, peak_src = measured_hbm_peak()
    achieved = alg_bytes / (avg_fe_ms / 1000.0) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic_of_record(os.path.join(ROOT, "dsp_audioreclabs_b200", "csrc", "frontend_pipe.cu")),
                "kernel": "frontend_pipe_kernel<true>", "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes, "ms_per_launch": avg_fe_ms,
                "share_of_step": avg_fe_ms / avg_step_ms}
    # pipeline-level HBM fraction (SURVEY.md 8(d)): the front end's bytes + 4 D per query + 4 D n_train once + 4 per label
    pipe_bytes = alg_bytes + 4.0 * 15 * n_utts + 4.0 * 15 * args.train_utts + 4.0 * n_utts
    pipeline = {"ms_per_step": avg_step_ms, "frontend_ms": avg_fe_ms, "zscore_knn_ms": avg_step_ms - avg_fe_ms,
                "algorithmic_bytes_per_step": pipe_bytes, "hbm_GBps": pipe_bytes / (avg_step_ms / 1e3) / 1e9,
                "hbm_frac": pipe_bytes / (avg_step_ms / 1e3) / 1e9 / peak,
                "knn": {"queries_per_gpu_per_step": n_utts, "train_rows": args.train_utts, "dim": 15, "k": 3,
                        "train_layout": "whole train set on the GPU" if world == 1 else
                        (f"rows sharded x{world}; per step: own queries against own rows (threshold hints), all-gather of the query features + hints, "
                         f"ONE NCCL all-gather of the packed top-k candidates ({world * n_utts} queries x 3 x 16 B per rank), merge + vote" if args.knn_path == "sharded" else
                         f"rows all-gathered once at fit (replicated), no per-step exchange")}}
    if world > 1 and args.knn_path == "sharded":
        # the same steps with the train rows all-gathered once at fit (the D = 15 fast path: no per-step exchange)
        try:
            with torch.cuda.stream(stream):
                for i in range(3):
                    models[WINDOWS[i]][2].predict_replicated(qn)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for i in range(6):
                    fe = frontends[WINDOWS[i % 3]]
                    fe.run(samples, stream=stream)
                    mean, std, knn, _ = models[WINDOWS[i % 3]]
                    devapi.zscore_apply_f32(fe.stats, mean, std, out=qn, ctx=ctx)
                    knn.predict_replicated(qn)
                e1.record(stream)
            stream.synchronize()
            t = torch.tensor([e0.elapsed_time(e1) / 6], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            pipeline["replicated_train_rows"] = {"ms_per_step_max_over_ranks": float(t.item()),
                                                 "audio_s_per_s": world * audio_s_per_step / (float(t.item()) / 1e3)}
        except Exception as exc:
            pipeline["replicated_train_rows"] = {"error": repr(exc)}
    frontend_only = {"workload": "configs[1]: batched front end only", "value": world * audio_s_per_step / (fe_ms_max / 1e3),
                     "unit": "audio-s/s", "ms_per_launch_max_over_ranks": fe_ms_max}

    # ---- the ragged variant of configs[1] (SURVEY.md 8(d) config 2: L ~ U(0.8, 1.2) s): every utterance generated at its
    # own length and packed back to back, i.e. arbitrary lengths AND arbitrary alignment; front end only, Hamming ---------
    per_config = {}
    try:
        rng = np.random.default_rng(99 + rank)
        lens = (rng.uniform(0.8, 1.2, n_utts) * SR).astype(np.int64)
        r_samples, r_off = synth_batch_device(n_utts, dev, seed=4321 + rank, first_index=rank * n_utts, lengths=lens)
        torch.cuda.synchronize()
        rf = devapi.DeviceFrontend(r_off, FL, FS, "hamming", ctx=ctx, device=dev)
        with torch.cuda.stream(stream):
            for _ in range(3):
                rf.run(r_samples, stream=stream)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(6):
                rf.run(r_samples, stream=stream)
            e1.record(stream)
        stream.synchronize()
        r_ms = e0.elapsed_time(e1) / 6
        r_bytes = rf.algorithmic_bytes()
        per_config["ragged_0.8-1.2s_packed_csr"] = {
            "utterances": int(len(r_off) - 1), "audio_s": float(r_off[-1] / SR), "ms": r_ms,
            "audio_s_per_s": float(r_off[-1] / SR) / (r_ms / 1e3), "hbm_frac": r_bytes / (r_ms / 1e3) / 1e9 / peak,
            "replayed_in_float64": int((rf.status >= 0x100).sum().item()),
            "odd_sample_offsets": int((r_off[:-1] & 1).sum()), "starts_not_16B_aligned": int(((r_off[:-1] * 2) % 16 != 0).sum())}
        del rf, r_samples
        torch.cuda.empty_cache()
    except Exception as exc:      # secondary numbers must never break the bench line
        per_config["error"] = repr(exc)

    # ---- BASELINE configs[3] on the same batch: the reference's default geometry and the ends of its ablation grids,
    # one launch per configuration (front end only, Hamming) ---------------------------------------------------------
    try:
        for gfl, gfs in ((1102, 441), (2205, 441), (1102, 132), (512, 256), (128, 64)):
            gf = devapi.DeviceFrontend(row_offsets, gfl, gfs, "hamming", ctx=ctx, device=dev)
            with torch.cuda.stream(stream):
                for _ in range(2):
                    gf.run(samples, stream=stream)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for _ in range(3):
                    gf.run(samples, stream=stream)
                e1.record(stream)
            stream.synchronize()
            g_ms = e0.elapsed_time(e1) / 3
            per_config[f"frame_{gfl}_shift_{gfs}"] = {"ms": g_ms, "audio_s_per_s": audio_s_per_step / (g_ms / 1e3),
                                                      "hbm_frac": gf.algorithmic_bytes() / (g_ms / 1e3) / 1e9 / peak,
                                                      "replayed_in_float64": int((gf.status >= 0x100).sum().item())}
            del gf
    except Exception as exc:      # secondary numbers must never break the bench line
        per_config["geometry_error"] = repr(exc)

    # ---- parity spot check against the oracle on a few of the benchmarked utterances -------------------------------------
    parity = None
    with torch.cuda.stream(stream):
        step(1)                                   # hamming; on EVERY rank: the sharded classify step is a collective
    stream.synchronize()
    if rank == 0:
        from oracle import frontend_oracle as fo
        f = frontends["hamming"]
        nchk = 24
        host = samples[: nchk * UTT_LEN].cpu().numpy()
        st, en, nf = f.start[:nchk].cpu().numpy(), f.end[:nchk].cpu().numpy(), f.n_frames[:nchk].cpu().numpy()
        zc = f.zcr.cpu().numpy()
        bad = 0
        for b in range(nchk):
            r = fo.frontend_utterance(host[b * UTT_LEN:(b + 1) * UTT_LEN], FL, FS, "hamming")
            o = int(f.h_feat_offsets[b])
            bad += not (r["start"] == st[b] and r["end"] == en[b] and r["n_frames"] == nf[b]
                        and np.array_equal(r["zcr"], zc[o:o + nf[b]].astype(np.float64)))
        parity = {"utterances_checked": nchk, "endpoint_or_zcr_mismatches": int(bad),
                  "replayed_in_float64": int((f.status >= 0x100).sum().item()),
                  "knn_accuracy_on_generated_classes": float((labels[0] == y_q).double().mean().item())}
        if world == 1:
            # KNN labels of the first queries against the float64 oracle on the SAME z-scored features
            from oracle import knn_oracle as ko
            nq = 64
            ref = ko.knn_predict(models["hamming"][3].cpu().numpy(), y_tr.cpu().numpy(), qn[:nq].cpu().numpy(), 3)
            parity["knn_label_mismatches_vs_oracle"] = int((ref != labels[0][:nq].cpu().numpy()).sum())
            parity["knn_not_certified_by_first_pass,scan_kind"] = list(models["hamming"][2].last_stats())

    # ---- e2e: the same pipeline through the host-buffer API (H2D + D2H inside) --------------------------------------------
    e2e = None
    if not args.no_e2e:
        host_models = {}
        for w in WINDOWS:
            mean, std, _, x_tr_n = models[w]
            if world > 1:
                xt = torch.cat(ddist._all_gather_rows(x_tr_n.contiguous()), dim=0).cpu().numpy()
                yt = torch.cat(ddist._all_gather_rows(y_tr.contiguous()), dim=0).cpu().numpy()
            else:
                xt, yt = x_tr_n.cpu().numpy(), y_tr.cpu().numpy()
            host_models[w] = (mean.cpu().numpy(), std.cpu().numpy(), batch.KNN(3, ctx=ctx).fit(xt, yt))
        h_samples = torch.empty(samples.numel(), dtype=torch.int16, pin_memory=True)
        h_samples.copy_(samples)
        torch.cuda.synchronize()
        hs = h_samples.numpy()

        def e2e_step(i):
            mu_h, sd_h, hknn = host_models[WINDOWS[i % 3]]
            res = batch.frontend_batch(hs, row_offsets, FL, FS, WINDOWS[i % 3], emit_frames=False, ctx=ctx)
            q = batch.zscore(res.stats.astype(np.float64), mu_h, sd_h, ctx=ctx)[0]
            return res, q, hknn.predict(q)

        res, q, pred = e2e_step(0)
        barrier()
        t0 = time.perf_counter()
        for i in range(args.e2e_steps):
            res, q, pred = e2e_step(i)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
        d2h = sum(a.nbytes for a in (res.start, res.end, res.n_epd_frames, res.n_frames, res.status, res.stats)) + 2 * q.nbytes + pred.nbytes
        e2e = {"value": world * audio_s_per_step * args.e2e_steps / dt, "unit": "audio-s/s",
               "h2d_bytes_per_step": int(hs.nbytes + 3 * row_offsets.nbytes + 2 * q.nbytes), "d2h_bytes_per_step": int(d2h),
               "steps": args.e2e_steps, "h2d_GBps_per_gpu": hs.nbytes * args.e2e_steps / dt / 1e9,
               "call": "batch.frontend_batch (dsp_frontend_batch_host: pinned host samples, chunked H2D/compute/D2H overlap; endpoints + frame counts + "
                       "status + 15 statistics read back) -> batch.zscore (dsp_zscore_host) -> batch.KNN.predict (dsp_knn_predict_host): host arrays in, labels out"}
        del h_samples, hs

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "audio-s/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": total_ms_max / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "i16->f32/f64", "data": "synthetic",
            "config": bench_config(args, world),
            "roofline": roofline, "pipeline": pipeline, "frontend_only": frontend_only, "per_window": per_window,
            "per_config": per_config, "clocks": clocks,
            "e2e": e2e, "gpu_launches": int(launches), "parity": parity, "numa": numa,
        }
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_single(args.cpu_utts)
        if world == 1 and not args.no_knn:
            line["knn"] = knn_section(dev, ctx)
        print(json.dumps(line), flush=True)
    faulthandler.cancel_dump_traceback_later()
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
