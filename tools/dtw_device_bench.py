#!/usr/bin/env python3
"""MFCC + DTW template matching on device tensors vs the host calls, at the BASELINE config 5 shape (DESIGN.md 3.5).

    python tools/dtw_device_bench.py [queries] [templates] [--out FILE]

DTW: queries and templates as tools/dtw_config5.py generates them (MFCC sequences of 400 synthetic utterances of
U(0.5, 1.5) s; queries = a random one + 1 % noise), k = 3, one GPU.  Host path: mfcc_dtw.DTWClassifier.kneighbors
(wall time of the call: uploads, cost matrix, top k, downloads).  Device path: device.DeviceDTW.topk on inputs already
on the device (CUDA events around the call), its fraction of abandoned pairs, and whether its outputs equal the host
path's bit for bit.  MFCC: device.DeviceMFCC.run (CUDA events, PCM and endpoints on the device) vs mfcc_batch (wall
time of the host call) over 2,000 utterances.  Prints one JSON line, with the card's name and power limit read in the
same run."""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from dsp_audioreclabs_b200 import batch, device, mfcc_dtw
from oracle import synth

REPEATS = 3


def card():
    name = torch.cuda.get_device_name(0)
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        power = r.stdout.strip() or "not read"
    except (OSError, subprocess.TimeoutExpired):
        power = "not read"
    return name, power


def event_seconds(fn):
    """Median over REPEATS of CUDA-event time around fn() on torch's current stream."""
    out = []
    for _ in range(REPEATS):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b) / 1e3)
    return float(np.median(out))


def wall_seconds(fn):
    out = []
    for _ in range(REPEATS):
        t0 = time.perf_counter()
        fn()
        out.append(time.perf_counter() - t0)
    return float(np.median(out))


def main():
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    out_path = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
    if out_path in args:
        args.remove(out_path)
    nq = int(args[0]) if len(args) > 0 else 10000
    nt = int(args[1]) if len(args) > 1 else 10000
    if not torch.cuda.is_available():
        raise SystemExit("dtw_device_bench needs a CUDA device")
    ctx = batch.default_context(0)
    name, power = card()

    # ---- DTW at the config 5 shape (tools/dtw_config5.py's generator)
    nbase = 400
    base = [synth.utterance_pcm(i, int(n), seed0=99) for i, n in enumerate(synth.ragged_lengths(nbase, 0.5, 1.5, seed=2))]
    s, o, l = batch.pack_aligned(base)
    res = batch.frontend_batch(s, o, 1102, 441, "hamming", lengths=l, emit_frames=False, ctx=ctx)
    mf, off = mfcc_dtw.mfcc_batch(s, o, res.start, res.end, lengths=l, ctx=ctx)
    seqs = [mf[off[b]:off[b + 1]] for b in range(nbase)]
    rng = np.random.default_rng(5)
    queries = [seqs[i] + 0.01 * rng.standard_normal(seqs[i].shape).astype(np.float32) for i in rng.integers(0, nbase, nq)]
    tsel = rng.integers(0, nbase, nt)
    templates = [seqs[i] for i in tsel]
    labels = (tsel % 10).astype(np.int32)
    qlen, tlen = np.array([len(a) for a in queries]), np.array([len(a) for a in templates])

    clf = mfcc_dtw.DTWClassifier(3, ctx=ctx).fit(templates, labels)
    host = clf.kneighbors(queries)                                   # warm-up: the host call's buffers are allocated here
    t_host = wall_seconds(lambda: clf.kneighbors(queries))

    qf, qo = mfcc_dtw.pack_sequences(queries, 13)
    tf, to = mfcc_dtw.pack_sequences(templates, 13)
    qf, qo, tf, to = (torch.from_numpy(a).cuda() for a in (qf, qo, tf, to))
    dtw = device.DeviceDTW(3).fit(tf, to, torch.from_numpy(labels).cuda())
    max_q = int(qlen.max())
    got = dtw.topk(qf, qo, max_q_frames=max_q)                       # warm-up: scratch sized here
    torch.cuda.synchronize()
    t_dev = event_seconds(lambda: dtw.topk(qf, qo, max_q_frames=max_q))
    scored, abandoned = dtw.last_stats()
    same = all(np.array_equal(a.cpu().numpy(), b) for a, b in zip(got, host))

    # ---- MFCC: 2,000 utterances
    n_utt = 2000
    utts = [base[i % nbase] for i in range(n_utt)]
    s2, o2, l2 = batch.pack_aligned(utts)
    r2 = batch.frontend_batch(s2, o2, 1102, 441, "hamming", lengths=l2, emit_frames=False, ctx=ctx)
    audio_s = float(l2.sum()) / 44100.0
    mfcc_dtw.mfcc_batch(s2, o2, r2.start, r2.end, lengths=l2, ctx=ctx)
    t_mfcc_host = wall_seconds(lambda: mfcc_dtw.mfcc_batch(s2, o2, r2.start, r2.end, lengths=l2, ctx=ctx))
    dm = device.DeviceMFCC(o2, lengths=l2)
    d_s, d_st, d_en = (torch.from_numpy(a).cuda() for a in (s2, r2.start, r2.end))
    dm.run(d_s, d_st, d_en)
    torch.cuda.synchronize()
    t_mfcc_dev = event_seconds(lambda: dm.run(d_s, d_st, d_en))

    line = {
        "tool": "dtw_device_bench",
        "card": name, "power_limit": power,
        "dtw": {"queries": nq, "templates": nt, "k": 3,
                "query_frames_min_mean_max": [int(qlen.min()), float(qlen.mean()), int(qlen.max())],
                "template_frames_min_mean_max": [int(tlen.min()), float(tlen.mean()), int(tlen.max())],
                "host_call_s": t_host, "device_topk_s": t_dev, "speedup": t_host / t_dev,
                "device_pairs_per_s": nq * nt / t_dev,
                "pairs_scored": scored, "pairs_abandoned": abandoned, "fraction_abandoned": abandoned / float(nq * nt),
                "device_equals_host": bool(same)},
        "mfcc": {"utterances": n_utt, "audio_s": audio_s,
                 "host_call_s": t_mfcc_host, "host_audio_s_per_s": audio_s / t_mfcc_host,
                 "device_s": t_mfcc_dev, "device_audio_s_per_s": audio_s / t_mfcc_dev},
        "timing": f"median of {REPEATS}; host calls: wall time; device calls: CUDA events, inputs already on the device",
    }
    text = json.dumps(line)
    print(text, flush=True)
    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
