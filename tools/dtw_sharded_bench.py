#!/usr/bin/env python3
"""Row-sharded DTW template matching at the BASELINE config 5 shape: the host path (dist.ShardedDTW, lists of NumPy
arrays through the host call) against the device path (dist.ShardedDeviceDTW, device tensors through the fused top-k),
alternated in one process per GPU.

    python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 tools/dtw_sharded_bench.py \
        [queries] [templates] [--reps R] [--out FILE]
    python tools/dtw_sharded_bench.py              # one rank

Data: tools/dtw_config5.py's generator (MFCC sequences of 400 synthetic utterances of U(0.5, 1.5) s; queries = a
random one + 1 % noise), k = 3, templates sharded by row over the ranks, queries replicated, one NCCL all-gather of
the candidates.  Each timing is the maximum over ranks of a host clock around the call, started after a barrier and a
device synchronise and stopped after a device synchronise; the median over `reps` alternations is reported.  The
device path's inputs are already on the device; the host path's call includes its uploads and downloads.

Second leg (rank 0, all templates on one GPU): DeviceDTW.topk with a rejection bound -- the median over queries of
the 1st-neighbour cost, the same for every query -- against the unbounded call, with last_stats for both.

Rank 0 prints one JSON line (and appends it to FILE), with the GPU's name, power limit and max SM clock read in the
same run."""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

from dsp_audioreclabs_b200 import batch, device, mfcc_dtw, dist as ddist
from oracle import synth

K = 3


def gpu_info(index):
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(index)], capture_output=True, text=True, timeout=30)
        return r.stdout.strip() or "not read"
    except (OSError, subprocess.TimeoutExpired):
        return "not read"


def config5_data(nq, nt, ctx):
    nbase = 400
    base = [synth.utterance_pcm(i, int(n), seed0=99) for i, n in enumerate(synth.ragged_lengths(nbase, 0.5, 1.5, seed=2))]
    s, o, l = batch.pack_aligned(base)
    res = batch.frontend_batch(s, o, 1102, 441, "hamming", lengths=l, emit_frames=False, ctx=ctx)
    mf, off = mfcc_dtw.mfcc_batch(s, o, res.start, res.end, lengths=l, ctx=ctx)
    seqs = [mf[off[b]:off[b + 1]] for b in range(nbase)]
    rng = np.random.default_rng(5)
    queries = [seqs[i] + 0.01 * rng.standard_normal(seqs[i].shape).astype(np.float32) for i in rng.integers(0, nbase, nq)]
    tsel = rng.integers(0, nbase, nt)
    return queries, [seqs[i] for i in tsel], (tsel % 10).astype(np.int32)


def timed(fn, dev, world):
    """Max over ranks of the host-clock time of fn() between device synchronises; returns (seconds, fn's result)."""
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize(dev)
    t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()), out


def main():
    args = [a for a in sys.argv[1:]]
    out_path = reps = None
    if "--out" in args:
        i = args.index("--out"); out_path = args[i + 1]; del args[i:i + 2]
    if "--reps" in args:
        i = args.index("--reps"); reps = int(args[i + 1]); del args[i:i + 2]
    reps = reps or 5
    nq = int(args[0]) if len(args) > 0 else 10000
    nt = int(args[1]) if len(args) > 1 else 10000
    if not torch.cuda.is_available():
        raise SystemExit("dtw_sharded_bench needs CUDA devices")
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29541")
    os.environ.setdefault("RANK", "0")
    os.environ.setdefault("WORLD_SIZE", "1")
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    world, rank = dist.get_world_size(), dist.get_rank()
    ctx = batch.default_context(local)

    queries, templates, labels = config5_data(nq, nt, ctx)
    tb = ddist.balanced_bounds(nt, world)
    lo, hi = int(tb[rank]), int(tb[rank + 1])
    max_q = max(len(q) for q in queries)
    host = ddist.ShardedDTW(K, device=dev).fit(templates[lo:hi], labels[lo:hi])
    qf, qo = (torch.from_numpy(a).to(dev) for a in mfcc_dtw.pack_sequences(queries, 13))
    tf, to = (torch.from_numpy(a).to(dev) for a in mfcc_dtw.pack_sequences(templates[lo:hi], 13))
    sdev = ddist.ShardedDeviceDTW(K).fit(tf, to, torch.from_numpy(labels[lo:hi]).to(dev))

    run_host = lambda: host.kneighbors(queries)
    run_dev = lambda: sdev.kneighbors(qf, qo, max_q_frames=max_q)
    run_host(), run_dev()                                       # warm-up: buffers and scratch are sized here
    t_host, t_dev = [], []
    for _ in range(reps):
        t, h_out = timed(run_host, dev, world); t_host.append(t)
        t, d_out = timed(run_dev, dev, world); t_dev.append(t)
    same = all(np.array_equal(a, b.cpu().numpy()) for a, b in zip(h_out, d_out))
    flag = torch.tensor([int(same)], dtype=torch.int32, device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    same = bool(flag.item())

    line = None
    if rank == 0:
        tfa, toa = (torch.from_numpy(a).to(dev) for a in mfcc_dtw.pack_sequences(templates, 13))
        one = device.DeviceDTW(K, device=dev).fit(tfa, toa, torch.from_numpy(labels).to(dev))
        free = one.topk(qf, qo, max_q_frames=max_q)
        radius = float(free[0][:, 0].median().item())
        bound = torch.full((nq,), radius, dtype=torch.float64, device=dev)
        one.topk(qf, qo, max_q_frames=max_q, bound=bound)
        leg = {}
        for name, b in (("unbounded", None), ("bounded", bound)):
            ts = []
            for _ in range(reps):
                torch.cuda.synchronize(dev)
                t0 = time.perf_counter()
                out = one.topk(qf, qo, max_q_frames=max_q, bound=b)
                torch.cuda.synchronize(dev)
                ts.append(time.perf_counter() - t0)
            scored, abandoned = one.last_stats()
            leg[name] = {"seconds": float(np.median(ts)), "pairs_scored": scored, "pairs_abandoned": abandoned,
                         "queries_with_a_match": int((out[1][:, 0] >= 0).sum().item())}
        kept = out                                              # the bounded call's outputs
        within = free[0] <= radius
        leg["bounded_equals_filtered_unbounded"] = bool(
            torch.equal(torch.where(within, free[1], -1), kept[1]) and
            torch.equal(torch.where(within, free[0], float("inf")), kept[0]))
        leg["bound"] = "median over queries of the 1st-neighbour cost: %.6g, the same for every query" % radius
        pairs = nq * nt
        line = {
            "tool": "dtw_sharded_bench", "gpus": world, "gpu": gpu_info(local),
            "queries": nq, "templates": nt, "k": K,
            "host_ShardedDTW_s": float(np.median(t_host)), "device_ShardedDeviceDTW_s": float(np.median(t_dev)),
            "host_pairs_per_s": pairs / float(np.median(t_host)), "device_pairs_per_s": pairs / float(np.median(t_dev)),
            "speedup": float(np.median(t_host)) / float(np.median(t_dev)),
            "host_s_all": t_host, "device_s_all": t_dev,
            "device_equals_host": same,
            "rejection_leg_one_gpu": leg,
            "timing": "median of %d alternations; each the max over ranks of a host clock between device synchronises; "
                      "host path incl. its copies, device path on inputs already on the device" % reps,
        }
        text = json.dumps(line)
        print(text, flush=True)
        if out_path:
            os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
            with open(out_path, "a") as f:
                f.write(text + "\n")
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
