"""Where the time of one bench-shaped KNN predict goes: torch.profiler (CUDA activities) over 12 calls.

  python tools/knn_launch_split.py [--calls 12] [--out launch_split.json]

Workload: the train and query features of bench.py (100k synthetic utterances each, frame 256 / shift 128, hamming
window, device front end, z-score with the train set's statistics), DeviceKNN(3).predict with the default tuning (tile
pruning automatic).  Every device activity of a call (kernels, memsets, copies) is put in one of four groups:

  seed    the first knn_tc16_filter_kernel launch of a pruned call (each unit against its nearest tiles)
  prep    everything before the main filter pass except the seed pass: curve keys, sorts, pack, unit boxes, seed lists,
          bounds, tile lists, start thresholds, memsets
  main    the last knn_tc16_filter_kernel launch
  tail    everything after it: rerank (certificate), refine, rescan, vote

Calls are synchronised and separated by an idle gap, so the trace splits into calls at the gaps.  `span_us` is first
start to last end of a call on the device (device time plus the gaps between launches).  Times are the medians over the
calls; `launches` lists the activities of the median call in launch order."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

GAP_US = 1000.0
CATS = ("kernel", "gpu_memset", "gpu_memcpy")


def bench_features(ctx, dev, n=100000):
    import torch
    import bench
    from dsp_audioreclabs_b200 import device as devapi
    tr_s, tr_o = bench.synth_batch_device(n, dev, seed=990000, first_index=0)
    fe = devapi.DeviceFrontend(tr_o, bench.FL, bench.FS, "hamming", ctx=ctx, device=dev)
    fe.run(tr_s)
    x_tr, mean, std = devapi.zscore_device(fe.stats.double().contiguous(), ctx=ctx)
    y_tr = (torch.arange(n, device=dev) % 10).to(torch.int32)
    del tr_s, fe
    q_s, q_o = bench.synth_batch_device(n, dev, seed=1234, first_index=0)
    qfe = devapi.DeviceFrontend(q_o, bench.FL, bench.FS, "hamming", ctx=ctx, device=dev)
    qfe.run(q_s)
    qn = torch.empty(n, 15, dtype=torch.float64, device=dev)
    devapi.zscore_apply_f32(qfe.stats, mean, std, out=qn, ctx=ctx)
    torch.cuda.synchronize()
    return x_tr.contiguous(), y_tr, qn


def split_calls(events):
    calls, cur, last_end = [], [], 0.0
    for e in events:
        if cur and e["ts"] - last_end > GAP_US:
            calls.append(cur)
            cur = []
        last_end = max(last_end, e["ts"] + e["dur"]) if cur else e["ts"] + e["dur"]
        cur.append(e)
    if cur:
        calls.append(cur)
    return calls


def classify(call):
    filt = [i for i, e in enumerate(call) if "knn_tc16_filter_kernel" in e["name"]]
    main = filt[-1]
    seed = filt[0] if len(filt) > 1 else None
    return ["main" if i == main else "seed" if i == seed else "prep" if i < main else "tail" for i in range(len(call))]


def short(name):
    """Kernel name without return type, namespaces and parameter list; template arguments stay."""
    n = name.replace("(anonymous namespace)::", "").split("(")[0]
    n = n[5:] if n.startswith("void ") else n
    depth, cut = 0, 0
    for i, ch in enumerate(n):
        depth += (ch == "<") - (ch == ">")
        if ch == ":" and depth == 0:
            cut = i + 1
    return n[cut:].strip()


def median(v):
    v = sorted(v)
    return v[len(v) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=12)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile
    from dsp_audioreclabs_b200 import batch, device as devapi
    dev = torch.device("cuda", 0)
    ctx = batch.default_context(0)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    x_tr, y_tr, qn = bench_features(ctx, dev)
    knn = devapi.DeviceKNN(3, ctx=ctx, device=dev).fit(x_tr, y_tr)
    for _ in range(3):
        knn.predict(qn)
    torch.cuda.synchronize()
    # predict wall time without the profiler, CUDA events on the launching stream
    wall = []
    for _ in range(args.calls):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        knn.predict(qn)
        e1.record()
        torch.cuda.synchronize()
        wall.append(e0.elapsed_time(e1) * 1e3)
    with tempfile.TemporaryDirectory() as tmp:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.calls):
                knn.predict(qn)
                torch.cuda.synchronize()
                time.sleep(0.005)
        path = os.path.join(tmp, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            trace = json.load(f)
    events = sorted((e for e in trace["traceEvents"] if e.get("ph") == "X" and e.get("cat") in CATS), key=lambda e: e["ts"])
    calls = split_calls(events)
    if len(calls) != args.calls:
        raise SystemExit(f"trace split into {len(calls)} calls, expected {args.calls}")
    per_call = []
    for call in calls:
        g = classify(call)
        sums = {k: 0.0 for k in ("seed", "prep", "main", "tail")}
        for e, k in zip(call, g):
            sums[k] += e["dur"]
        per_call.append({"groups_us": sums, "busy_us": sum(sums.values()), "launches": len(call),
                         "span_us": call[-1]["ts"] + call[-1]["dur"] - call[0]["ts"]})
    order = sorted(range(len(calls)), key=lambda i: per_call[i]["span_us"])
    mid = order[len(order) // 2]
    res = {
        "gpu": gpu,
        "workload": "bench features 100k x 100k, D = 15, k = 3, DeviceKNN.predict, knn_prune automatic",
        "calls": args.calls,
        "predict_us_events_median": median(wall),
        "span_us_median": median([c["span_us"] for c in per_call]),
        "busy_us_median": median([c["busy_us"] for c in per_call]),
        "groups_us_median": {k: median([c["groups_us"][k] for c in per_call]) for k in ("seed", "prep", "main", "tail")},
        "launches_per_call": per_call[mid]["launches"],
        "launches": [{"name": short(e["name"]), "group": k, "us": e["dur"]} for e, k in zip(calls[mid], classify(calls[mid]))],
    }
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
