"""KNN classify with and without tile pruning (tuning key knn_prune), on the bench's own features and on isotropic data.

  python tools/knn_prune_bench.py [--reps 5] [--out knn_prune.json]

Workload 1 ("bench"): the train and query features of bench.py (100k synthetic utterances each, frame 256 / shift 128,
hamming window, device front end, z-score with the train set's statistics), KNN(3).  Workload 2 ("isotropic"): the
bench's secondary statistical_d15 case, 1 M Gaussian queries x 100 k train rows around 10 centres.  predict() is timed
with CUDA events, knn_prune 0 and 1 alternated; the fraction of tile visits the lists keep comes from the DSP_KNN_DEBUG
report of one extra call."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def kept_fraction(knn, q):
    """One predict() with DSP_KNN_DEBUG=1; its report goes to the process's stderr (fd 2), read back via a temp file."""
    import tempfile
    import torch
    os.environ["DSP_KNN_DEBUG"] = "1"
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+") as f:
        os.dup2(f.fileno(), 2)
        try:
            knn.predict(q)
            torch.cuda.synchronize()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["DSP_KNN_DEBUG"]
        f.seek(0)
        text = f.read()
    for line in text.splitlines():
        if "prune: tile visits kept=" in line:
            kept, total = line.split("kept=")[1].split(" (")[0].split(" of ")
            return int(kept) / int(total), line.split("(")[-1].rstrip(")")
    return None, text.strip()


def time_modes(ctx, knn, q, reps):
    import torch
    out = {0: [], 1: []}
    labels = {}
    for mode in (0, 1):
        ctx.set_tuning("knn_prune", mode)
        labels[mode] = knn.predict(q).cpu()          # warm-up of this mode's shapes
    for _ in range(reps):
        for mode in (0, 1):
            ctx.set_tuning("knn_prune", mode)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            knn.predict(q)
            e1.record()
            torch.cuda.synchronize()
            out[mode].append(e0.elapsed_time(e1))
    ctx.set_tuning("knn_prune", 1)
    frac, how = kept_fraction(knn, q)
    return {"ms_prune_off": out[0], "ms_prune_auto": out[1],
            "median_off": sorted(out[0])[len(out[0]) // 2], "median_auto": sorted(out[1])[len(out[1]) // 2],
            "tile_visits_kept": frac, "main_pass": how,
            "labels_identical": bool(torch.equal(labels[0], labels[1]))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import bench
    from dsp_audioreclabs_b200 import batch, device as devapi
    dev = torch.device("cuda", 0)
    ctx = batch.default_context(0)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    res = {"gpu": gpu}

    n = 100000
    tr_s, tr_o = bench.synth_batch_device(n, dev, seed=990000, first_index=0)
    fe = devapi.DeviceFrontend(tr_o, bench.FL, bench.FS, "hamming", ctx=ctx, device=dev)
    fe.run(tr_s)
    x_tr_n, mean, std = devapi.zscore_device(fe.stats.double().contiguous(), ctx=ctx)
    y_tr = (torch.arange(n, device=dev) % 10).to(torch.int32)
    del tr_s, fe
    q_s, q_o = bench.synth_batch_device(n, dev, seed=1234, first_index=0)
    qfe = devapi.DeviceFrontend(q_o, bench.FL, bench.FS, "hamming", ctx=ctx, device=dev)
    qfe.run(q_s)
    qn = torch.empty(n, 15, dtype=torch.float64, device=dev)
    devapi.zscore_apply_f32(qfe.stats, mean, std, out=qn, ctx=ctx)
    torch.cuda.synchronize()
    knn = devapi.DeviceKNN(3, ctx=ctx, device=dev).fit(x_tr_n.contiguous(), y_tr)
    res["bench_100k_x_100k"] = time_modes(ctx, knn, qn, args.reps)
    del knn, q_s, qfe
    torch.cuda.empty_cache()

    m, n, d = 1000000, 100000, 15
    g = torch.Generator(device=dev).manual_seed(5)
    centers = torch.randn(10, d, device=dev, generator=g, dtype=torch.float64) * 1.5
    ytr = torch.randint(0, 10, (n,), device=dev, generator=g)
    xtr = centers[ytr] + torch.randn(n, d, device=dev, generator=g, dtype=torch.float64)
    yq = torch.randint(0, 10, (m,), device=dev, generator=g)
    xq = centers[yq] + torch.randn(m, d, device=dev, generator=g, dtype=torch.float64)
    knn = devapi.DeviceKNN(3, ctx=ctx, device=dev).fit(xtr.contiguous(), ytr.to(torch.int32))
    res["isotropic_1M_x_100k"] = time_modes(ctx, knn, xq, args.reps)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
