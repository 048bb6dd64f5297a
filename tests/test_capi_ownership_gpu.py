"""Ownership of the library's device memory: a context and its KNN / DTW handles give back everything they allocated
when they are freed, and the MFCC host call stays one launch."""
import gc

import numpy as np
import pytest
import torch

SCAN_TC16 = 3             # dsp_knn_last_stats: the tensor-core filter, whose fit builds the tile-pruning plan


def _free_bytes():
    torch.cuda.synchronize()
    gc.collect()
    torch.cuda.empty_cache()
    return torch.cuda.mem_get_info()[0]


def _inputs():
    """Host arrays and device tensors shared by every cycle, made once before any measurement."""
    from dsp_audioreclabs_b200 import batch, mfcc_dtw
    from oracle import synth
    lens = synth.ragged_lengths(12, 0.25, 1.0, seed=5)
    utts = [synth.utterance_pcm(i, int(n), seed0=77) for i, n in enumerate(lens)]
    s, o, l = batch.pack_aligned(utts)
    res = batch.frontend_batch(s, o, 1102, 441, "hamming", lengths=l, emit_frames=False)
    rng = np.random.default_rng(4)
    train = rng.standard_normal((300_000, 15))
    train_y = rng.integers(0, 5, 300_000)
    queries = rng.standard_normal((4096, 15))
    seqs = [rng.standard_normal((int(n), 13)).astype(np.float32) for n in rng.integers(5, 60, 64)]
    seq_y = np.arange(64) % 4
    tf, to = mfcc_dtw.pack_sequences(seqs, 13)
    dev = dict(samples=torch.from_numpy(s).cuda(), start=torch.from_numpy(res.start).cuda(),
               end=torch.from_numpy(res.end).cuda(), tf=torch.from_numpy(tf).cuda(), to=torch.from_numpy(to).cuda(),
               tl=torch.from_numpy(seq_y.astype(np.int32)).cuda())
    return dict(s=s, o=o, l=l, start=res.start, end=res.end, train=train, train_y=train_y, queries=queries,
                seqs=seqs, seq_y=seq_y), dev


def _cycle(h, dev):
    """One context through every owner it keeps: window tables, staging slots, the MFCC table cache, the one-shot
    scratch, a KNN handle on the tensor-core filter with tile pruning, a DTW handle.  Returns the free memory with
    the handles alive."""
    from dsp_audioreclabs_b200 import batch, device, mfcc_dtw
    c = batch.Context(0)
    for window in ("hamming", "hanning"):
        batch.frontend_batch(h["s"], h["o"], 1102, 441, window, lengths=h["l"], ctx=c)
    before = c.launch_count
    mfcc_dtw.mfcc_batch(h["s"], h["o"], h["start"], h["end"], lengths=h["l"], ctx=c)
    assert c.launch_count - before == 1
    dm = device.DeviceMFCC(h["o"], lengths=h["l"], ctx=c)
    dm.run(dev["samples"], dev["start"], dev["end"])
    knn = batch.KNN(3, ctx=c).fit(h["train"], h["train_y"])
    knn.kneighbors(h["queries"])
    assert knn.last_stats()[1] == SCAN_TC16
    before = c.launch_count
    mfcc_dtw.DTWClassifier(3, ctx=c).fit(h["seqs"], h["seq_y"]).kneighbors(h["seqs"])
    assert c.launch_count - before == 2
    dtw = device.DeviceDTW(3, ctx=c).fit(dev["tf"], dev["to"], dev["tl"])
    dtw.topk(dev["tf"], dev["to"])
    alive = _free_bytes()
    knn._free()
    dtw.free()
    c.close()
    return alive


@pytest.mark.gpu
def test_context_and_handles_give_back_their_device_memory():
    h, dev = _inputs()
    _cycle(h, dev)                                       # warm-up: modules, torch's cache, the library's first loads
    base = _free_bytes()
    for i in range(3):
        alive = _cycle(h, dev)
        assert base - alive >= 64 << 20, (i, base - alive)    # the measurement sees the library's allocations
    after = _free_bytes()
    assert abs(base - after) <= 16 << 20, base - after
