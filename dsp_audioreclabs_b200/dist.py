"""One process per GPU: how the path shards across the GPUs of a box (SURVEY.md section 8(e)).

* Front end: independent utterances -> contiguous utterance ranges per rank, balanced by
  sample count, NO collective on the data path (`utterance_shards`).
* KNN: the train set is sharded by row.  Every rank scores the (all-gathered) queries against
  its own rows, keeps its local top-k (distance, global row, label), and ONE all-gather of
  those candidate lists -- packed into a single buffer -- over NCCL/NVLink lets each rank merge
  and vote for its own queries (`ShardedKNN.predict_sharded`).  When the train matrix is small
  (D = 15: 12 MB) the cheaper equivalent is to all-gather the train rows once per fit and
  classify locally (`ShardedKNN.predict_replicated`); `ShardedKNN.predict` picks by size.

* DTW template matching (the self-specified MFCC + DTW variant): templates sharded by row, queries replicated,
  the same single all-gather of top-k candidates (`ShardedDTW` on lists of NumPy arrays through the host call,
  `ShardedDeviceDTW` on device tensors through the fused top-k).

torch.distributed is plumbing only; the compute callbacks default to the CUDA library and can
be replaced (the CPU gloo tests plug in the oracle, since there is no CPU implementation here).
"""
import numpy as np
import torch
import torch.distributed as dist


def bind_to_gpu_numa(device_index):
    """Pin this process (its threads and, by first touch, the pinned staging buffers it allocates afterwards) to the
    CPUs of the NUMA node the GPU hangs off: with one process per GPU, eight ranks left on node 0 push all their
    host->device traffic through one socket's memory controllers (round 1: 0.44 end-to-end efficiency at 8 GPUs).
    Reads the PCI bus id from the CUDA runtime and the node / cpu list from sysfs.  Returns a dict describing what was
    done (for the bench line); never raises -- a box without the sysfs entries is left as it is."""
    import os
    info = {"gpu": int(device_index), "numa_node": None, "cpus": None, "bound": False}
    try:
        bus = torch.cuda.get_device_properties(device_index).pci_bus_id
        dom = torch.cuda.get_device_properties(device_index).pci_domain_id
        dev = torch.cuda.get_device_properties(device_index).pci_device_id
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev:02x}.0/numa_node"
        node = int(open(path).read().strip())
        info["numa_node"] = node
        if node < 0:
            return info
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = cpus & set(os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
            info["cpus"] = len(allowed)
            info["bound"] = True
    except Exception as exc:          # noqa: BLE001 -- best effort by design
        info["error"] = repr(exc)
    return info


def balanced_bounds(n, world):
    """Contiguous ranges [b[r], b[r+1]) of n items, sizes differing by at most one."""
    base, rem = divmod(int(n), int(world))
    sizes = [base + (1 if r < rem else 0) for r in range(world)]
    return np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)


def utterance_shards(offsets, world):
    """Contiguous utterance ranges per rank balanced by total samples (ragged batches):
    boundaries at the utterances closest to k/world of the cumulative sample count."""
    offsets = np.asarray(offsets, dtype=np.int64)
    b = len(offsets) - 1
    total = offsets[-1] - offsets[0]
    targets = offsets[0] + (np.arange(1, world) * total) // world
    cuts = np.searchsorted(offsets, targets, side="left")
    bounds = np.concatenate([[0], np.clip(cuts, 0, b), [b]]).astype(np.int64)
    return np.maximum.accumulate(bounds)


def _all_gather_rows(x, group=None):
    """all-gather of [n_r, ...] tensors with different n_r: returns the list of per-rank tensors.  One tiny
    all-gather of the row counts, one all_gather_into_tensor of the rows padded to the largest shard."""
    world = dist.get_world_size(group)
    n = torch.tensor([x.shape[0]], dtype=torch.int64, device=x.device)
    sizes = torch.empty(world, dtype=torch.int64, device=x.device)
    dist.all_gather_into_tensor(sizes, n, group=group)
    sizes = [int(v) for v in sizes.tolist()]
    mx = max(sizes)
    pad = torch.zeros((mx,) + tuple(x.shape[1:]), dtype=x.dtype, device=x.device)
    pad[: x.shape[0]] = x
    out = torch.empty((world * mx,) + tuple(x.shape[1:]), dtype=x.dtype, device=x.device)
    dist.all_gather_into_tensor(out, pad, group=group)
    return [out[r * mx: r * mx + s] for r, s in enumerate(sizes)]


def pack_candidates(d2, idx, lab):
    """(sqdist f64 [m,k], global row i64 [m,k], label i32 [m,k]) -> ONE int64 buffer [m, k, 3] (the float64 bit
    patterns travel as int64), so that the candidate exchange is a single collective."""
    return torch.stack([d2.contiguous().view(torch.int64), idx.to(torch.int64), lab.to(torch.int64)], dim=2).contiguous()


def unpack_candidates(packed):
    """[..., k, 3] int64 -> (sqdist f64, idx i64, label i32) as contiguous tensors."""
    return (packed[..., 0].contiguous().view(torch.float64), packed[..., 1].contiguous(),
            packed[..., 2].to(torch.int32).contiguous())


def all_gather_candidates(d2, idx, lab, group=None):
    """The single candidate exchange of the row-sharded design: every rank contributes its local top-k of the SAME
    m queries; returns [R, m, k] x 3."""
    world = dist.get_world_size(group)
    mine = pack_candidates(d2, idx, lab)
    out = torch.empty((world,) + tuple(mine.shape), dtype=torch.int64, device=mine.device)
    dist.all_gather_into_tensor(out.view(-1), mine.view(-1), group=group)
    return unpack_candidates(out)


class ShardedKNN:
    """Row-sharded KNN classify across the ranks of a process group.

    local_topk(train, labels, queries, k, index_base) -> (sqdist[m,k] f64, idx[m,k] i64, label[m,k] i32)
    merge_vote(cand_sqdist[R,m,k], cand_idx[R,m,k], cand_label[R,m,k]) -> labels[m] i32
    Both default to the CUDA library (device tensors).  Labels are class indices >= 0 (the kernels use negative
    labels for empty candidate slots); encode other label sets to 0..C-1 first, as batch.KNN does.

    replicate_below: `predict` classifies against an all-gathered copy of the train set, with NO per-call
    candidate exchange, when the whole train set is at most this many bytes (the 15-dim statistical features:
    100,000 rows are 12 MB); larger train sets (sequence features, DTW templates) take the row-sharded exchange.
    Pass 0 to force the exchange."""

    def __init__(self, n_neighbors=3, group=None, local_topk=None, merge_vote=None, replicate_below=64 << 20, hints=True):
        import inspect
        self.k = int(n_neighbors)
        self.group = group
        self._topk = local_topk or self._cuda_topk
        # local_topk may accept bound=<float64 [m] upper bounds on the k-th squared distance> (see predict_sharded)
        self._takes_bound = "bound" in inspect.signature(self._topk).parameters
        self.hints = bool(hints)
        self._merge = merge_vote or self._cuda_merge
        self.replicate_below = int(replicate_below)
        self._knn = {}
        self._full = None

    # -- CUDA callbacks ---------------------------------------------------------------------
    def _cuda_topk(self, train, labels, queries, k, index_base, bound=None):
        from .device import DeviceKNN
        key = (train.data_ptr(), train.shape[0], index_base)
        knn = self._knn.get(key)
        if knn is None:
            knn = self._knn[key] = DeviceKNN(k, device=train.device, index_base=index_base).fit(train, labels)
        return knn.topk(queries, bound)

    def _cuda_merge(self, cd, ci, cl):
        from .device import DeviceKNN
        helper = next(iter(self._knn.values()), None) or DeviceKNN(self.k, device=cd.device)
        return helper.merge_vote(cd, ci, cl)[0]

    # -- API -------------------------------------------------------------------------------
    def fit(self, train_shard, labels_shard):
        """Keep this rank's rows; the global row index of its first row and the size of the whole train set come
        from one all-gather of the shard sizes.  A second fit() starts from scratch."""
        world, rank = dist.get_world_size(self.group), dist.get_rank(self.group)
        if labels_shard.numel() and int(labels_shard.min()) < 0:
            raise ValueError("labels must be class indices >= 0 (encode them with np.unique(..., return_inverse=True))")
        for knn in self._knn.values():
            knn.free()
        self._knn, self._full = {}, None
        n = torch.tensor([train_shard.shape[0]], dtype=torch.int64, device=train_shard.device)
        sizes = torch.empty(world, dtype=torch.int64, device=train_shard.device)
        dist.all_gather_into_tensor(sizes, n, group=self.group)
        sizes = [int(v) for v in sizes.tolist()]
        self.index_base = int(sum(sizes[:rank]))
        self.n_total = int(sum(sizes))
        self._min_shard = int(min(sizes))
        self.train, self.labels = train_shard.contiguous(), labels_shard.contiguous()
        return self

    def train_bytes(self):
        return self.n_total * int(self.train.shape[1]) * self.train.element_size()

    def predict(self, queries_local, counts=None):
        """Labels for this rank's queries: the replicated-train path when the train set is small, else the
        row-sharded exchange (every rank must take the same branch: the choice depends on global sizes only).
        counts: the per-rank query counts when the caller knows them (see predict_sharded)."""
        if self.train_bytes() <= self.replicate_below:
            return self.predict_replicated(queries_local)
        return self.predict_sharded(queries_local, counts)

    def predict_sharded(self, queries_local, counts=None):
        """The north-star exchange: all-gather the query features, score ALL queries against the local rows, ONE
        all-gather of the packed per-shard top-k candidates (16 bytes per candidate: the float64 distance, and the
        global row with the label in one int64), merge + vote for the rank's own queries (only their slice of the
        gathered buffer is unpacked)."""
        rank = dist.get_rank(self.group)
        world = dist.get_world_size(self.group)
        q_local = queries_local.contiguous()
        # Threshold hints: a rank first classifies its OWN queries against its own rows; the k-th distance it finds is an
        # upper bound on the query's k-th distance in the whole train set, and travels with the query.  The other shards
        # then only have to return their rows inside that radius: their candidate filters start at the threshold instead
        # of paying ~k ln(n / k) insertions per query and shard to discover one (eight shards of 12,500 rows cost 6 x the
        # insertion work of one pass over 100,000 rows without it).
        hinted = self._takes_bound and self.hints and self._min_shard >= self.k      # the same on every rank
        if hinted:
            own_d2 = self._topk(self.train, self.labels, q_local, self.k, self.index_base)[0]
            payload = torch.cat([q_local, own_d2[:, self.k - 1:self.k].to(q_local.dtype)], dim=1).contiguous()
        else:
            payload = q_local
        if counts is not None and len(set(int(c) for c in counts)) == 1 and int(counts[rank]) == payload.shape[0]:
            # equal, known query counts (a batch sharded evenly): no size exchange, no padding and -- what matters --
            # no host synchronisation on the step: the whole classify step stays enqueued behind the front end
            p_all = torch.empty((world * payload.shape[0],) + tuple(payload.shape[1:]), dtype=payload.dtype, device=payload.device)
            dist.all_gather_into_tensor(p_all, payload, group=self.group)
            per_rank_n = [payload.shape[0]] * world
        else:
            parts = _all_gather_rows(payload, self.group)
            per_rank_n = [t.shape[0] for t in parts]
            p_all = torch.cat(parts, dim=0)
        if hinted:
            q_all = p_all[:, :-1].contiguous()
            d2, idx, lab = self._topk(self.train, self.labels, q_all, self.k, self.index_base, bound=p_all[:, -1].contiguous())
        else:
            q_all = p_all
            d2, idx, lab = self._topk(self.train, self.labels, q_all, self.k, self.index_base)
        if self.n_total >= (1 << 31):
            raise ValueError("row-sharded KNN packs the global row index into 32 bits: at most 2^31 train rows")
        mine = torch.stack([d2.contiguous().view(torch.int64),
                            (idx.to(torch.int64) << 32) | (lab.to(torch.int64) & 0xFFFFFFFF)], dim=2).contiguous()
        out = torch.empty((world,) + tuple(mine.shape), dtype=torch.int64, device=mine.device)
        dist.all_gather_into_tensor(out.view(-1), mine.view(-1), group=self.group)      # the single candidate exchange
        lo = sum(per_rank_n[:rank])
        own = out[:, lo:lo + queries_local.shape[0]]
        cd = own[..., 0].contiguous().view(torch.float64)
        ci = (own[..., 1] >> 32).contiguous()
        cl = ((own[..., 1] << 32) >> 32).to(torch.int32).contiguous()       # sign-extended low word (-1 = empty slot)
        return self._merge(cd, ci, cl)

    def predict_replicated(self, queries_local):
        """All-gather the (small) train shards once per fit, classify own queries with no candidate exchange.
        Same result as `predict_sharded`."""
        if self._full is None:
            tr = torch.cat(_all_gather_rows(self.train, self.group), dim=0)
            lb = torch.cat(_all_gather_rows(self.labels, self.group), dim=0)
            self._full = (tr.contiguous(), lb.contiguous())
        d2, idx, lab = self._topk(self._full[0], self._full[1], queries_local.contiguous(), self.k, 0)
        return self._merge(d2[None], idx[None], lab[None])


def merge_topk(cost, idx, lab, k):
    """k-way selection over R candidate lists [R, m, k] (cost f64, global index i64, label i32), by (cost, global
    index), empty slots (index < 0) last: a stable sort by index followed by a stable sort by cost, with torch sorts on
    the tensors' device (no host synchronisation).  Returns (cost, index, label) [m, k]."""
    m = cost.shape[1]
    cost = cost.permute(1, 0, 2).reshape(m, -1)
    idx = idx.permute(1, 0, 2).reshape(m, -1)
    lab = lab.permute(1, 0, 2).reshape(m, -1)
    key = torch.where(idx < 0, torch.full_like(idx, torch.iinfo(torch.int64).max), idx)
    o1 = torch.argsort(key, dim=1, stable=True)
    o2 = torch.argsort(cost.gather(1, o1), dim=1, stable=True)
    order = o1.gather(1, o2)[:, :k]
    return tuple(a.gather(1, order) for a in (cost, idx, lab))


class ShardedDTW:
    """Row-sharded DTW template matching (BASELINE config 5: templates sharded by row, queries replicated, ONE
    all-gather of the packed per-shard top-k candidates).  Sequences are lists of [frames, dim] float32 arrays.

    local_topk(templates, labels, queries, k, index_base) -> (cost[m,k] f64, idx[m,k] i64, label[m,k] i32), sorted by
    (cost, index); defaults to the CUDA library (mfcc_dtw.DTWClassifier).  The merge is a k-way selection by
    (cost, global index) with torch sorts on the device the group communicates on (CUDA under NCCL: pass `device`)."""

    def __init__(self, n_neighbors=1, group=None, local_topk=None, device=None):
        self.k = int(n_neighbors)
        self.group = group
        self._topk = local_topk or self._cuda_topk
        self._clf = None
        self.device = device          # torch.device for the exchange buffers; None = CPU (gloo)

    def _cuda_topk(self, templates, labels, queries, k, index_base):
        from .mfcc_dtw import DTWClassifier
        if self._clf is None:
            # this rank's GPU: the library context of the device the exchange buffers live on (without it every rank of a
            # box computed on GPU 0)
            ctx = None
            if self.device is not None and torch.device(self.device).type == "cuda":
                from .batch import default_context
                ctx = default_context(torch.device(self.device).index or 0)
            self._clf = DTWClassifier(k, ctx=ctx, index_base=index_base).fit(templates, labels)
        nc, ni, nl = self._clf.kneighbors(queries)
        return nc, ni, self._clf.classes_[np.clip(nl, 0, None)].astype(np.int32) * (nl >= 0) - (nl < 0)

    def fit(self, template_shard, labels_shard):
        world, rank = dist.get_world_size(self.group), dist.get_rank(self.group)
        self._clf = None                      # a second fit() must not answer from the old shard
        n = torch.tensor([len(template_shard)], dtype=torch.int64, device=self.device)
        sizes = torch.empty(world, dtype=torch.int64, device=self.device)
        dist.all_gather_into_tensor(sizes, n, group=self.group)
        self.index_base = int(sum(int(v) for v in sizes.tolist()[:rank]))
        self.templates, self.labels = list(template_shard), np.asarray(labels_shard)
        return self

    def kneighbors(self, queries):
        """(cost[m,k], global template index[m,k], label[m,k]) for the (replicated) queries."""
        c, i, l = self._topk(self.templates, self.labels, queries, self.k, self.index_base)
        c, i, l = (torch.from_numpy(np.ascontiguousarray(a)) for a in (c.astype(np.float64), i.astype(np.int64), l.astype(np.int32)))
        if self.device is not None:
            c, i, l = c.to(self.device), i.to(self.device), l.to(self.device)
        cc, ci, cl = all_gather_candidates(c, i, l, self.group)            # the single candidate exchange
        return tuple(a.cpu().numpy() for a in merge_topk(cc, ci, cl, self.k))

    def predict(self, queries):
        _, _, lab = self.kneighbors(queries)
        out = np.empty(len(lab), dtype=np.int64)
        for q, row in enumerate(lab):
            vals, cnt = np.unique(row[row >= 0], return_counts=True)
            out[q] = vals[np.argmax(cnt)] if len(vals) else -1      # argmax: first maximum = smallest label
        return out


class ShardedDeviceDTW:
    """Row-sharded DTW template matching on device tensors (BASELINE config 5's exchange: templates sharded by row,
    queries replicated, ONE all-gather of the packed per-shard top-k candidates).  Sequences are packed as
    device.DeviceDTW takes them: float32 [frames, dim] feats, int64 offsets [n + 1] in frames, optional int32 lengths.

    The queries must be the same on every rank (same sequences, same order): the ranks exchange candidates for query
    positions, and nothing checks that the positions mean the same sequence everywhere.  Once the shapes are warm a
    call enqueues its work with no host synchronisation.

    local_topk(t_feats, t_offsets, t_labels, q_feats, q_offsets, k, index_base, bound=None, t_lengths=None,
    q_lengths=None, max_q_frames=None) -> (cost f64, global index i64, label i32) [nq, k], sorted by (cost, index),
    (inf, -1, -1) in empty slots, only templates with cost <= bound[q] when a bound is given; defaults to the fused
    top-k of device.DeviceDTW.  merge_vote(cost [R, nq, k], idx, label) -> int32 [nq] labels; defaults to
    dsp_knn_merge_vote_device.  Labels are class indices >= 0 (-1 marks an empty slot)."""

    def __init__(self, n_neighbors=1, group=None, local_topk=None, merge_vote=None):
        self.k = int(n_neighbors)
        self.group = group
        self._topk = local_topk or self._cuda_topk
        self._merge = merge_vote or self._cuda_merge
        self._dtw = None
        self._merger = None

    # -- CUDA callbacks ---------------------------------------------------------------------
    def _cuda_topk(self, t_feats, t_offsets, t_labels, q_feats, q_offsets, k, index_base, bound=None, t_lengths=None,
                   q_lengths=None, max_q_frames=None):
        from .device import DeviceDTW
        if self._dtw is None:
            self._dtw = DeviceDTW(k, device=q_feats.device, index_base=index_base)
            if t_offsets.numel() > 1:
                self._dtw.fit(t_feats, t_offsets, t_labels, t_lengths)
        if self._dtw.handle is None:            # a shard without templates: every slot empty
            nq = q_offsets.numel() - 1
            return (torch.full((nq, k), float("inf"), dtype=torch.float64, device=q_feats.device),
                    torch.full((nq, k), -1, dtype=torch.int64, device=q_feats.device),
                    torch.full((nq, k), -1, dtype=torch.int32, device=q_feats.device))
        return self._dtw.topk(q_feats, q_offsets, q_lengths, max_q_frames, bound)

    def _cuda_merge(self, cost, idx, lab):
        from .device import DeviceKNN
        if self._merger is None:
            self._merger = DeviceKNN(self.k, device=cost.device)
        return self._merger.merge_vote(cost, idx, lab)[0]

    # -- API -------------------------------------------------------------------------------
    def fit(self, feats, offsets, labels, lengths=None):
        """Keep this rank's template shard; the global index of its first template and the size of the whole template
        set come from one all-gather of the shard sizes.  A second fit() starts from scratch."""
        world, rank = dist.get_world_size(self.group), dist.get_rank(self.group)
        if labels.numel() and int(labels.min()) < 0:
            raise ValueError("labels must be class indices >= 0 (encode them with np.unique(..., return_inverse=True))")
        if self._dtw is not None:
            self._dtw.free()
        self._dtw = None
        n = torch.tensor([offsets.numel() - 1], dtype=torch.int64, device=offsets.device)
        sizes = torch.empty(world, dtype=torch.int64, device=offsets.device)
        dist.all_gather_into_tensor(sizes, n, group=self.group)
        sizes = [int(v) for v in sizes.tolist()]
        self.index_base = int(sum(sizes[:rank]))
        self.n_total = int(sum(sizes))
        self.feats, self.offsets, self.labels, self.lengths = feats, offsets, labels, lengths
        return self

    def _gathered(self, q_feats, q_offsets, q_lengths, bound, max_q_frames):
        c, i, l = self._topk(self.feats, self.offsets, self.labels, q_feats, q_offsets, self.k, self.index_base,
                             bound=bound, t_lengths=self.lengths, q_lengths=q_lengths, max_q_frames=max_q_frames)
        return all_gather_candidates(c, i, l, self.group)                 # the single candidate exchange

    def kneighbors(self, q_feats, q_offsets, q_lengths=None, bound=None, max_q_frames=None):
        """(cost f64, global template index i64, label i32) [nq, k] on the device for the (replicated) queries, ties to
        the lower index, (inf, -1, -1) in empty slots.  bound (optional float64 [nq]): only templates with cost <=
        bound[q] (device.DeviceDTW.topk); every shard abandons the pairs above it from its first template on.
        max_q_frames (optional) only picks the kernel build."""
        return merge_topk(*self._gathered(q_feats, q_offsets, q_lengths, bound, max_q_frames), self.k)

    def predict(self, q_feats, q_offsets, q_lengths=None, bound=None, max_q_frames=None):
        """Majority label of the k cheapest templates over all shards, ties to the smallest label, -1 where no template
        lies within the bound: int32 [nq] on the device."""
        return self._merge(*self._gathered(q_feats, q_offsets, q_lengths, bound, max_q_frames))


def zscore_stats_allreduce(x_local, group=None):
    """Train-set mean / population std over the rows of ALL ranks: one tiny all-reduce of
    (count, sum, sum of squares about the global mean) -- float64, two passes like np.std."""
    n = torch.tensor([x_local.shape[0]], dtype=torch.float64, device=x_local.device)
    s = x_local.sum(dim=0)
    buf = torch.cat([n, s])
    dist.all_reduce(buf, group=group)
    mean = buf[1:] / buf[0]
    ss = ((x_local - mean) ** 2).sum(dim=0)
    dist.all_reduce(ss, group=group)
    std = torch.sqrt(ss / buf[0])
    return mean, std
