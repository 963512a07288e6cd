"""Multi-GPU counting: one process per GPU, key-range ownership, one exchange step.

The reference has no multi-device path (SURVEY.md 2.2 row C*); this is the one place the
path shards (SURVEY.md 8(e)).  Each rank packs its own reads into super-window records and
counts them locally FIRST (a key crosses NVLink once per rank, with its count, instead of once
per occurrence).  The ranks then all-gather a 1024-bin histogram of their records' leading
bits, cut the key space into P contiguous ranges of about equal record totals, and every rank
pulls the records of its range out of all ranks' grouped arrays -- the pull is the load side of
the level-2 placement kernel (kc_xchg_pull), so the transfer over NVLink / NVSwitch happens
inside the kernel that consumes it.  Rank r ends with the sorted unique records of key range r;
the artefact is the concatenation in rank order.

torch.distributed is plumbing only: the tiny all-gather and two stream-ordered barriers.
The NCCL all-to-all-v of run slices below (exchange_and_combine) is kept for keys the
super-window path does not take (k > 64).
"""
import numpy as np

XCHG_BINS = 1024            # histogram bins = leading 10 key bits (kXB1 in kc_super.cu)


def plan_owner_ranges(all_hist, world):
    """Host model of the device plan (x_plan_kernel): all_hist[s][b] = records of rank s whose
    leading 10 key bits are b.  Bucket b belongs to the rank in whose equal share of the total
    the middle of the bucket falls; returns lo[0..world]: rank o owns buckets [lo[o], lo[o+1])."""
    h = np.asarray(all_hist, dtype=np.uint64).reshape(world, XCHG_BINS)
    tot = h.sum(axis=0)
    total = int(tot.sum())
    lo = [XCHG_BINS] * (world + 1)
    cum = 0
    for b in range(XCHG_BINS):
        t = int(tot[b])
        owner = min(world - 1, (cum + t // 2) * world // total) if total else 0
        lo[owner] = min(lo[owner], b)
        cum += t
    for o in range(world - 1, -1, -1):
        lo[o] = min(lo[o], lo[o + 1])
    lo[0] = 0
    return lo


class Exchange:
    """kc_xchg_* driven by torch.distributed (one process per GPU).

    The counter's stream must be torch's current stream: the all-gather and the barriers are
    ordered against the kernels by stream order alone, the host never waits inside a step."""

    def __init__(self, counter, device, expected_reads, group=None):
        import torch
        import torch.distributed as dist
        self.c, self.dev, self.group = counter, device, group
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        counter.xchg_begin(self.rank, self.world, expected_reads)
        everyone = [None] * self.world
        dist.all_gather_object(everyone, (counter.xchg_export(), counter.canonical), group=group)
        if any(c != counter.canonical for _, c in everyone):
            raise ValueError("multigpu.Exchange: every rank's Counter must have the same canonical setting")
        for r, (h, _) in enumerate(everyone):
            if r != self.rank:
                counter.xchg_import(r, h)           # the peer's workspace, mapped into this process (CUDA IPC)
        hp, ap = counter.xchg_hist()
        self.hist = torch.as_tensor(_CudaView(hp, (XCHG_BINS,), "<i4"), device=device)
        self.all_hist = torch.as_tensor(_CudaView(ap, (self.world * XCHG_BINS,), "<i4"), device=device)
        self.flag = torch.zeros(1, dtype=torch.int32, device=device)
        dist.barrier(group=group)

    def barrier(self):
        """Stream-ordered: a one-element all-reduce queued behind this rank's kernels."""
        import torch.distributed as dist
        dist.all_reduce(self.flag, group=self.group)

    def add_device(self, d_ptr, n_bytes):
        self.c.accum_add_device(d_ptr, n_bytes)

    def finish(self):
        """Everything accumulated on all ranks -> this rank's key range as a Run. Collective."""
        import torch.distributed as dist
        c = self.c
        self.barrier()                              # every rank's bins are complete
        c.xchg_count_local()                        # (reads the peers' bins over NVLink)
        dist.all_gather_into_tensor(self.all_hist, self.hist, group=self.group)
        c.xchg_group_local()
        self.barrier()                              # every rank's grouped records and counters are final
        c.xchg_pull()
        self.barrier()                              # nobody reads a peer's grouped records any more
        return c.xchg_finish()


def count_shard(counter, d_reads_ptr, n_bytes, device, group=None, exchange=None):
    """This rank's share of the distributed count: returns the Run of this rank's key range.
    Collective. With an Exchange (k <= 64) the records are pulled over NVLink inside the placement
    kernel; without one, run slices travel by an NCCL all-to-all-v and are merged (merge path)."""
    import torch.distributed as dist
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    if exchange is not None and world > 1:
        exchange.add_device(d_reads_ptr, n_bytes)
        return exchange.finish()
    local = counter.count_device(d_reads_ptr, n_bytes)
    if world == 1:
        return local
    return exchange_and_combine(counter, local, device, group)


def histogram(run, n_bins=10001, group=None):
    """Count spectrum of the whole distributed artefact: every rank's Run.histogram summed by one
    all-reduce; every rank gets the same uint64[n_bins]. Collective.

    After the exchange (Exchange.finish, or exchange_and_combine for k > 64) rank r holds key range r
    with its final counts, so this sum is the spectrum of the concatenated artefact. For the same
    reason Run.filter may be applied rank by rank: the concatenation of the filtered runs in rank
    order is the filtered artefact."""
    import torch
    import torch.distributed as dist
    h = run.histogram(n_bins)
    t = torch.from_numpy(h.view(np.int64).copy())             # sums stay far below 2^63
    if dist.get_backend(group) == "nccl":                     # NCCL reduces device tensors: the run's device
        t = t.to(torch.device("cuda", run._c.device))
    dist.all_reduce(t, group=group)
    return t.cpu().numpy().view(np.uint64)


# ------------------------------------------------------------------ ownership
def range_splitters(world, words):
    """P-1 ascending splitter keys cutting the key space into P equal-width ranges
    of the most significant word.  Shape [P-1, words] uint64."""
    sp = np.zeros((max(world - 1, 0), words), dtype=np.uint64)
    for i in range(1, world):
        sp[i - 1, 0] = np.uint64((i << 64) // world)
    return sp


def owner_of(keys_hi, world):
    """Owner rank of keys given their most significant word (host-side model, used by tests)."""
    sp = range_splitters(world, 1)[:, 0]
    return np.searchsorted(sp, np.asarray(keys_hi, dtype=np.uint64), side="right")


def slice_offsets_host(keys, splitters):
    """Host model of Run.split / kc_run_split: lower-bound offsets of the splitters in a
    sorted [n, W] uint64 key array -> P+1 offsets.  (CPU tests; the product path calls
    the device kernel through kc_run_split.)"""
    n, W = keys.shape
    off = [0]
    for s in splitters:
        lo, hi = 0, n
        while lo < hi:
            mid = (lo + hi) // 2
            if tuple(keys[mid]) < tuple(s):
                lo = mid + 1
            else:
                hi = mid
        off.append(lo)
    off.append(n)
    return np.asarray(off, dtype=np.int64)


# ------------------------------------------------------------------- exchange
def exchange_slices(keys_t, counts_t, offsets, group=None):
    """All-to-all-v of run slices.  keys_t [n, W] int64 and counts_t [n] int32 are this
    rank's run (any device); slice p = rows offsets[p]:offsets[p+1] goes to rank p.
    Returns (recv_keys, recv_counts, recv_sizes): the slices received, concatenated in
    source-rank order, and their lengths."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group)
    send = [int(offsets[p + 1] - offsets[p]) for p in range(world)]
    dev = keys_t.device
    send_t = torch.tensor(send, dtype=torch.int64, device=dev)
    recv_t = torch.empty_like(send_t)
    backend = dist.get_backend(group)
    if backend == "nccl":
        dist.all_to_all_single(recv_t, send_t, group=group)
    else:
        _p2p_all_to_all(recv_t, send_t, [1] * world, [1] * world, group)
    recv = [int(x) for x in recv_t.tolist()]
    W = keys_t.shape[1]
    rk = torch.empty((sum(recv), W), dtype=keys_t.dtype, device=dev)
    rc = torch.empty((sum(recv),), dtype=counts_t.dtype, device=dev)
    if backend == "nccl":
        dist.all_to_all_single(rk, keys_t, output_split_sizes=recv, input_split_sizes=send, group=group)
        dist.all_to_all_single(rc, counts_t, output_split_sizes=recv, input_split_sizes=send, group=group)
    else:
        _p2p_all_to_all(rk, keys_t, recv, send, group)
        _p2p_all_to_all(rc, counts_t, recv, send, group)
    return rk, rc, recv


def _p2p_all_to_all(out, inp, recv_sizes, send_sizes, group):
    """all_to_all_single for backends without it (gloo on CPU): batched isend/irecv."""
    import torch.distributed as dist
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    so = np.concatenate([[0], np.cumsum(send_sizes)])
    ro = np.concatenate([[0], np.cumsum(recv_sizes)])
    out[ro[rank]:ro[rank + 1]] = inp[so[rank]:so[rank + 1]]
    ops = []
    for p in range(world):
        if p == rank:
            continue
        if send_sizes[p]:
            ops.append(dist.P2POp(dist.isend, inp[so[p]:so[p + 1]].contiguous(), dist.get_global_rank(group, p) if group else p, group))
        if recv_sizes[p]:
            ops.append(dist.P2POp(dist.irecv, out[ro[p]:ro[p + 1]], dist.get_global_rank(group, p) if group else p, group))
    if ops:
        for w in dist.batch_isend_irecv(ops):
            w.wait()


# ---------------------------------------------------------------- device glue
class _CudaView:
    """Expose a raw device pointer to torch through __cuda_array_interface__."""

    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"data": (ptr, False), "shape": shape, "typestr": typestr, "version": 2}


def run_as_tensors(run, device):
    """Zero-copy torch views of a device-resident run: keys [n, W] int64, counts [n] int32."""
    import torch
    kptr, cptr, n = run.device_arrays()
    W = run._c.words
    if n == 0:
        return (torch.empty((0, W), dtype=torch.int64, device=device),
                torch.empty((0,), dtype=torch.int32, device=device))
    keys = torch.as_tensor(_CudaView(kptr, (n, W), "<i8"), device=device)
    counts = torch.as_tensor(_CudaView(cptr, (n,), "<i4"), device=device)
    return keys, counts


def exchange_and_combine(counter, local, device, group=None, splitters=None):
    """Second half of count_shard: `local` is this rank's run; returns the run of this rank's
    key range. Frees `local`."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group)
    keys_t, counts_t = run_as_tensors(local, device)
    if splitters is None:
        splitters = range_splitters(world, counter.words)
    off = local.split(splitters)
    # the run was produced on the counter's stream and is complete (count_device synchronises)
    rk, rc, sizes = exchange_slices(keys_t, counts_t, off, group)
    torch.cuda.current_stream().synchronize()
    local.free()
    parts, pos = [], 0
    for sz in sizes:
        parts.append(counter.run_from_device(rk.data_ptr() + pos * counter.words * 8, rc.data_ptr() + pos * 4, sz))
        pos += sz
    merged = counter.merge(parts)
    for p in parts:
        p.free()
    return merged
