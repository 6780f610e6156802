"""Multi-GPU plumbing: one process per GPU, records sharded with no data-path collective, and a single
end-of-run reduction of the per-GPU result blocks over NCCL (torch.distributed is only the transport).

Merge rule = StreamCounter::join (src/kmerstream/StreamCounter.hpp:95-112): counters, F2 tables and
sumCount add; every 4-bit sketch counter becomes min(sum, 15).  The sketch travels as one uint8 per counter
so that the sum of up to 17 ranks cannot overflow before the clamp (done by bqc_sketch_import_u8).
"""
import numpy as np


def shard_regions(lengths, rank, world, gap=5000, margin=0):
    """Genome slice of `rank`: {contig: (begin, end)}.  Neighbouring shards are separated by `gap` bp with no
    fragment starts, so that the first qualifying read of a shard always re-anchors the coverage windows
    (beginPos - shift > 2*vsize, src/OverallNumbers.hpp:91) and per-shard coverage histograms add exactly."""
    assert gap > 2000 + 1000
    out = {}
    for c, n in enumerate(lengths):
        lo = n * rank // world
        hi = n * (rank + 1) // world
        if rank > 0:
            lo += gap
        if hi - lo > margin:
            out[c] = (lo, hi)
    return out


def reduce_tensors(counters, sketch_u8, group=None):
    """All-reduce (sum) the counter block (int64 view of the uint64 counters) and the uint8 sketch in place."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(counters, op=dist.ReduceOp.SUM, group=group)
        if sketch_u8.numel():
            dist.all_reduce(sketch_u8, op=dist.ReduceOp.SUM, group=group)
    return counters, sketch_u8


def reduce_engine(engine, bufs=None, group=None):
    """Export this GPU's tables, all-reduce them over NCCL, import the merged tables back (every rank ends
    with the whole-job result).  `bufs` lets the caller reuse the two device tensors across steps."""
    import torch
    import torch.distributed as dist
    dev = torch.device("cuda", engine.device)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        # the layout of the block depends on the longest read a rank has seen: same capacity everywhere first
        cap = torch.tensor([engine.lib.bqc_read_len_capacity(engine.handle)], dtype=torch.int64, device=dev)
        dist.all_reduce(cap, op=dist.ReduceOp.MAX, group=group)
        if int(cap.item()) != engine.lib.bqc_read_len_capacity(engine.handle):
            engine._check(engine.lib.bqc_reserve_read_len(engine.handle, int(cap.item())))
            bufs = None
    if bufs is None or bufs[0].numel() != engine.counters_len():
        bufs = (torch.empty(engine.counters_len(), dtype=torch.int64, device=dev),
                torch.empty(max(1, engine.sketch_len()), dtype=torch.uint8, device=dev))
    c, s = bufs
    engine.export_to(c.data_ptr(), s.data_ptr())
    reduce_tensors(c, s[: engine.sketch_len()], group)
    torch.cuda.synchronize(dev)
    engine.import_from(c.data_ptr(), s.data_ptr())
    return bufs


# ------------------------------------------------------------------------------------------------------
# One coordinate-ordered record stream cut at arbitrary records across engines (SURVEY 8e "the exception"): everything
# but the coverage windows adds up; the windows are resolved with the four-step protocol of include/bamqc_b200.h.
# `exchange(array) -> [array of piece 0, array of piece 1, ...]` is the only communication (an all-gather).
# ------------------------------------------------------------------------------------------------------
_SHARD_BYTES = None


def _shard_to_array(sh):
    import ctypes
    return np.frombuffer(ctypes.string_at(ctypes.addressof(sh), ctypes.sizeof(sh)), dtype=np.uint8).copy()


def _combine(lib, shard_arrays):
    import ctypes
    from . import _lib
    n = len(shard_arrays)
    arr = (_lib.bqc_cov_shard * n)()
    for k, a in enumerate(shard_arrays):
        ctypes.memmove(ctypes.addressof(arr[k]), np.ascontiguousarray(a, dtype=np.uint8).ctypes.data, ctypes.sizeof(_lib.bqc_cov_shard))
    delta = np.zeros(101, dtype=np.int64)
    lib.bqc_cov_shards_combine(ctypes.cast(arr, ctypes.c_void_p), n, delta.ctypes.data)
    return delta


def _resolve(engine, piece, exchange, lanes):
    """The protocol for the lanes of one piece at once: each exchange carries one row per lane, so there are three
    exchanges whatever the number of lanes.  `lanes`: the keyword arguments that select a lane in the engine's calls."""
    b = [engine.cov_shard_boundary(**kw) for kw in lanes]
    bounds = exchange(np.array([[x.n, x.first_rid, x.first_b, x.last_rid, x.last_b] for x in b], dtype=np.int64))
    prev = []
    for lane in range(len(lanes)):
        have_prev, prid, pb = 0, 0, 0
        for k in range(piece):
            if int(bounds[k][lane][0]) > 0:
                have_prev, prid, pb = 1, int(bounds[k][lane][3]), int(bounds[k][lane][4])
        prev.append((have_prev, prid, pb))
    tables = exchange(np.stack([engine.cov_shard_function(*prev[lane], **kw) for lane, kw in enumerate(lanes)]))
    shards = []
    for lane, kw in enumerate(lanes):
        p = 0
        for k in range(piece):
            if int(bounds[k][lane][0]) > 0:
                p = int(engine.lib.bqc_cov_apply(np.ascontiguousarray(tables[k][lane], dtype=np.uint16).ctypes.data, p))
        shards.append(_shard_to_array(engine.cov_shard_run(*prev[lane], p, **kw)))
    shards = exchange(np.stack(shards))
    return [_combine(engine.lib, [s[lane] for s in shards]) for lane in range(len(lanes))]


def resolve_coverage_shards(engine, piece, exchange):
    """Coverage statistic of piece number `piece` (stream order) of a record stream cut across engines in shard mode
    (Engine.cov_defer()); call it on every piece after Engine.finish().  Returns the correction to add to the SUM of
    the pieces' poscov tables (Engine.poscov_adjust on the merged result) -- identical on every piece."""
    return _resolve(engine, piece, exchange, [{}])[0]


def resolve_coverage_shards_lanes(engine, piece, exchange, n_lanes):
    """resolve_coverage_shards for an engine with `n_lanes` read groups: every lane's records are a stream of their own,
    cut where the file is cut.  Returns one correction per lane (Engine.poscov_adjust(delta[lane], lane)), with the
    same three exchanges as one lane."""
    return _resolve(engine, piece, exchange, [dict(lane=lane) for lane in range(n_lanes)])


def _resolve_local(engines, resolve):
    import threading
    n = len(engines)
    slots = {}
    barrier = threading.Barrier(n)
    out = [None] * n

    def run(k):
        step = [0]

        def exchange(a):
            key = step[0]
            step[0] += 1
            slots[(key, k)] = np.array(a, copy=True)
            barrier.wait()
            res = [slots[(key, j)] for j in range(n)]
            barrier.wait()
            return res
        out[k] = resolve(engines[k], k, exchange)
    ths = [threading.Thread(target=run, args=(k,)) for k in range(n)]
    [t.start() for t in ths]
    [t.join() for t in ths]
    return out[0]


def resolve_coverage_local(engines):
    """The same protocol for engines that live in one process (pieces in list order)."""
    return _resolve_local(engines, resolve_coverage_shards)


def resolve_coverage_local_lanes(engines, n_lanes):
    """resolve_coverage_shards_lanes for engines that live in one process: one correction per lane."""
    return _resolve_local(engines, lambda e, k, x: resolve_coverage_shards_lanes(e, k, x, n_lanes))


def torch_exchange(device=None, group=None):
    """exchange() over torch.distributed (NCCL: device tensors; gloo: CPU tensors)."""
    import torch
    import torch.distributed as dist

    def exchange(a):
        a = np.ascontiguousarray(a)
        t = torch.from_numpy(a.view(np.uint8).reshape(-1).copy())
        if device is not None:
            t = t.to(device)
        outs = [torch.empty_like(t) for _ in range(dist.get_world_size(group))]
        dist.all_gather(outs, t, group=group)
        return [o.cpu().numpy().view(a.dtype).reshape(a.shape) for o in outs]
    return exchange


def clamp_sketch_numpy(total_u8):
    """Host restatement of the import clamp (for CPU tests)."""
    return np.minimum(total_u8, 15).astype(np.uint8)
