"""
Multi-GPU plumbing of the bulk path: one process per GPU (torch.distributed), reads sharded by
rank, the annotation index replicated, per-GPU counters merged with ONE all-reduce.

The bulk units are independent and the tally is a commutative integer sum (SURVEY.md 8e), so there
is no data-path collective besides the merge of `n_ensg + 8` int64 counters (about 0.3 MB, latency
bound).  On GPUs the all-reduce runs over NCCL directly on the library's device counter block
(`tec_bulk_counts_dev`) and on the library's stream: no host round trip, no extra copy.
"""
import numpy as np


def shard_units(n_units, rank, world, align=1):
    """[lo, hi) of this rank's contiguous slice of n_units units (any contiguous split is valid:
    the reference's result does not depend on read order in bulk mode)."""
    lo = (n_units * rank // world) // align * align
    hi = n_units if rank == world - 1 else (n_units * (rank + 1) // world) // align * align
    return lo, hi


class _DevArray:
    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 2}


def counts_tensor(engine, n_ensg, device):
    """torch view (no copy) of the engine's device counter block: int64[n_ensg + BULK_NSTATS], followed by the
    row counters in a run with loci (its length is the library's "bulk_counter_words")."""
    import torch
    return torch.as_tensor(_DevArray(engine.bulk_counts_dev(), engine.get_info("bulk_counter_words"), "<i8"), device=device)


def comm_init(engine, group=None):
    """Give the engine its own NCCL communicator over the ranks of `group` (the library then issues its
    collectives itself: tec_bulk_allreduce, tec_sc_exchange, tec_sc_allgather_triples).  The 128-byte id is
    the only thing that travels through torch.distributed.  Returns False where the backend is not NCCL
    (CPU-side tests over gloo keep the callback path)."""
    import torch.distributed as dist
    if dist.get_backend(group) != "nccl":
        return False
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    box = [engine.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(box, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
    engine.comm_init(box[0], rank, world)
    return True


def allreduce_counts_device(engine, n_ensg, device, group=None):
    """Sum the counter blocks of all ranks in place (NCCL), ordered on the engine's stream."""
    import torch
    import torch.distributed as dist
    if engine.comm_world()[1] > 1:                # the library's own communicator
        engine.bulk_allreduce()
        return counts_tensor(engine, n_ensg, device)
    t = counts_tensor(engine, n_ensg, device)
    with torch.cuda.stream(torch.cuda.ExternalStream(engine.stream, device=device)):
        dist.all_reduce(t, group=group)
    return t


def allreduce_counts_host(counts, stats, group=None):
    """Host-side merge of (counts, stats) as returned by Engine.bulk_finish: used where the ranks
    finished independently (e.g. one te_count process per BAM shard), any backend."""
    import torch
    import torch.distributed as dist
    t = torch.from_numpy(np.concatenate([np.asarray(counts, np.int64), np.asarray(stats, np.int64)]))
    dist.all_reduce(t, group=group)
    out = t.numpy()
    return out[:len(counts)].copy(), out[len(counts):].copy()


def bulk_name_exchange(engine, device, group=None):
    """Paired end by read name over byte ranges (include/tecount.h tec_bulk_name_partition_dev): after every rank's
    DeviceBam.count_range(4, ...), the rows go to the rank that owns their read name and each owner pairs what it
    receives.  Returns the number of records this rank received.  Collective."""
    import torch
    import torch.distributed as dist
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    if engine.comm_world()[1] == world and world > 1:        # comm_init was called: everything inside the library
        return engine.bulk_name_exchange()
    send, ptr = engine.bulk_name_partition_dev(world)
    src = _dev_tensor(ptr, sum(send) * 4, "<i8", device)         # 4 x int64 per record
    parts = [None] * world                                       # gloo (ranks that share a GPU): through the host
    dist.all_gather_object(parts, [x.cpu() for x in torch.split(src, [x * 4 for x in send])], group=group)
    dst = torch.cat([parts[r][rank] for r in range(world)]).to(device)
    torch.cuda.synchronize(device)
    n = int(dst.numel() // 4)
    engine.bulk_name_import_dev(n, dst.data_ptr() if n else None)
    return n


# ------------------------------------------------------------------------------------ single cell
# One process per GPU.  Each rank pushes its slice of the (coordinate-sorted) file; the survivors of
# Part 1's filter are then exchanged by cell id (all-to-all) with their position in the job-wide
# survivor order, and tec_sc_finalize runs per rank, calling back into `allreduce` at the points
# that are global (include/tecount.h).  Triples stay with the rank that owns the cell and are
# concatenated at the end ("allgather-merge"): cells are disjoint, so no counts are added.
_TORCH_DT = {0: ("<u4", "int32"), 1: ("<u8", "int64"), 2: ("<i8", "int64")}


def _dev_tensor(ptr, n, typestr, device):
    import torch
    if n == 0 or not ptr:
        return torch.empty(0, dtype={"<i4": torch.int32, "<i8": torch.int64}[typestr], device=device)
    return torch.as_tensor(_DevArray(ptr, n, typestr), device=device)


def make_allreduce(device, group=None):
    """The callback for Engine.sc_set_collective.  NCCL: reduces the device buffer in place; any
    other backend (gloo in the CPU-side tests): staged through host memory."""
    import torch
    import torch.distributed as dist
    ops = {0: dist.ReduceOp.SUM, 1: dist.ReduceOp.MIN, 2: dist.ReduceOp.MAX}
    on_gpu = dist.get_backend(group) == "nccl"

    def allreduce(ptr, count, dtype, op):
        if count == 0:
            return
        if dtype == 0:                                   # u32: widen (MIN / MAX must be unsigned)
            t32 = _dev_tensor(ptr, count, "<i4", device)
            t = t32.to(torch.int64) & 0xFFFFFFFF
        else:                                            # u64 / i64 values stay below 2^63
            t32 = None
            t = _dev_tensor(ptr, count, "<i8", device)
        if on_gpu:
            dist.all_reduce(t, op=ops[op], group=group)
            r = t
        else:
            h = t.cpu()
            dist.all_reduce(h, op=ops[op], group=group)
            r = h.to(device)
        if t32 is not None:
            t32.copy_((((r + 2 ** 31) % 2 ** 32) - 2 ** 31).to(torch.int32))       # back to the u32 bit pattern
        elif r is not t:
            t.copy_(r)
        torch.cuda.synchronize(device)

    return allreduce


TIMING = {}          # phase -> seconds of the last sc_exchange_by_cell (set TEC_DIST_TIMING=1)


def sc_exchange_by_cell(engine, device, group=None):
    """All-to-all of the survivors by owner rank (cell id % world) + job-wide positions; installs
    the received records in the engine.  Returns the number of records this rank now owns."""
    import os
    import time
    import torch
    import torch.distributed as dist
    timing = bool(os.environ.get("TEC_DIST_TIMING"))

    def mark(name, t0):
        if timing:
            torch.cuda.synchronize(device)
            TIMING[name] = TIMING.get(name, 0.0) + time.perf_counter() - t0
        return time.perf_counter()

    tm = time.perf_counter()
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    on_gpu = dist.get_backend(group) == "nccl"
    if engine.comm_world()[1] == world and world > 1:        # comm_init was called: everything inside the library
        n2 = engine.sc_exchange()
        mark("library_exchange", tm)
        return n2
    n = engine.sc_survivors()
    counts = [None] * world
    dist.all_gather_object(counts, int(n), group=group)
    base = sum(counts[:rank])
    tm = mark("counts", tm)
    # 32-byte records grouped by owner rank, file order kept inside a group (one kernel in the library)
    send, ptr = engine.sc_partition_dev(world, base)
    src = _dev_tensor(ptr, n * 4, "<i8", device)                 # 4 x int64 per record
    recv_all = [None] * world
    dist.all_gather_object(recv_all, send, group=group)
    recv = [recv_all[r][rank] for r in range(world)]
    tm = mark("partition", tm)
    if on_gpu:
        dst = torch.empty(sum(recv) * 4, dtype=torch.int64, device=device)
        dist.all_to_all_single(dst, src, [x * 4 for x in recv], [x * 4 for x in send], group=group)
    else:                                                         # gloo has no all-to-all: gather everything, keep my part
        parts = [None] * world
        dist.all_gather_object(parts, [x.cpu() for x in torch.split(src, [x * 4 for x in send])], group=group)
        dst = torch.cat([parts[r][rank] for r in range(world)]).to(device)
    torch.cuda.synchronize(device)
    tm = mark("all_to_all", tm)
    # Each rank's file slice precedes the next rank's, every sender sends in file order and the
    # received parts are laid out by source rank: the records are already ascending in position.
    n2 = int(dst.numel() // 4)
    engine.sc_import_packed_dev(n2, dst.data_ptr())
    engine.sc_set_collective(make_allreduce(device, group), rank, world)
    mark("import", tm)
    return n2


def sc_gather_triples(ensg, cell, count, group=None):
    """Concatenate the ranks' (ensg, cell, count) triples and sort by (ensg, cell): the job's
    final_results.  Every rank gets the full list (numpy arrays).  Host-side version for the gloo tests;
    with a library communicator use Engine.sc_allgather_triples() before sc_fetch instead."""
    import torch.distributed as dist
    world = dist.get_world_size(group)
    parts = [None] * world
    dist.all_gather_object(parts, (np.asarray(ensg), np.asarray(cell), np.asarray(count)), group=group)
    e = np.concatenate([q[0] for q in parts])
    c = np.concatenate([q[1] for q in parts])
    v = np.concatenate([q[2] for q in parts])
    o = np.lexsort((c, e))
    return e[o], c[o], v[o]
