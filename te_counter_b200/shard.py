"""
One BAM file counted by several ranks (one process per GPU): every rank decodes a byte range of the file on its own
GPU (tec_bam_count_range: BGZF inflate, record split and packing on the device), the ranks check that their ranges tile
the file's record chain exactly, and the partial results are merged -- one all-reduce of the counters in bulk mode
(te_count.py:42-277), the exchange of the survivors by cell plus the job-wide collectives of tec_sc_finalize in
single-cell mode (te_count.py:298-707; the records of rank r precede those of rank r + 1, so the job-wide record order
is the file's).

Paired end: the reference pairs records by their global index (te_count.py:76-79: record 2i is read1, 2i + 1 read2, a
trailing odd record is dropped), whose parity a rank cannot know before the ranks in front of it have counted theirs.
So every rank counts every adjacent pair of its range into one of two counter banks (pair (j, j + 1) of range-local
index j into bank j & 1), and once the gathered record counts give its global offset o it keeps bank o & 1
(pair_plan).  If o is odd, the rank's first record is read2 of a pair whose read1 is the last record of the nearest
rank in front that has records: the ranks hand out their first and last records with their range info, and the rank
parses that pair on the host and counts it.

Paired end by read name (parse_bampe(pairing='name'), mode 4): the k-th read1 of a name pairs with its k-th read2 over
the whole file, and mates lie in any range.  So a rank's range pairs nothing: its rows are held, then sent to the rank
that owns their name (dist.bulk_name_exchange), which pairs them in file order.  There is no pair plan.

The reference has no counterpart (it is one process); results are identical to the single-GPU run, byte for byte.
"""
import os


def byte_range(size, rank, world):
    """[lo, hi) of rank's share of a file of `size` bytes; rank 0 starts at 0 (the BAM header)."""
    return size * rank // world, size * (rank + 1) // world


def chain_is_consistent(infos):
    """infos[rank] = DeviceBam.count_range(...) of every rank, in rank order.  True iff the ranges tile the record chain:
    rank 0 starts at the header, every exit is the start of the next rank that has records, the last exit is the end of
    the file.  (A first record found by the block-parallel guess is only proven right by the rank in front of it.)"""
    if not infos or tuple(infos[0]["start"])[0] != -1:
        return False
    at = None
    for i in infos:
        s, e = tuple(i["start"]), tuple(i["exit"])
        if s[0] == -2:                       # no record starts in this range
            if i["n"]:
                return False
            continue
        if at is not None and s != at:
            return False
        at = e
    return at is not None and at == (infos[0]["size"], 0)


def pair_plan(infos):
    """Paired end, for infos that pass chain_is_consistent (each with n, and first / last = raw first / last record of
    the range): per rank {"bank": parity of the rank's global record offset, "border": (read1, read2) raw records of the
    pair across the rank's front border, or None}."""
    plan, offset, last = [], 0, None
    for i in infos:
        border = (last, i["first"]) if i["n"] and offset & 1 else None
        plan.append({"bank": offset & 1, "border": border})
        if i["n"]:
            last = i["last"]
        offset += i["n"]
    return plan


def world_info(group=None):
    """(rank, world) of the torch.distributed job this process belongs to, (0, 1) outside one."""
    try:
        import torch.distributed as dist
    except ImportError:
        return 0, 1
    if not (dist.is_available() and dist.is_initialized()):
        return 0, 1
    return dist.get_rank(group), dist.get_world_size(group)


def count_ranges(open_and_bind, mode, qual, group=None):
    """Every rank decodes its byte range into the running count of its engine.  open_and_bind() returns the rank's
    DeviceBam (opened, chromosome map and whitelist set).  Returns (records of this rank, records of the job, pair),
    or None when a rank's decoder refused the file or the ranges do not tile it: the caller then starts over with one
    decoder.  Modes: 0 single end, 1 paired end, 2 single cell, 4 paired end by read name (rows held for the exchange).
    pair is None except in paired-end mode (1), where it is (bank to keep, columns of the border pair or None;
    pair_plan): the caller passes the bank to Engine.bulk_keep_bank and pushes the two rows.
    Collective: every rank of the group must call it."""
    import torch.distributed as dist
    rank, world = world_info(group)
    dev_bam = None
    try:
        try:
            dev_bam = open_and_bind()
            lo, hi = byte_range(os.path.getsize(dev_bam.filename), rank, world)
            info = dev_bam.count_range(mode, qual, lo, hi)
            if os.environ.get("TEC_TEST_SHARD_REFUSE") == str(rank):     # tests: one rank reports a start its neighbour cannot confirm
                info["start"] = (info["start"][0], info["start"][1] + 1)
        except Exception as e:               # a refusal on one rank must reach all of them
            info = {"error": "%s: %s" % (type(e).__name__, e)}
        infos = [None] * world
        dist.all_gather_object(infos, info, group=group)
        if any("error" in i for i in infos) or not chain_is_consistent(infos):
            return None
        pair = None
        if mode == 1:
            plan = pair_plan(infos)[rank]
            try:
                border = dev_bam.pair_columns(*plan["border"], qual) if plan["border"] else None
                ok = True
            except Exception:
                border, ok = None, False
            oks = [None] * world             # the border parse is the last step that can fail on one rank alone
            dist.all_gather_object(oks, ok, group=group)
            if not all(oks):
                return None
            pair = (plan["bank"], border)
        return info["n"], sum(i["n"] for i in infos), pair
    finally:
        if dev_bam is not None:
            dev_bam.close()


def join_collectives(engine, group=None):
    """Give the engine its NCCL communicator once (dist.comm_init) where the job runs over NCCL; True when the library
    issues the collectives itself, False when they go through torch.distributed on the host (gloo)."""
    from . import dist as tdist
    rank, world = world_info(group)
    if world <= 1:
        return False
    if engine.comm_world()[1] == world:
        return True
    return tdist.comm_init(engine, group)
