"""Paired end by read name over byte ranges (csrc/bam_orch.h decode_range with MODE_PE_NAME_RANGE; include/tecount.h
tec_bam_count_range mode 4 and tec_bulk_name_partition_dev), run with host loops in place of the kernels
(tools/bgzf_dev_host.cpp).  For any number of ranks: the rows of the ranges, concatenated, are the rows of the whole file;
the rows each owner rank receives (key_lo % world, laid out by source rank) pair, by tests/pair_name_oracle.collate_by_name,
into exactly the whole file's pairs of the names it owns; and pairing inside each range would give other pairs."""
import ctypes
import os

import numpy as np
import pytest

import helpers as H
from bam_writer import write_bam
from pair_name_oracle import collate_by_name
from te_counter_b200 import reads, shard
from test_bam_ranges_pe_cpu import _session
from test_bgzf_dev_cpu import lib   # noqa: F401  (fixture)
from test_gpu_pair_name import _sorted_file

MODE_PE_NAME, MODE_PE_NAME_RANGE = 3, 4
COLS = ("start", "end", "chrom", "mapq", "flag", "key_hi", "key_lo", "role")
WORLDS = (1, 2, 3, 8, 37)
WINDOWS = (1, 7, 65536)


def _fetch(so, h, n):
    c = {"start": np.zeros(n, np.int32), "end": np.zeros(n, np.int32), "chrom": np.zeros(n, np.uint16),
         "mapq": np.zeros(n, np.uint8), "flag": np.zeros(n, np.uint8), "key_hi": np.zeros(n, np.uint64),
         "key_lo": np.zeros(n, np.uint64), "role": np.zeros(n, np.uint8)}
    p = lambda k: c[k].ctypes.data_as(ctypes.c_void_p)   # noqa: E731
    so.bgzfdev_fetch(h, p("start"), p("end"), p("chrom"), p("mapq"), p("flag"), None, None)
    so.bgzfdev_fetch_named(h, p("key_hi"), p("key_lo"), p("role"))
    return c


def _cm():
    return reads.ChromMap(H.load_index("idx_rand_a.glb").chrom_keys)


def _whole(so, path, window_blocks):
    h = _session(so, path, _cm())
    try:
        n = ctypes.c_int64(0)
        assert so.bgzfdev_decode(h, MODE_PE_NAME, 20, window_blocks, ctypes.byref(n)) == 0
        return _fetch(so, h, n.value)
    finally:
        so.bgzfdev_close(h)


def _range(so, path, window_blocks, lo, hi):
    h = _session(so, path, _cm())
    try:
        out = (ctypes.c_int64 * 6)()
        rc = so.bgzfdev_decode_range(h, MODE_PE_NAME_RANGE, 20, window_blocks, ctypes.c_int64(lo), ctypes.c_int64(hi), out)
        assert rc == 0, (rc, so.bgzfdev_error(h).decode())
        info = {"n": out[0], "start": (out[1], out[2]), "exit": (out[3], out[4]), "size": out[5]}
        return info, _fetch(so, h, out[0])
    finally:
        so.bgzfdev_close(h)


def _records(rows, index):
    """rows as collate_by_name input: the name is the 128-bit key, the SAM flag is rebuilt from the role"""
    flag = {0: 0, 1: 0x41, 2: 0x81}
    return [{"name": (int(a), int(b)), "flag": flag[int(r)], "i": int(i)}
            for a, b, r, i in zip(rows["key_hi"], rows["key_lo"], rows["role"], index)]


def _pairs(collated):
    return sorted((collated[k]["i"], collated[k + 1]["i"]) for k in range(0, len(collated), 2))


def _check_world(so, path, whole, window_blocks, world):
    """the three claims of the module docstring for one split; returns the per-range rows and the whole-file pairs"""
    size = os.path.getsize(path)
    infos, parts = zip(*[_range(so, path, window_blocks, *shard.byte_range(size, r, world)) for r in range(world)])
    assert shard.chain_is_consistent(list(infos)), (world, window_blocks, infos)
    for k in COLS:
        assert np.array_equal(np.concatenate([p[k] for p in parts]), whole[k]), (world, window_blocks, k)
    n = len(whole["start"])
    all_pairs, w_excl, w_no_mate = collate_by_name(_records(whole, range(n)))
    all_pairs = _pairs(all_pairs)
    owner_of = {i: int(k) % world for i, k in enumerate(whole["key_lo"])}
    base = np.cumsum([0] + [len(p["start"]) for p in parts])
    excluded = int(sum((p["role"] == 0).sum() for p in parts))            # the partition's count, rank by rank
    got, no_mate = [], 0
    for o in range(world):
        # what owner o receives: every rank's non-excluded rows of o's names, laid out by source rank, each in file order
        recv = []
        for r, p in enumerate(parts):
            keep = (p["role"] != 0) & (p["key_lo"] % np.uint64(world) == np.uint64(o))
            recv += _records({k: p[k][keep] for k in COLS}, base[r] + np.flatnonzero(keep))
        col, e, m = collate_by_name(recv)
        assert e == 0
        no_mate += m
        mine = _pairs(col)
        assert mine == [q for q in all_pairs if owner_of[q[0]] == o], (world, window_blocks, o)
        got += mine
    assert sorted(got) == all_pairs and excluded == w_excl and no_mate == w_no_mate
    return parts, all_pairs


@pytest.mark.parametrize("seed", [11, 12])
def test_owners_pair_the_sorted_files_like_the_whole_file(lib, tmp_path, seed):   # noqa: F811
    path = str(tmp_path / "s.bam")
    recs = _sorted_file(seed, 2000, path, block=1500)
    for window_blocks in WINDOWS:
        whole = _whole(lib, path, window_blocks)
        assert len(whole["start"]) == len(recs)
        for world in WORLDS:
            _check_world(lib, path, whole, window_blocks, world)


def _acdb_file(path):
    """One name q with read1 a (about 10 % into the file), read1 c and read2 d (about 45 % and 55 %) and read2 b (about
    90 %), between adjacent unique pairs; small blocks, so three byte ranges put a, {c, d} and b in ranges 0, 1, 2."""
    recs = []
    special = {100: ("q", 0x41, 1001), 450: ("q", 0x41, 1003), 550: ("q", 0x81, 1004), 900: ("q", 0x81, 1002)}
    for i in range(1000):
        if i in special:
            name, flag, start = special[i]
        else:
            name, flag, start = "f%d" % (i // 2), 0x41 if i % 2 == 0 else 0x81, 5000 + i
        recs.append({"name": name, "flag": flag, "chrom": "chr1", "start": start, "end": start + 60, "mapq": 60})
    write_bam(path, recs, block=400)


def test_the_acdb_name_across_three_ranges(lib, tmp_path):   # noqa: F811
    path = str(tmp_path / "acdb.bam")
    _acdb_file(path)
    for window_blocks in WINDOWS:
        whole = _whole(lib, path, window_blocks)
        idx = {int(s): i for i, s in enumerate(whole["start"]) if 1001 <= s <= 1004}
        a, b, c, d = idx[1001], idx[1002], idx[1003], idx[1004]
        for world in WORLDS:
            parts, all_pairs = _check_world(lib, path, whole, window_blocks, world)
            assert (a, d) in all_pairs and (c, b) in all_pairs and (c, d) not in all_pairs
            if world != 3:
                continue
            # the layout the case is about: a in range 0, c and d in range 1, b in range 2
            where = [{int(s) for s in p["start"] if 1001 <= s <= 1004} for p in parts]
            assert where == [{1001}, {1003, 1004}, {1002}]
            # pairing inside each range would count (c, d) and leave a and b without a mate
            base = np.cumsum([0] + [len(p["start"]) for p in parts])
            local = []
            for r, p in enumerate(parts):
                local += _pairs(collate_by_name(_records(p, base[r] + np.arange(len(p["start"]))))[0])
            assert (c, d) in local and (a, d) not in local and (c, b) not in local
            assert sorted(local) != all_pairs

