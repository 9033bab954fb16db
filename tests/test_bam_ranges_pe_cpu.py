"""Paired end over byte ranges (csrc/bam_orch.h decode_range with MODE_PE; include/tecount.h tec_bam_count_range mode 1,
tec_bam_range_record, tec_bam_pair_columns), run with host loops in place of the kernels (tools/bgzf_dev_host.cpp): for
any number of ranks, each rank's border pair (parsed on the host) followed by the column set of its parity
(shard.pair_plan), concatenated in rank order, are the columns of the whole file decoded in one piece -- row for row,
flag bits included."""
import ctypes
import functools
import os
import tempfile

import numpy as np
import pytest

import helpers as H
from bam_writer import write_bam
from te_counter_b200 import reads, shard
from test_bgzf_dev_cpu import _decode, lib   # noqa: F401  (fixture)
from test_fastbam import _mixed_records

KEYS = ("start", "end", "chrom", "mapq", "flag")
F_NAME_MISMATCH = 16
WORLDS = (1, 2, 3, 8, 37)


def _session(so, path, cm):
    h = ctypes.c_void_p()
    assert so.bgzfdev_open(path.encode(), ctypes.byref(h)) == 0
    refs = [so.bgzfdev_reference_name(h, i).decode() for i in range(so.bgzfdev_n_references(h))]
    bulk = np.array([cm.bulk_id(n) for n in refs], dtype=np.uint16)
    sc = np.zeros(len(refs), dtype=np.uint16)
    assert so.bgzfdev_set_chrom_map(h, bulk.ctypes.data_as(ctypes.c_void_p), sc.ctypes.data_as(ctypes.c_void_p), len(refs), cm.n_index) == 0
    return h


def _cols(n):
    return {"start": np.zeros(n, np.int32), "end": np.zeros(n, np.int32), "chrom": np.zeros(n, np.uint16),
            "mapq": np.zeros(n, np.uint8), "flag": np.zeros(n, np.uint8)}


def _ptrs(cols):
    return [cols[k].ctypes.data_as(ctypes.c_void_p) for k in KEYS]


def _record(so, h, which):
    n = ctypes.c_int64(0)
    assert so.bgzfdev_range_record(h, which, None, ctypes.c_int64(0), ctypes.byref(n)) == 0
    buf = ctypes.create_string_buffer(max(1, n.value))
    assert so.bgzfdev_range_record(h, which, buf, ctypes.c_int64(n.value), ctypes.byref(n)) == 0
    return buf.raw[:n.value]


def _decode_range_pe(so, path, cm, qual, window_blocks, lo, hi):
    """info (n, start, exit, size, first, last) and the two column sets of one range"""
    h = _session(so, path, cm)
    try:
        out = (ctypes.c_int64 * 6)()
        rc = so.bgzfdev_decode_range(h, 1, qual, window_blocks, ctypes.c_int64(lo), ctypes.c_int64(hi), out)
        assert rc == 0, (rc, so.bgzfdev_error(h).decode())
        sets = []
        for bank in (0, 1):
            c = _cols(so.bgzfdev_set_rows(h, bank))
            so.bgzfdev_fetch_set(h, bank, *_ptrs(c))
            sets.append(c)
        info = {"n": out[0], "start": (out[1], out[2]), "exit": (out[3], out[4]), "size": out[5],
                "first": _record(so, h, 0), "last": _record(so, h, 1)}
        return info, sets
    finally:
        so.bgzfdev_close(h)


def _pair(so, h, rec1, rec2, qual):
    c = _cols(2)
    rc = so.bgzfdev_pair_columns(h, rec1, ctypes.c_int64(len(rec1)), rec2, ctypes.c_int64(len(rec2)), qual, *_ptrs(c))
    assert rc == 0, (rc, so.bgzfdev_error(h).decode())
    return c


def _long_name_records(n, style):
    """200-character names (records longer than a 97-byte block: many ranks get 0 or 1 records); every third pair's
    mates differ before the '/'; some pairs rejected by read2's flags or read1's MAPQ."""
    recs = []
    for i in range(n):
        k = i // 2
        stem = ("n" * 190 + "%06d" % k) if style == 0 else ("q%d_" % k).ljust(196, "n")
        if i % 2 and k % 3 == 0:
            stem += "x"
        flag = 0x400 if i % 2 and k % 7 == 2 else 0
        recs.append({"chrom": "chr1", "start": 100 + i, "end": 180 + i, "flag": flag, "mapq": 5 if i % 2 == 0 and k % 5 == 1 else 60,
                     "name": "%s/%d" % (stem, i % 2 + 1)})
    return recs


# name: (records, count, block bytes, window_blocks, world sizes).  With windows of one or two 97-byte blocks a range's
# first-record guess is only checked inside its window, and at larger world sizes the chain check refuses some splits
# of these files (in single-end mode too; the callers then decode the file in one piece): those cases run at the world
# sizes the split accepts.
CASES = {
    "odd_3000B_whole": ("mixed", 5001, 3000, 1 << 20, WORLDS),
    "even_700B_w5": ("mixed", 5000, 700, 5, WORLDS),
    "odd_65kB_w2": ("mixed", 6001, 65000, 2, WORLDS),
    "long_names_odd_w7": ("long0", 61, 97, 7, WORLDS),
    "long_names_even_w7": ("long1", 80, 97, 7, WORLDS),
    "long_names_odd_w1": ("long0", 61, 97, 1, (1, 2, 3)),
    "long_names_even_w2": ("long1", 80, 97, 2, (1, 2)),
}


@functools.lru_cache(maxsize=None)
def _run_case(so, name):
    kind, n, block, window_blocks, worlds = CASES[name]
    recs = _mixed_records(n, 91 + block, False)[0] if kind == "mixed" else _long_name_records(n, int(kind[-1]))
    path = os.path.join(tempfile.mkdtemp(prefix="pe_ranges_"), "x.bam")
    write_bam(path, recs, block=block)
    idx = H.load_index("idx_rand_a.glb")
    cm = lambda: reads.ChromMap(idx.chrom_keys)   # noqa: E731
    rc, _, whole = _decode(so, path, "pe", cm(), None, 20, window_blocks)
    assert rc == 0 and len(whole["start"]) == n - n % 2
    size = os.path.getsize(path)
    seen = {"border": 0, "banks": set(), "border_mismatch": 0, "zero_or_one": 0}
    h = _session(so, path, cm())
    try:
        for world in worlds:
            infos, sets = [], []
            for rank in range(world):
                info, s = _decode_range_pe(so, path, cm(), 20, window_blocks, *shard.byte_range(size, rank, world))
                infos.append(info)
                sets.append(s)
            assert shard.chain_is_consistent(infos), (world, infos)
            assert sum(i["n"] for i in infos) == n
            plan = shard.pair_plan(infos)
            parts = []
            for p, s in zip(plan, sets):
                if p["border"] is not None:
                    b = _pair(so, h, *p["border"], 20)
                    parts.append(b)
                    seen["border"] += 1
                    seen["border_mismatch"] += int(b["flag"][0] & F_NAME_MISMATCH != 0)
                parts.append(s[p["bank"]])
                seen["banks"].add(p["bank"])
            for k in KEYS:
                got = np.concatenate([q[k] for q in parts])
                assert np.array_equal(got, whole[k]), (name, world, k)
            seen["zero_or_one"] += sum(1 for i in infos if i["n"] <= 1)
    finally:
        so.bgzfdev_close(h)
    return seen


@pytest.mark.parametrize("name", sorted(CASES))
def test_pe_ranges_concatenate_to_the_whole_file(lib, name):   # noqa: F811
    seen = _run_case(lib, name)
    if name.startswith("long_names") and CASES[name][4] == WORLDS:
        assert seen["zero_or_one"] > 0            # ranks with 0 or 1 records took part


def test_the_cases_meet_border_pairs_both_banks_and_a_mismatched_border(lib):   # noqa: F811
    runs = [_run_case(lib, name) for name in sorted(CASES)]
    assert sum(r["border"] for r in runs) > 0
    assert set().union(*(r["banks"] for r in runs)) == {0, 1}
    assert sum(r["border_mismatch"] for r in runs) > 0


def test_pair_across_windows_is_counted_once(lib, tmp_path):   # noqa: F811
    """One range (the whole file) at one block per window: the two sets together hold every adjacent pair once."""
    recs = _mixed_records(701, 5, False)[0]
    path = str(tmp_path / "x.bam")
    write_bam(path, recs, block=150)
    cm = reads.ChromMap(H.load_index("idx_rand_a.glb").chrom_keys)
    info, sets = _decode_range_pe(lib, path, cm, 20, 1, 0, os.path.getsize(path))
    assert info["n"] == 701
    assert len(sets[0]["start"]) == 700 and len(sets[1]["start"]) == 700      # 700 adjacent pairs, 350 in each set
    rc, _, whole = _decode(lib, path, "pe", cm, None, 20, 1)
    for k in KEYS:
        assert np.array_equal(sets[0][k], whole[k]), k
    # set 1 holds the pairs (1, 2), (3, 4), ...: read2 rows are read1 rows of set 0 shifted by one record
    assert np.array_equal(sets[1]["start"][0::2], whole["start"][1::2])
    assert np.array_equal(sets[1]["start"][1:-1:2], whole["start"][2::2])


def test_pair_columns_refuses_a_partial_record(lib, tmp_path):   # noqa: F811
    recs = _mixed_records(10, 3, False)[0]
    path = str(tmp_path / "x.bam")
    write_bam(path, recs)
    cm = reads.ChromMap(["1"])
    info, _ = _decode_range_pe(lib, path, cm, 20, 4, 0, os.path.getsize(path))
    h = _session(lib, path, cm)
    try:
        c = _cols(2)
        a, b = info["first"], info["last"]
        assert lib.bgzfdev_pair_columns(h, a, ctypes.c_int64(len(a)), b, ctypes.c_int64(len(b)), 20, *_ptrs(c)) == 0
        assert lib.bgzfdev_pair_columns(h, a, ctypes.c_int64(len(a) - 1), b, ctypes.c_int64(len(b)), 20, *_ptrs(c)) == -4
    finally:
        lib.bgzfdev_close(h)


def _info(n, first=b"", last=b""):
    return {"n": n, "first": first, "last": last}


def test_pair_plan_by_hand():
    # ranks without records are skipped when looking for read1 of a border pair
    infos = [_info(3, b"a0", b"a2"), _info(0), _info(1, b"b0", b"b0"), _info(0), _info(2, b"c0", b"c1"), _info(1, b"d0", b"d0")]
    plan = shard.pair_plan(infos)
    assert [p["bank"] for p in plan] == [0, 1, 1, 0, 0, 0]
    assert [p["border"] for p in plan] == [None, None, (b"a2", b"b0"), None, None, None]
    # odd total: nobody claims the last record
    plan = shard.pair_plan([_info(1, b"x", b"x"), _info(1, b"y", b"y"), _info(1, b"z", b"z")])
    assert [p["bank"] for p in plan] == [0, 1, 0]
    assert [p["border"] for p in plan] == [None, (b"x", b"y"), None]
    # a rank of one record after an odd offset is read2 and nothing else
    plan = shard.pair_plan([_info(0), _info(5, b"p", b"q"), _info(1, b"r", b"r"), _info(0), _info(4, b"s", b"t")])
    assert [p["bank"] for p in plan] == [0, 0, 1, 0, 0]
    assert plan[2]["border"] == (b"q", b"r") and plan[4]["border"] is None
