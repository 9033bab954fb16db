"""Pairing paired-end mates by read name (parse_bampe(pairing='name')) on CPU: the name key of csrc/bgzf_dev.h against a
numpy restatement, the device decoder's MODE_PE_NAME rows run by the host rehearsal (tools/bgzf_dev_host.cpp) against
bam.py, the collation rule of tests/pair_name_oracle.py on hand-made cases, and the CLI.  The device pairing stage is
held against collate_by_name in test_gpu_pair_name.py."""
import ctypes
import random

import numpy as np
import pytest

import helpers as H
from bam_writer import write_bam
from oracle import te_oracle
from pair_name_oracle import collate_by_name, name_role
from te_counter_b200 import bam, reads, sharded
from test_bgzf_dev_cpu import lib  # noqa: F401  (fixture: builds and loads tools/libbgzfdevhost.so)

MODE_PE_NAME = 3
U = np.uint64


def _mix(h):
    h = h ^ (h >> U(30))
    h = h * U(0xbf58476d1ce4e5b9)
    h = h ^ (h >> U(27))
    h = h * U(0x94d049bb133111eb)
    return h ^ (h >> U(31))


def np_name_key(names):
    """bgzfdev::name_key restated: (hi, lo) uint64 arrays for a list of byte strings."""
    n = len(names)
    ln = np.array([len(x) for x in names], dtype=np.uint64)
    width = int(ln.max()) if n else 0
    buf = np.zeros((n, max(width, 1)), dtype=np.uint64)
    for i, x in enumerate(names):
        buf[i, :len(x)] = np.frombuffer(x, dtype=np.uint8)
    a = np.full(n, 0xcbf29ce484222325, dtype=np.uint64)
    b = np.uint64(0x9e3779b97f4a7c15) ^ ln
    with np.errstate(over="ignore"):
        for i in range(width):
            live = ln > U(i)
            c = buf[:, i]
            a2 = (a ^ c) * U(0x100000001b3)
            b2 = (b + c + U(1)) * U(0xff51afd7ed558ccd)
            b2 = b2 ^ (b2 >> U(29))
            a = np.where(live, a2, a)
            b = np.where(live, b2, b)
        return _mix(a ^ (ln << U(56))), _mix(b)


def test_name_key_matches_numpy(lib):  # noqa: F811
    lib.bgzfdev_name_key.argtypes = [ctypes.c_char_p, ctypes.c_uint32, ctypes.c_void_p]
    rnd = random.Random(5)
    names = [bytes(rnd.randrange(0x21, 0x7f) for _ in range(k)) for k in range(1, 255)]
    names += [b"q1", b"q1/1", b"q1/2", b"q2", b"A" * 254]
    hi, lo = np_name_key(names)
    for i, x in enumerate(names):
        out = np.zeros(2, np.uint64)
        lib.bgzfdev_name_key(x, len(x), out.ctypes.data)
        assert (int(out[0]), int(out[1])) == (int(hi[i]), int(lo[i])), x
    assert len(set(zip(hi.tolist(), lo.tolist()))) == len(names)


def test_name_role_matches_oracle(lib):  # noqa: F811
    for f in range(0, 0x1000):
        assert lib.bgzfdev_name_role(f) == name_role(f), hex(f)


def _named_records(n, seed):
    """Records of every flag kind, names of 1 to 200 characters, some names shared by several records."""
    rnd = random.Random(seed)
    flags = [0x41, 0x81, 0x61, 0x91, 0x141, 0x881, 0x1, 0xc1, 0x40, 0x45, 0x89, 0x441, 0x281, 0]
    recs = []
    for i in range(n):
        name = "r%d_" % rnd.randrange(n // 3 + 1) + "x" * rnd.randrange(0, 190)
        f = rnd.choice(flags)
        chrom = None if f & 4 and rnd.random() < 0.5 else rnd.choice(["chr1", "chr2", "chrX", "chrUn_x"])
        s = rnd.randrange(0, 200000)
        recs.append({"chrom": chrom, "start": s if chrom else -1, "end": s + rnd.randrange(20, 300) if chrom else -1,
                     "flag": f, "mapq": rnd.choice([0, 10, 30, 60, 255]), "name": name})
    return recs


@pytest.mark.parametrize("block,window_blocks", [(97, 1), (97, 7), (700, 2), (3000, 1 << 20), (20000, 3), (65000, 1)])
def test_mode3_rows_keys_roles_match_bam_py(lib, tmp_path, block, window_blocks):  # noqa: F811
    recs = _named_records(3001, block)
    path = str(tmp_path / "x.bam")
    write_bam(path, recs, block=block)
    idx = H.load_index("idx_rand_a.glb")
    cm = reads.ChromMap(idx.chrom_keys)
    f = bam.AlignmentFile(path, "r")
    want = list(f)
    f.close()
    h = ctypes.c_void_p()
    assert lib.bgzfdev_open(path.encode(), ctypes.byref(h)) == 0
    try:
        lib.bgzfdev_reference_name.restype = ctypes.c_char_p
        refs = [lib.bgzfdev_reference_name(h, i).decode() for i in range(lib.bgzfdev_n_references(h))]
        bulk = np.array([cm.bulk_id(x) for x in refs], dtype=np.uint16)
        assert lib.bgzfdev_set_chrom_map(h, bulk.ctypes.data_as(ctypes.c_void_p), bulk.ctypes.data_as(ctypes.c_void_p), len(refs), cm.n_index) == 0
        n = ctypes.c_int64(0)
        assert lib.bgzfdev_decode(h, MODE_PE_NAME, 20, window_blocks, ctypes.byref(n)) == 0
        n = n.value
        assert n == len(want)
        cols = {"start": np.zeros(n, np.int32), "end": np.zeros(n, np.int32), "chrom": np.zeros(n, np.uint16),
                "mapq": np.zeros(n, np.uint8), "flag": np.zeros(n, np.uint8)}
        lib.bgzfdev_fetch(h, *[cols[k].ctypes.data_as(ctypes.c_void_p) for k in cols], None, None)
        key_hi, key_lo, role = np.zeros(n, np.uint64), np.zeros(n, np.uint64), np.zeros(n, np.uint8)
        lib.bgzfdev_fetch_named(h, key_hi.ctypes.data_as(ctypes.c_void_p), key_lo.ctypes.data_as(ctypes.c_void_p),
                                role.ctypes.data_as(ctypes.c_void_p))
        # byte ranges refuse the mode: pairing needs the whole file
        out = (ctypes.c_int64 * 6)()
        assert lib.bgzfdev_decode_range(h, MODE_PE_NAME, 20, window_blocks, 0, 1 << 40, out) == -4
    finally:
        lib.bgzfdev_close(h)
    hi, lo = np_name_key([r.query_name.encode() for r in want])
    w_role = np.array([name_role(r.flag) for r in want], np.uint8)
    assert np.array_equal(role, w_role)
    part = w_role > 0
    assert np.array_equal(key_hi, np.where(part, hi, 0)) and np.array_equal(key_lo, np.where(part, lo, 0))
    assert np.array_equal(cols["start"], [r.reference_start if r.reference_start is not None else -1 for r in want])
    assert np.array_equal(cols["end"], [r.reference_end if r.reference_end is not None else -1 for r in want])
    assert np.array_equal(cols["chrom"], [cm.bulk_id(r.reference_name) for r in want])
    assert np.array_equal(cols["mapq"], [r.mapping_quality for r in want])
    assert np.array_equal(cols["flag"], [reads._flagbits(r) for r in want])


def _r(name, flag, i):
    return {"name": name, "flag": flag, "i": i}


def _ids(collated):
    return [r["i"] for r in collated]


def test_collate_hand_made_cases():
    # mates next to each other, far apart (other blocks / windows), first and last record of the file
    recs = [_r("a", 0x41, 0), _r("b", 0x41, 1), _r("b", 0x81, 2), _r("c", 0x81, 3), _r("c", 0x41, 4), _r("a", 0x81, 5)]
    col, excl, no_mate = collate_by_name(recs)
    assert _ids(col) == [1, 2, 4, 3, 0, 5] and (excl, no_mate) == (0, 0)
    # secondary, supplementary, 0x1 clear, both or neither mate flag: excluded
    recs = [_r("a", 0x141, 0), _r("a", 0x841, 1), _r("a", 0x40, 2), _r("a", 0xc1, 3), _r("a", 0x1, 4), _r("a", 0x41, 5), _r("a", 0x81, 6)]
    col, excl, no_mate = collate_by_name(recs)
    assert _ids(col) == [5, 6] and (excl, no_mate) == (5, 0)
    # two read1 and one read2: the first read1 pairs, the second has no mate
    col, excl, no_mate = collate_by_name([_r("a", 0x41, 0), _r("a", 0x41, 1), _r("a", 0x81, 2)])
    assert _ids(col) == [0, 2] and (excl, no_mate) == (0, 1)
    # k-th read1 with k-th read2, whichever comes first
    col, _, no_mate = collate_by_name([_r("a", 0x81, 0), _r("a", 0x41, 1), _r("a", 0x41, 2), _r("a", 0x81, 3), _r("a", 0x81, 4)])
    assert _ids(col) == [1, 0, 2, 3] and no_mate == 1
    # a missing mate; names that differ only after a '/' are different names; an odd record total
    col, excl, no_mate = collate_by_name([_r("q/1", 0x41, 0), _r("q/2", 0x81, 1), _r("z", 0x41, 2)])
    assert col == [] and (excl, no_mate) == (0, 3)
    # an unmapped mate is still a mate (the PE loop rejects the pair as QC fail)
    col, _, _ = collate_by_name([_r("u", 0x49, 0), _r("u", 0x85, 1)])
    assert _ids(col) == [0, 1]


def test_collate_on_mates_on_other_chromosomes_gives_the_reference_counts():
    """A pair whose mates are on two chromosomes, collated, counts as read1's chromosome (te_count.py:96)."""
    idx = H.load_index("idx_toy.glb")
    oidx = te_oracle.Index(idx.chrom_id, idx.L, idx.R, idx.ensg_id, idx.type_code, idx.strand_code, idx.n_ensg, idx.bucket_size)
    cm = reads.ChromMap(idx.chrom_keys)
    recs = [{"name": "p", "flag": 0x41, "chrom": "chr1", "start": 1600, "mapq": 60},
            {"name": "o", "flag": 0x41, "chrom": "chr1", "start": 5100, "mapq": 60},
            {"name": "o", "flag": 0x81, "chrom": "chr1", "start": 20100, "mapq": 60},
            {"name": "p", "flag": 0x81, "chrom": "chrZ", "start": 1700, "mapq": 60}]
    col, _, _ = collate_by_name(recs)
    cols = [[r["start"] for r in col], [r["start"] + 50 for r in col], [cm.bulk_id(r["chrom"]) for r in col],
            [r["mapq"] for r in col], [0] * len(col)]
    counts, st = te_oracle.bulk_count(oidx, True, 20, *cols)
    assert st["total_reads"] == 3 and st["badchrom"] == 0 and sum(counts) > 0


@pytest.mark.parametrize("name", H.case_names("bulk_pe"))
def test_collate_of_a_collated_file_is_index_pairing(name):
    """On a name-collated file of primary pairs, collate_by_name gives back the pairs of index pairing."""
    case = H.load_case(name)
    recs = [dict(r, i=i, name="p%d" % (i // 2), flag=(r.get("flag", 0) & ~0x900) | (0x41 if i % 2 == 0 else 0x81))
            for i, r in enumerate(case["records"])]
    col, excl, no_mate = collate_by_name(recs)
    n = len(recs) // 2 * 2
    assert _ids(col) == list(range(n)) and excl == 0 and no_mate == len(recs) - n


def test_cli_rejects_name_pairing_outside_paired_end(capsys):
    for mode in ("se", "sc"):
        with pytest.raises(SystemExit) as e:
            sharded.main(["--glb", "x.glb", "--bam", "x.bam", "--mode", mode, "--pairing", "name", "-o", "out"])
        assert e.value.code == 2
        assert "--pairing name" in capsys.readouterr().err
