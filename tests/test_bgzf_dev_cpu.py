"""The block-parallel BAM decoder that runs on the GPU (csrc/bgzf_dev.h per-block routines,
csrc/bam_orch.h window loop), executed here with host loops in place of the kernels
(tools/bgzf_dev_host.cpp): same arrays as libtecbam (tests/test_fastbam.py pins that one to the
Python packing), the same refusals on damaged files, inflate equal to zlib."""
import ctypes
import os
import subprocess
import zlib

import numpy as np
import pytest

import helpers as H
from bam_writer import write_bam
from te_counter_b200 import build, fastbam, reads
from test_fastbam import _mixed_records, _native_batches

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "tools", "libbgzfdevhost.so")
MODES = {"se": 0, "pe": 1, "sc": 2}


@pytest.fixture(scope="module")
def lib():
    build.build_bam()
    src = [os.path.join(ROOT, "tools", "bgzf_dev_host.cpp"), os.path.join(ROOT, "te_counter_b200", "csrc", "bgzf_dev.h"),
           os.path.join(ROOT, "te_counter_b200", "csrc", "bam_orch.h")]
    if not os.path.exists(LIB) or any(os.path.getmtime(s) > os.path.getmtime(LIB) for s in src):
        subprocess.run(["g++", "-O2", "-std=c++17", "-Wall", "-shared", "-fPIC", src[0], "-lz", "-o", LIB], check=True)
    so = ctypes.CDLL(LIB)
    so.bgzfdev_error.restype = ctypes.c_char_p
    so.bgzfdev_reference_name.restype = ctypes.c_char_p
    return so


def _decode(so, path, mode, cm, wl, qual, window_blocks, decline=0):
    h = ctypes.c_void_p()
    rc = so.bgzfdev_open(path.encode(), ctypes.byref(h))
    assert rc == 0, rc
    try:
        refs = [so.bgzfdev_reference_name(h, i).decode() for i in range(so.bgzfdev_n_references(h))]
        bulk = np.array([cm.bulk_id(n) for n in refs], dtype=np.uint16)
        sc = np.empty(len(refs), dtype=np.uint16)
        for i, n in enumerate(refs):
            try:
                sc[i] = cm.sc_id(n)
            except ValueError:
                sc[i] = fastbam.CHROM_SC_BAD
        assert so.bgzfdev_set_chrom_map(h, bulk.ctypes.data_as(ctypes.c_void_p), sc.ctypes.data_as(ctypes.c_void_p), len(refs), cm.n_index) == 0
        if wl is not None:
            enc = [b.encode() for b in wl.id_to_barcode]
            off = np.zeros(len(enc) + 1, dtype=np.int64)
            np.cumsum([len(b) for b in enc], out=off[1:])
            assert so.bgzfdev_set_whitelist(h, b"".join(enc), off.ctypes.data_as(ctypes.c_void_p), len(enc)) == 0
        so.bgzfdev_force_decline(h, decline)
        n = ctypes.c_int64(0)
        rc = so.bgzfdev_decode(h, MODES[mode], qual, window_blocks, ctypes.byref(n))
        if rc:
            return rc, so.bgzfdev_error(h).decode(), None
        n = n.value
        cols = {"start": np.zeros(n, np.int32), "end": np.zeros(n, np.int32), "chrom": np.zeros(n, np.uint16),
                "mapq": np.zeros(n, np.uint8), "flag": np.zeros(n, np.uint8), "cell": np.zeros(n, np.uint32), "umi": np.zeros(n, np.uint64)}
        so.bgzfdev_fetch(h, *[cols[k].ctypes.data_as(ctypes.c_void_p) for k in ("start", "end", "chrom", "mapq", "flag", "cell", "umi")])
        return 0, so.bgzfdev_declined(h), cols
    finally:
        so.bgzfdev_close(h)


def _native(path, mode, cm, wl, qual):
    bs = _native_batches(path, mode, cm, wl, qual, 1 << 16, 2)
    return {k: np.concatenate([getattr(b, k)[:b.n] for b, _ in bs]) for k in
            ("start", "end", "chrom", "mapq", "flag") + (("cell", "umi") if mode == "sc" else ())}


@pytest.mark.parametrize("mode", ["se", "pe", "sc"])
@pytest.mark.parametrize("block,window_blocks,decline", [(3000, 1 << 20, 0), (700, 5, 0), (65000, 1, 0), (64, 13, 0), (20000, 3, 2)])
def test_same_arrays_as_libtecbam(lib, tmp_path, mode, block, window_blocks, decline):
    recs, wl_list = _mixed_records(5000 + (mode == "pe"), 23 + block, mode == "sc")
    path = str(tmp_path / "x.bam")
    write_bam(path, recs, block=block)
    idx = H.load_index("idx_rand_a.glb")
    wl = None
    if mode == "sc":
        wlf = tmp_path / "wl.txt"
        wlf.write_text("".join(w + "\n" for w in wl_list))
        wl = reads.Whitelist(str(wlf))
    want = _native(path, mode, reads.ChromMap(idx.chrom_keys), wl, 20)
    rc, declined, got = _decode(lib, path, mode, reads.ChromMap(idx.chrom_keys), wl, 20, window_blocks, decline)
    assert rc == 0, declined
    assert (declined > 0) == (decline > 0)   # the block inflate handles everything zlib emits
    for k in want:
        assert np.array_equal(want[k], got[k]), k


def test_long_records_and_tiny_blocks(lib, tmp_path):
    """Records much longer than a block (no record start in most blocks) and a window of one block."""
    recs = [{"chrom": "chr1", "start": 100 + i, "end": 150 + i, "name": "n" * 200 + str(i)} for i in range(300)]
    path = str(tmp_path / "x.bam")
    write_bam(path, recs, block=97)
    cm = reads.ChromMap(["1"])
    want = _native(path, "se", cm, None, 0)
    for wb in (1, 2, 7, 1000):
        rc, _, got = _decode(lib, path, "se", reads.ChromMap(["1"]), None, 0, wb)
        assert rc == 0
        for k in want:
            assert np.array_equal(want[k], got[k]), (k, wb)


def test_empty_truncated_and_corrupt(lib, tmp_path):
    path = str(tmp_path / "e.bam")
    write_bam(path, [])
    rc, _, got = _decode(lib, path, "pe", reads.ChromMap(["1"]), None, 20, 8)
    assert rc == 0 and len(got["start"]) == 0
    recs = [{"chrom": "chr1", "start": 100 + i, "end": 150 + i} for i in range(2000)]
    write_bam(path, recs, block=20000)
    raw = open(path, "rb").read()

    def run(data):
        p = str(tmp_path / "y.bam")
        open(p, "wb").write(data)
        return _decode(lib, p, "se", reads.ChromMap(["1"]), None, 0, 4)[:2]

    assert run(raw)[0] == 0
    flipped = bytearray(raw)
    flipped[len(raw) // 2] ^= 0x55
    assert run(bytes(flipped))[0] == -2
    assert run(raw[:len(raw) // 2])[0] == -2
    blocks, o = [], 0
    while o < len(raw):
        n = int.from_bytes(raw[o + 16:o + 18], "little") + 1
        blocks.append(raw[o:o + n])
        o += n
    rc, msg = run(b"".join(blocks[:3]))
    assert rc == -2 and "truncated" in msg


def test_record_errors_name_the_first_record(lib, tmp_path):
    ok = {"chrom": "chr1", "start": 1600, "end": 1650, "CB": "AAAA", "UB": "ACGT"}
    wlf = tmp_path / "wl.txt"
    wlf.write_text("AAAA\n")
    wl = reads.Whitelist(str(wlf))
    idx = H.load_index("idx_toy.glb")
    path = str(tmp_path / "x.bam")
    for bad, code in ((dict(ok, CB=None), 10), (dict(ok, UB=None), 11), (dict(ok, UB="ACGX"), 12), (dict(ok, end=1600), 13),
                      (dict(ok, chrom="HLA:A"), 14)):
        write_bam(path, [ok] * 7 + [bad] + [ok] * 5 + [bad], block=300)
        rc, msg, _ = _decode(lib, path, "sc", reads.ChromMap(idx.chrom_keys), wl, 20, 3)
        assert rc == -100 - code and msg == "record 7", (rc, msg)


def test_block_inflate_equals_zlib(lib):
    rng = np.random.default_rng(9)
    n_declined = 0
    for trial in range(300):
        n = int(rng.integers(0, 65537 if trial % 5 == 0 else 4000))
        data = rng.integers(0, 1 + int(rng.integers(1, 200)), n, dtype=np.uint8).tobytes()
        if trial % 3 == 0 and n > 100:
            data = (data[:97] * (n // 97 + 1))[:n]
        co = zlib.compressobj(int(rng.integers(0, 10)), zlib.DEFLATED, -15, 8,
                              [zlib.Z_DEFAULT_STRATEGY, zlib.Z_FIXED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE][trial % 4])
        comp = co.compress(data) + co.flush()
        out = np.zeros(max(1, n), np.uint8)
        st = lib.bgzfdev_inflate_raw(comp, len(comp), out.ctypes.data_as(ctypes.c_void_p), n)
        if st == 2:
            n_declined += 1
            continue
        assert st == 0 and out[:n].tobytes() == data
        if comp and trial % 2:
            c = bytearray(comp)
            c[int(rng.integers(len(c)))] ^= 1 << int(rng.integers(8))
            st = lib.bgzfdev_inflate_raw(bytes(c), len(c), out.ctypes.data_as(ctypes.c_void_p), n)
            if st == 0:
                assert zlib.decompress(bytes(c), -15) == out[:n].tobytes()
    assert n_declined < 30


def test_warp_crc32_equals_zlib(lib):
    lib.bgzfdev_crc32_lanes.restype = ctypes.c_uint32
    rng = np.random.default_rng(4)
    for n in [0, 1, 2, 31, 32, 33, 63, 64, 65, 1000, 2047, 2048, 65279, 65280, 65535, 65536] + [int(x) for x in rng.integers(0, 65537, 40)]:
        data = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
        assert lib.bgzfdev_crc32_lanes(data, n) == (zlib.crc32(data) & 0xFFFFFFFF), n


@pytest.mark.parametrize("mode", ["se", "pe", "sc"])
@pytest.mark.parametrize("window_blocks", [3, 1 << 16])
def test_committed_bam_fixtures(lib, mode, window_blocks):
    """The block-parallel decoder against the committed fixtures of tests/make_bam_golden.py (arrays of the
    Python packing); ids of chromosomes outside the index are compared up to renaming, as in test_fastbam."""
    from test_fastbam import _canon_chrom
    want = np.load(os.path.join(H.GOLD, "bam_mixed_expected.npz"))
    idx = H.load_index("idx_rand_a.glb")
    wl = reads.Whitelist(os.path.join(H.GOLD, "bam_mixed_whitelist.txt")) if mode == "sc" else None
    rc, _, got = _decode(lib, os.path.join(H.GOLD, "bam_mixed_%s.bam" % mode), mode, reads.ChromMap(idx.chrom_keys), wl, 20, window_blocks)
    assert rc == 0 and len(got["start"]) == 600

    class _B:
        pass
    a, b = _B(), _B()
    a.n = b.n = 600
    a.chrom, b.chrom = want["%s_chrom" % mode], got["chrom"]
    n_index = len(idx.chrom_keys)
    assert np.array_equal(_canon_chrom([(a, False)], n_index, mode != "sc")[0], _canon_chrom([(b, False)], n_index, mode != "sc")[0])
    for k in ("start", "end", "mapq", "flag") + (("cell", "umi") if mode == "sc" else ()):
        assert np.array_equal(want["%s_%s" % (mode, k)], got[k]), k


def _split_blocks(raw):
    out, o = [], 0
    while o < len(raw):
        n = int.from_bytes(raw[o + 16:o + 18], "little") + 1
        out.append(raw[o:o + n])
        o += n
    return out


def test_header_over_many_blocks_empty_blocks_and_no_references(lib, tmp_path):
    """Layouts around the records: a header much longer than a block (3000 reference sequences), empty
    BGZF blocks in the middle of the file, a file without reference sequences (all reads unmapped)."""
    from bam_writer import _bgzf_block
    rng = np.random.default_rng(12)
    recs = [{"chrom": "contig_%04d" % int(rng.integers(3000)), "start": int(rng.integers(1, 50000)), "end": 0,
             "flag": int(rng.choice([0, 16, 1024]))} for _ in range(4000)]
    for r in recs:
        r["end"] = r["start"] + 76
    recs += [{"chrom": "contig_%04d" % i, "start": 5, "end": 90} for i in range(3000)]      # every contig in the header
    path = str(tmp_path / "many.bam")
    write_bam(path, recs, block=500)
    blocks = _split_blocks(open(path, "rb").read())
    with_empty = []
    for i, b in enumerate(blocks):
        with_empty.append(b)
        if i % 7 == 3:
            with_empty.append(_bgzf_block(b""))
    open(path, "wb").write(b"".join(with_empty))
    keys = ["contig_%04d" % i for i in range(0, 3000, 3)]
    want = _native(path, "se", reads.ChromMap(keys), None, 0)
    assert len(want["start"]) == 7000
    for wb in (1, 64, 1 << 16):
        rc, msg, got = _decode(lib, path, "se", reads.ChromMap(keys), None, 0, wb)
        assert rc == 0, (wb, msg)
        from test_fastbam import _canon_chrom

        class _B:
            pass
        a, b = _B(), _B()
        a.n = b.n = 7000
        a.chrom, b.chrom = want["chrom"], got["chrom"]
        assert np.array_equal(_canon_chrom([(a, False)], len(keys))[0], _canon_chrom([(b, False)], len(keys))[0])
        for k in ("start", "end", "mapq", "flag"):
            assert np.array_equal(want[k], got[k]), (k, wb)
    # no reference sequences at all
    path2 = str(tmp_path / "unaligned.bam")
    write_bam(path2, [{"chrom": None, "start": -1, "end": -1, "flag": 4 | (77 if i % 2 == 0 else 141)} for i in range(501)], block=333)
    want = _native(path2, "pe", reads.ChromMap(["1"]), None, 20)
    rc, _, got = _decode(lib, path2, "pe", reads.ChromMap(["1"]), None, 20, 2)
    assert rc == 0 and len(got["start"]) == 500
    for k in want:
        assert np.array_equal(want[k], got[k]), k


# ---- the whitelist hash table at the size of a 10x v2 whitelist (737 280 barcodes of 16 bases + "-1")

def wl_hash(bc):
    """bgzf_dev.h wl_hash restated over equal-length barcodes: uint8 array (n, length) -> uint64 (n,)."""
    h = np.full(len(bc), 0xcbf29ce484222325, np.uint64)
    for i in range(bc.shape[1]):
        h = (h ^ bc[:, i]) * np.uint64(0x100000001b3)
    h ^= h >> np.uint64(29)
    h *= np.uint64(0xbf58476d1ce4e5b9)
    return h ^ (h >> np.uint64(32))


def wl_table(hashes):
    """bam_orch.h set_whitelist: open addressing in id order.  (capacity, slot of every id)"""
    cap = 16
    while cap < 2 * len(hashes) + 2:
        cap <<= 1
    slot, at = [0] * cap, []
    for h in (hashes & np.uint64(cap - 1)).tolist():
        while slot[h]:
            h = (h + 1) & (cap - 1)
        slot[h] = len(at) + 1
        at.append(h)
    return cap, np.array(at), slot


def _barcodes(v):
    """16-base barcodes + '-1' of the 32-bit values v, as an uint8 array (n, 18)"""
    b = np.frombuffer(b"ACGT", np.uint8)[(v.astype(np.uint32)[:, None] >> (2 * np.arange(15, -1, -1, dtype=np.uint32))) & np.uint32(3)]
    return np.concatenate([b, np.tile(np.frombuffer(b"-1", np.uint8), (len(v), 1))], axis=1)


def _strings(a):
    return [bytes(x).decode() for x in a]


def _variants(s):
    """the prefixes and one-character extensions of a barcode that a lookup without the length test would confuse with it"""
    return [s[:-1], s[:16], s + "A"]


def tenx_whitelist(seed=3, n=737_280):
    """A whitelist of n barcodes and the barcodes a lookup can trip over: whitelisted ones whose probe chain wraps past
    the table's last slot, absent ones whose chain starts in that full run, one-base neighbours of whitelisted ones,
    and prefixes and extensions of whitelisted barcodes.  For six whitelisted barcodes a prefix or extension has the
    same home slot, so its probe chain passes the barcode and only the length test in wl_find tells them apart."""
    rng = np.random.default_rng(seed)
    n_tail, n_same = 4, 6
    v = np.unique(rng.integers(0, 1 << 32, n + 200_000, dtype=np.uint64))
    v = rng.permutation(v)[:n - n_tail - n_same]
    cap = 16
    while cap < 2 * n + 2:
        cap <<= 1
    m = np.uint64(cap - 1)
    tail, same = set(), set()                               # not yet whitelisted: home in the last two slots / shared with a variant
    while len(tail) < 2 * n_tail or len(same) < n_same:
        c = rng.integers(0, 1 << 32, 1 << 20, dtype=np.uint64)
        c = c[~np.isin(c, v)]
        b = _barcodes(c)
        home = wl_hash(b) & m
        tail |= set(c[home >= cap - 2].tolist())
        ext = np.concatenate([b, np.full((len(b), 1), ord("A"), np.uint8)], axis=1)
        hit = ((wl_hash(b[:, :17]) & m) == home) | ((wl_hash(b[:, :16]) & m) == home) | ((wl_hash(ext) & m) == home)
        same |= set(c[hit].tolist())
    same = sorted(same - tail)[:n_same]
    tail = sorted(tail)[:2 * n_tail]
    same_s = _strings(_barcodes(np.array(same, np.uint64)))
    wl = sorted(_strings(_barcodes(np.array(list(v) + tail[:n_tail] + same, np.uint64))))
    assert len(wl) == n
    absent_tail = _strings(_barcodes(np.array(tail[n_tail:], np.uint64)))
    a = np.frombuffer("".join(wl).encode(), np.uint8).reshape(len(wl), 18)
    cap_, at, slot = wl_table(wl_hash(a))
    assert cap_ == cap
    home = (wl_hash(a) & m).astype(np.int64)
    wrapped = [wl[i] for i in np.flatnonzero(at < home)]
    assert len(wrapped) >= 2 and all(slot[cap - 2:])        # chains run over the last slot
    wls = set(wl)
    shadow = []                                             # absent variants whose probe chain passes their barcode's slot
    for s in same_s:
        i = wl.index(s)
        for p in _variants(s):
            h = int(wl_hash(np.frombuffer(p.encode(), np.uint8)[None, :])[0] & m)
            while slot[h] and h != at[i]:
                h = (h + 1) & (cap - 1)
            if h == at[i] and p not in wls:
                shadow.append(p)
    assert len(shadow) >= n_same
    near = []
    for i in rng.integers(0, len(wl), 300).tolist():
        s, j = wl[i], int(rng.integers(16))
        c = s[:j] + "ACGT"[("ACGT".index(s[j]) + 1 + int(rng.integers(3))) % 4] + s[j + 1:]
        if c not in wls:
            near.append(c)
    part = []
    for s in [wl[i] for i in rng.integers(0, len(wl), 100).tolist()] + wrapped:
        part += [x for x in _variants(s) + [s + "1"] if x not in wls]
    return wl, {"wrapped": wrapped, "absent_tail": absent_tail, "near": near, "prefix_extension": part,
                "same_home": shadow + same_s}


def tenx_records(wl, groups, n, seed):
    """single-cell records whose CB tags cycle through whitelisted barcodes and every group of tenx_whitelist"""
    rng = np.random.default_rng(seed)
    kinds = [wl] * 5 + [groups[k] for k in ("wrapped", "absent_tail", "near", "prefix_extension", "same_home")]
    chroms = ["chr1", "chr2", "2", "chrX", "scaffold7"]
    recs = []
    for i in range(n):
        pool = kinds[i % len(kinds)]
        start = int(rng.integers(0, 150000))
        recs.append({"chrom": chroms[int(rng.integers(len(chroms)))], "start": start, "end": start + 60,
                     "flag": 16 * int(rng.integers(2)), "mapq": 60, "CB": pool[int(rng.integers(len(pool)))],
                     "UB": "".join("ACGT"[int(x)] for x in rng.integers(0, 4, 12)), "name": "r%d" % i})
    return recs


def test_wl_hash_restatement(lib):
    lib.bgzfdev_wl_hash.restype = ctypes.c_uint64
    lib.bgzfdev_wl_hash.argtypes = [ctypes.c_char_p, ctypes.c_uint32]
    rng = np.random.default_rng(8)
    for length in (0, 1, 2, 7, 8, 16, 18, 19, 40):
        a = rng.integers(0, 256, (64, length), dtype=np.uint8)
        a[:8] = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, (8, length))]
        want = [lib.bgzfdev_wl_hash(bytes(x), length) for x in a]
        assert wl_hash(a).tolist() == want, length


@pytest.fixture(scope="module")
def tenx():
    return tenx_whitelist()


@pytest.mark.parametrize("window_blocks", [1, 5])
def test_10x_whitelist_lookups(lib, tmp_path, tenx, window_blocks):
    """The block-parallel decoder's whitelist table at 737 280 barcodes against libtecbam and the dictionary lookup:
    probe chains that wrap past the last slot, absent barcodes that walk a full chain, one-base neighbours, prefixes
    and extensions of whitelisted barcodes, among them ones whose probe chain passes the barcode they extend."""
    wl_list, groups = tenx
    recs = tenx_records(wl_list, groups, 6000, 5)
    path = str(tmp_path / "x.bam")
    write_bam(path, recs, block=3000)
    wlf = tmp_path / "wl.txt"
    wlf.write_text("".join(w + "\n" for w in wl_list))
    wl = reads.Whitelist(str(wlf))
    idx = H.load_index("idx_rand_a.glb")
    want = _native(path, "sc", reads.ChromMap(idx.chrom_keys), wl, 20)
    rc, msg, got = _decode(lib, path, "sc", reads.ChromMap(idx.chrom_keys), wl, 20, window_blocks)
    assert rc == 0, msg
    for k in want:
        assert np.array_equal(want[k], got[k]), k
    ids = np.array([wl.barcode_to_id.get(r["CB"], reads.CELL_INVALID) for r in recs], np.uint32)
    assert np.array_equal(got["cell"], ids)
    n_group = {k: sum(r["CB"] in set(v) for r in recs) for k, v in groups.items()}
    assert min(n_group.values()) > 100 and (ids != reads.CELL_INVALID).sum() == sum(r["CB"] in wl.barcode_to_id for r in recs)
