"""Paired end by read name on the device (parse_bampe(pairing='name'), tec_bulk_begin(ctx, 2, qual), tec_bulk_push_named,
tec_bam_count mode 3; csrc/pair_name.cuh).  The oracle is the rule restated in tests/pair_name_oracle.collate_by_name
followed by the unchanged paired-end oracle: collate, then count as the reference counts adjacent pairs."""
import os
import random
import sys

import numpy as np
import pytest

import helpers as H
import te_counter_b200
from bam_writer import write_bam
from oracle import te_oracle_c
from oracle.ref_runner import CaptureLog
from pair_name_oracle import collate_by_name
from te_counter_b200 import _lib, bam, reads, synth_bam
from test_gpu_sharded_pe import _launch

pytestmark = pytest.mark.gpu
GLB = "idx_rand_a.glb"
EXTRA = "records were not paired by name"


@pytest.fixture(scope="module")
def engine():
    eng = _lib.Engine(0)
    eng.upload_index(H.load_index(GLB))
    yield eng
    eng.close()


def _pairable(records):
    """Golden paired-end records made pairable by name: pair i (records 2i, 2i+1) gets its own QNAME and the flags 0x1
    and 0x40 / 0x80; the secondary bit, which the bulk rules do not read, is cleared.  A trailing odd record is a read1
    without a mate."""
    return [dict(r, name="p%d" % (i // 2), flag=(r.get("flag", 0) & ~0x900) | (0x41 if i % 2 == 0 else 0x81))
            for i, r in enumerate(records)]


def _coordinate_sorted(records):
    """samtools sort order: by reference (unplaced records last), then start; ties keep file order"""
    order = {}
    for r in records:
        if r["chrom"] is not None:
            order.setdefault(r["chrom"], len(order))
    return sorted(records, key=lambda r: (r["chrom"] is None, order.get(r["chrom"], 0), r["start"]))


def _sorted_file(seed, n_pairs, path, block=3000):
    """Seeded coordinate-sorted paired-end file over the chromosomes of idx_rand_a: mates 50 to 400 bp apart, 5 % on
    another chromosome, and duplicates, QC fails, unmapped mates, low MAPQ, secondary and supplementary records,
    records without 0x1, lone mates and a name with two read1.  Returns the records in file order."""
    rnd = random.Random(seed)
    chroms = ["chrX", "chr2", "chr1", "chr9"]
    recs = []

    def rec(name, flag, chrom, start):
        extra = rnd.choice([0] * 30 + [0x10, 0x400, 0x200, 0x4, 0x100, 0x800])
        return {"name": name, "flag": flag | extra, "chrom": chrom, "start": start, "end": start + rnd.randrange(30, 150),
                "mapq": rnd.choice([255, 255, 60, 30, 10, 0])}

    for i in range(n_pairs):
        c1 = rnd.choice(chroms)
        s1 = rnd.randrange(0, 125000)
        c2, s2 = (rnd.choice(chroms), rnd.randrange(0, 125000)) if rnd.random() < 0.05 else (c1, s1 + rnd.randrange(50, 401))
        name = "NB5012:7:%d:%d" % (seed, i)
        kind = rnd.random()
        if kind < 0.01:
            recs.append(rec(name, 0x41, c1, s1))                      # a lone mate
        elif kind < 0.015:
            recs.append(rec(name, 0x40, c1, s1))                      # 0x1 clear
            recs.append(rec(name, 0x80, c2, s2))
        else:
            recs.append(rec(name, 0x41, c1, s1))
            recs.append(rec(name, 0x81, c2, s2))
            if kind > 0.995:
                recs.append(rec(name, 0x41, c2, s2 + 3))              # a second read1
    recs = _coordinate_sorted(recs)
    write_bam(path, recs, block=block)
    return recs


def _oracle(path, qual=20):
    """(counts, stats[7], excluded, no_mate) of the rule on the records of the file, read by bam.py"""
    idx = H.load_index(GLB)
    cm = reads.ChromMap(idx.chrom_keys)
    f = bam.AlignmentFile(path, "r")
    recs = [{"name": r.query_name, "flag": r.flag, "r": r} for r in f]
    f.close()
    col, excl, no_mate = collate_by_name(recs)
    rr = [x["r"] for x in col]
    cols = [[r.reference_start if r.reference_start is not None else -1 for r in rr],
            [r.reference_end if r.reference_end is not None else -1 for r in rr],
            [cm.bulk_id(r.reference_name) for r in rr], [r.mapping_quality for r in rr], [reads._flagbits(r) for r in rr]]
    oc = te_oracle_c.Index(idx.chrom_id, idx.L, idx.R, idx.ensg_id, idx.type_code, idx.n_chrom, idx.n_ensg, idx.bucket_size)
    counts, st = te_oracle_c.bulk_count(oc, True, qual, *cols)
    return counts, st, excl, no_mate


def _device(engine, path, window_blocks=65536):
    idx = H.load_index(GLB)
    engine.set_option("bam_window_blocks", window_blocks)
    try:
        d = engine.bam_open(path)
        d.bind(reads.ChromMap(idx.chrom_keys))
        engine.bulk_begin(True, 20, pairing="name")
        n = d.count(3, 20)
        d.close()
    finally:
        engine.set_option("bam_window_blocks", 65536)
    counts, st = engine.bulk_finish()
    return n, counts, st


def _named_columns(path):
    """the columns of reads.fill_bulk_named for the whole file"""
    idx = H.load_index(GLB)
    f = bam.AlignmentFile(path, "r")
    n = sum(1 for _ in f)
    f.close()
    b = reads.Batch(n + 1, named=True)
    f = bam.AlignmentFile(path, "r")
    reads.fill_bulk_named(b, f, reads.ChromMap(idx.chrom_keys))
    f.close()
    return b


def _push_named(engine, b, step):
    engine.bulk_begin(True, 20, pairing="name")
    for a in range(0, b.n, step):
        z = min(b.n, a + step)
        off = b.name_off[a:z + 1] - b.name_off[a]
        engine.bulk_push_named(z - a, b.start[a:z], b.end[a:z], b.chrom[a:z], b.mapq[a:z], b.flag[a:z], b.samflag[a:z], off,
                               b.names[b.name_off[a]:b.name_off[z]])
    return engine.bulk_finish()


@pytest.mark.parametrize("decoder", ["gpu", "python"])
@pytest.mark.parametrize("name", H.case_names("bulk_pe"))
def test_golden_cases_coordinate_sorted(monkeypatch, tmp_path, name, decoder):
    case = H.load_case(name)
    recs = _pairable(case["records"])
    if any(r["end"] <= r["start"] and not r.get("flag", 0) & 4 for r in recs):
        pytest.skip("case has zero-length alignments a file cannot carry")
    path = str(tmp_path / "x.bam")
    write_bam(path, _coordinate_sorted(recs), block=500)
    monkeypatch.setitem(sys.modules, "pysam", None)
    monkeypatch.setenv("TEC_BAM_DECODER", decoder)
    mte = te_counter_b200.measureTE("test", case["qual"], device=0)
    mte.bind_genome(H.GOLD + "/" + case["glb"])
    mte.load_genome()
    log = CaptureLog()
    res = mte.parse_bampe(path, log=log, pairing="name")
    assert res == case["expected"]["result"] and mte.total_reads == case["expected"]["total_reads"]
    lines = [m for _, m in log.lines]
    assert [m for m in lines if EXTRA not in m] == [m for m in case["expected"]["log"] if not m.startswith("Saved")]
    no_mate = len(recs) % 2
    assert "%d records were not paired by name: 0 not primary or without exactly one mate flag, %d without a mate" % (no_mate, no_mate) in lines
    out = tmp_path / "o.tsv"
    mte.save_result_bulk(res, str(out), log=log)
    assert out.read_text() == case["expected"]["tsv"]


@pytest.mark.parametrize("seed", [1, 2])
def test_sorted_files_against_the_oracle(engine, tmp_path, seed):
    path = str(tmp_path / "s.bam")
    recs = _sorted_file(seed, 6000, path)
    o_counts, o_st, excl, no_mate = _oracle(path)
    assert excl > 0 and no_mate > 0
    for wb in (1, 2, 7, 65536):
        n, counts, st = _device(engine, path, wb)
        assert n == len(recs)
        assert np.array_equal(counts, o_counts), wb
        assert np.array_equal(st[:7], o_st), wb
        assert st[_lib.BS_NO_MATE] == excl + no_mate and engine.get_info("bulk_name_excluded") == excl
        if wb == 1:
            assert engine.get_info("bulk_name_pending_peak") > 0


def test_synth_bam_sorted_against_the_oracle(engine, tmp_path):
    path = str(tmp_path / "synth.bam")
    synth_bam.write(path, 60000, "pe", sorted_pe=True, seed=7, procs=2)
    o_counts, o_st, excl, no_mate = _oracle(path)
    n, counts, st = _device(engine, path, 4)
    assert n == 60000 and np.array_equal(counts, o_counts) and np.array_equal(st[:7], o_st)
    assert st[_lib.BS_NO_MATE] == excl + no_mate


def test_device_host_and_direct_pushes_agree(engine, monkeypatch, tmp_path):
    path = str(tmp_path / "s.bam")
    _sorted_file(3, 3000, path)
    _, counts, st = _device(engine, path, 3)
    b = _named_columns(path)
    for step in (1, 777, b.n):
        c2, s2 = _push_named(engine, b, step)
        assert np.array_equal(c2, counts) and np.array_equal(s2, st), step
    monkeypatch.setitem(sys.modules, "pysam", None)
    monkeypatch.setenv("TEC_BAM_DECODER", "python")
    mte = te_counter_b200.measureTE("test", 20, device=0)
    mte.bind_genome(H.GOLD + "/" + GLB)
    mte.load_genome()
    res = mte.parse_bampe(path, log=CaptureLog(), pairing="name")
    assert list(res.values()) == counts.tolist() and mte.total_reads == st[_lib.BS_UNITS] + 1


def test_worst_order_all_read1_then_all_read2(engine):
    n_pairs = 500000
    rnd = np.random.default_rng(4)
    names = [b"w%07d" % i for i in range(n_pairs)]
    n = 2 * n_pairs
    b = reads.Batch(n, named=True)
    b.n = n
    b.start[:] = rnd.integers(0, 120000, n)
    b.end[:] = b.start + 100
    b.chrom[:] = rnd.integers(0, 3, n)
    b.mapq[:] = 60
    b.flag[:] = 0
    b.samflag[:n_pairs] = 0x41
    b.samflag[n_pairs:] = 0x81
    perm = rnd.permutation(n_pairs)
    order = names + [names[i] for i in perm]
    np.cumsum([len(x) for x in order], out=b.name_off[1:n + 1])
    b.names = b"".join(order)
    counts, st = _push_named(engine, b, 100000)                     # the read1 end with a batch: all of them wait at once
    assert st[_lib.BS_UNITS] == n_pairs and st[_lib.BS_NO_MATE] == 0
    assert engine.get_info("bulk_name_pending_peak") == n_pairs
    # the same pairs, collated, through index pairing
    start, chrom = np.empty(n, np.int32), np.empty(n, np.uint16)
    start[0::2], start[1::2] = b.start[:n_pairs][perm], b.start[n_pairs:]
    chrom[0::2], chrom[1::2] = b.chrom[:n_pairs][perm], b.chrom[n_pairs:]
    engine.bulk_begin(True, 20)
    engine.bulk_push(n, start, start + 100, chrom, np.full(n, 60, np.uint8), np.zeros(n, np.uint8))
    c2, s2 = engine.bulk_finish()
    assert np.array_equal(counts, c2) and np.array_equal(st[:7], s2[:7])


def test_collated_file_same_under_both_pairings(monkeypatch, tmp_path):
    case = H.load_case("bulk_pe_rand_b")
    path = str(tmp_path / "c.bam")
    write_bam(path, _pairable(case["records"]))
    monkeypatch.setenv("TEC_BAM_DECODER", "gpu")
    mte = te_counter_b200.measureTE("test", 20, device=0)
    mte.bind_genome(H.GOLD + "/" + case["glb"])
    mte.load_genome()
    by_index = mte.parse_bampe(path, log=CaptureLog())
    t_index = mte.total_reads
    by_name = mte.parse_bampe(path, log=CaptureLog(), pairing="name")
    assert by_index == by_name == case["expected"]["result"] and mte.total_reads == t_index
    with pytest.raises(ValueError):
        mte.parse_bampe(path, log=CaptureLog(), pairing="position")


def test_abi_edges(engine, tmp_path):
    path = str(tmp_path / "s.bam")
    _sorted_file(5, 500, path)
    engine.bulk_begin(True, 20, pairing="name")
    one = np.zeros(2, np.int32)
    with pytest.raises(_lib.TecError) as e:
        engine.bulk_push(2, one, one, one.astype(np.uint16), one.astype(np.uint8), one.astype(np.uint8))
    assert e.value.status == -3
    d = engine.bam_open(path)
    d.bind(reads.ChromMap(H.load_index(GLB).chrom_keys))
    with pytest.raises(_lib.TecError) as e:
        d.count(1, 20)                                              # index pairing in a name-pairing run
    assert e.value.status == -3
    with pytest.raises(_lib.TecError) as e:
        d.count_range(3, 20, 0, os.path.getsize(path))
    assert e.value.status == -2
    engine.bulk_begin(True, 20)
    with pytest.raises(_lib.TecError) as e:
        d.count(3, 20)                                              # mode 3 needs the name-pairing begin
    assert e.value.status == -3
    d.close()
    # a new begin clears the pending set: read1s of one run never meet read2s of the next
    b = reads.Batch(4, named=True)
    b.n = 2
    b.start[:2], b.end[:2], b.chrom[:2], b.mapq[:2], b.flag[:2] = 100, 200, 0, 60, 0
    b.samflag[:2] = 0x41
    b.name_off[:3] = [0, 1, 2]
    b.names = b"ab"
    engine.bulk_begin(True, 20, pairing="name")
    engine.bulk_push_named(2, b.start[:2], b.end[:2], b.chrom[:2], b.mapq[:2], b.flag[:2], b.samflag[:2], b.name_off[:3], b.names)
    assert engine.get_info("bulk_name_pending_peak") == 2
    b.samflag[:2] = 0x81
    _, st = _push_named(engine, b, 2)
    assert st[_lib.BS_UNITS] == 0 and st[_lib.BS_NO_MATE] == 2


def test_sharded_cli_two_ranks_same_tsv(tmp_path):
    path = str(tmp_path / "s.bam")
    _sorted_file(6, 20000, path, block=20000)
    glb = os.path.join(H.GOLD, GLB)
    one = str(tmp_path / "one.tsv")
    rc, log = _launch(1, 0, ["--glb", glb, "--bam", path, "--mode", "pe", "--pairing", "name", "-o", one])
    assert rc == 0, log[-3000:]
    assert EXTRA in log
    two = str(tmp_path / "two.tsv")
    rc, log = _launch(2, 29672, ["--glb", glb, "--bam", path, "--mode", "pe", "--pairing", "name", "-o", two])
    assert rc == 0, log[-3000:]
    assert open(two, "rb").read() == open(one, "rb").read()
