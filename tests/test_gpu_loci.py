"""Counts per index row on the device (tec_set_option "bulk_loci", tec_bulk_loci; measureTE(..., loci=True)).
The device rows equal the C / Python oracle for single end, paired end by index and by name, through every push and the
device decoder; loci on leaves the per-name counts and statistics alone, loci off changes nothing; ranks in turn sum to
the whole file; the sharded CLI writes the same locus TSV at 1, 2 and 3 ranks; the ABI refuses out-of-order calls."""
import os
import sys

import numpy as np
import pytest

import helpers as H
import te_counter_b200
from bam_writer import write_bam
import locus_oracle as LO
from oracle.ref_runner import CaptureLog
from pair_name_oracle import collate_by_name
from te_counter_b200 import _lib, bam, reads, shard, synth
from test_gpu_pair_name import GLB, _named_columns, _sorted_file
from test_gpu_sharded_file import _records
from test_gpu_sharded_pe import _launch

pytestmark = pytest.mark.gpu
COLS = ("start", "end", "chrom", "mapq", "flag")


@pytest.fixture(scope="module")
def engine():
    eng = _lib.Engine(0)
    yield eng
    eng.close()


def oracle_rows(idx, paired, qual, cols, strand=False):
    """(counts, stats[7], loci in the device's row order)"""
    c, st, loci = LO.c_bulk_count_loci(LO.CIndex(idx), paired, qual, *[cols[k] for k in COLS],
                                       strand_code=idx.strand_code if strand else None)
    return c, st, loci[idx.sorted_layout()["order"]]


def run(engine, paired, cols, loci=True, strand=False, push="host", pairing="index"):
    engine.set_option("bulk_loci", 1 if loci else 0)
    engine.set_option("bulk_strand", 1 if strand else 0)
    try:
        engine.bulk_begin(paired, 20, pairing=pairing)
        n = len(cols["start"])
        if push == "host":
            engine.bulk_push(n, *[cols[k] for k in COLS])
        else:
            import torch
            t = [torch.from_numpy(np.ascontiguousarray(cols[k])).cuda() for k in COLS]
            torch.cuda.synchronize()
            engine.bulk_push_dev(n, *[x.data_ptr() for x in t])
            engine.sync()
        counts, st = engine.bulk_finish()
        return counts, st, (engine.bulk_loci() if loci else None)
    finally:
        engine.set_option("bulk_loci", 0)
        engine.set_option("bulk_strand", 0)


@pytest.mark.parametrize("push", ["host", "dev"])
@pytest.mark.parametrize("strand", [False, True])
@pytest.mark.parametrize("paired", [False, True])
def test_device_rows_equal_the_oracle(engine, paired, strand, push):
    idx = synth.synth_index(61, n_te=30000, n_exon=9000, n_gene=600, chrom_len=3_000_000, n_chrom=3)
    r = synth.synth_bulk_reads(62, idx, 80000, paired=paired, edge_frac=0.1)
    engine.upload_index(idx)
    counts, st, loci = run(engine, paired, r, strand=strand, push=push)
    oc, ost, ol = oracle_rows(idx, paired, 20, r, strand)
    assert np.array_equal(counts, oc) and np.array_equal(st[:7], ost)
    assert np.array_equal(loci, ol)
    per_name = np.bincount(idx.sorted_layout()["ensg_id"], weights=loci, minlength=idx.n_ensg)
    assert (per_name >= counts).all() and loci.sum() > 1000


def test_pileup_beyond_the_register_rows(engine):
    """more hit rows than BULK_LOCI_REG: the second walk"""
    n = 40
    from te_counter_b200.index import GlbIndex
    idx = GlbIndex(["1"], np.zeros(n, np.int32), np.full(n, 1000, np.int32) + np.arange(n, dtype=np.int32),
                   np.full(n, 5000, np.int32), np.arange(n, dtype=np.int32) % 30, np.full(n, 2, np.uint8),
                   np.zeros(n, np.uint8), ["e%02d" % i for i in range(30)])
    engine.upload_index(idx)
    r = {"start": np.array([2000, 1010, 900, 1003], np.int32), "end": np.array([2100, 1011, 1001, 1004], np.int32),
         "chrom": np.zeros(4, np.uint16), "mapq": np.full(4, 60, np.uint8), "flag": np.zeros(4, np.uint8)}
    counts, st, loci = run(engine, False, r)
    oc, ost, ol = oracle_rows(idx, False, 20, r)
    assert np.array_equal(counts, oc) and np.array_equal(loci, ol) and loci.max() == 4


@pytest.mark.parametrize("algo", [-1, 0, 2])
@pytest.mark.parametrize("paired", [False, True])
def test_loci_on_leaves_names_and_statistics_alone(engine, paired, algo):
    idx = synth.synth_index(63, n_te=30000, n_exon=9000, n_gene=600, chrom_len=3_000_000, n_chrom=3)
    r = synth.synth_bulk_reads(64, idx, 80000, paired=paired, edge_frac=0.05)
    engine.set_option("bulk_algo", algo)
    try:
        engine.upload_index(idx)
        off = run(engine, paired, r, loci=False)
        on = run(engine, paired, r, loci=True)
    finally:
        engine.set_option("bulk_algo", -1)
    assert np.array_equal(off[0], on[0]) and np.array_equal(off[1], on[1])


def test_loci_off_changes_nothing(engine):
    """an engine that had the option on and off again launches and counts exactly as one that never saw it"""
    idx = synth.synth_index(65, n_te=20000, n_exon=6000, n_gene=400, chrom_len=2_000_000, n_chrom=2)
    r = synth.synth_bulk_reads(66, idx, 50000, paired=True)
    fresh = _lib.Engine(0)
    try:
        out = []
        for e in (fresh, engine):
            e.upload_index(idx)
            if e is engine:
                run(e, True, r, loci=True)                      # a run with loci, then the option off
            n0 = e.launch_count()
            e.bulk_begin(True, 20)
            e.bulk_push(len(r["start"]), *[r[k] for k in COLS])
            counts, st = e.bulk_finish()
            out.append((e.launch_count() - n0, counts, st, e.get_info("bulk_counter_words")))
            with pytest.raises(_lib.TecError) as ei:
                e.bulk_loci()
            assert ei.value.status == -3
        assert out[0][0] == out[1][0] and out[0][3] == out[1][3] == idx.n_ensg + _lib.BULK_NSTATS
        assert np.array_equal(out[0][1], out[1][1]) and np.array_equal(out[0][2], out[1][2])
    finally:
        fresh.close()


def _collated_columns(path):
    """the name-collated pairs of the file as columns (tests/pair_name_oracle.py)"""
    idx = H.load_index(GLB)
    cm = reads.ChromMap(idx.chrom_keys)
    f = bam.AlignmentFile(path, "r")
    recs = [{"name": r.query_name, "flag": r.flag, "r": r} for r in f]
    f.close()
    rr = [x["r"] for x in collate_by_name(recs)[0]]
    return {"start": np.array([r.reference_start if r.reference_start is not None else -1 for r in rr], np.int32),
            "end": np.array([r.reference_end if r.reference_end is not None else -1 for r in rr], np.int32),
            "chrom": np.array([cm.bulk_id(r.reference_name) for r in rr], np.uint16),
            "mapq": np.array([r.mapping_quality for r in rr], np.uint8),
            "flag": np.array([reads._flagbits(r) for r in rr], np.uint8)}


def test_pairs_by_name(engine, tmp_path):
    """device decoder (mode 3) and tec_bulk_push_named against the oracle on the name-collated pairs"""
    idx = H.load_index(GLB)
    engine.upload_index(idx)
    path = str(tmp_path / "s.bam")
    _sorted_file(67, 6000, path, block=1500)
    oc, ost, ol = oracle_rows(idx, True, 20, _collated_columns(path))
    engine.set_option("bulk_loci", 1)
    try:
        d = engine.bam_open(path)
        d.bind(reads.ChromMap(idx.chrom_keys))
        engine.bulk_begin(True, 20, pairing="name")
        d.count(3, 20)
        d.close()
        loci = engine.bulk_loci()                             # flushes the rows still waiting, as bulk_finish does
        counts, st = engine.bulk_finish()
        assert np.array_equal(counts, oc) and np.array_equal(st[:7], ost) and np.array_equal(loci, ol)
        b = _named_columns(path)
        engine.bulk_begin(True, 20, pairing="name")
        for a in range(0, b.n, 777):
            z = min(b.n, a + 777)
            engine.bulk_push_named(z - a, b.start[a:z], b.end[a:z], b.chrom[a:z], b.mapq[a:z], b.flag[a:z], b.samflag[a:z],
                                   b.name_off[a:z + 1] - b.name_off[a], b.names[b.name_off[a]:b.name_off[z]])
        counts, st = engine.bulk_finish()
        assert np.array_equal(counts, oc) and np.array_equal(engine.bulk_loci(), ol)
    finally:
        engine.set_option("bulk_loci", 0)


@pytest.mark.parametrize("decoder", ["gpu", "python"])
@pytest.mark.parametrize("name", H.case_names("bulk"))
def test_golden_files_through_the_mirror(monkeypatch, tmp_path, name, decoder):
    """bam_writer files -> parse_bamse / parse_bampe(loci=True): the reference's result and TSV, rows equal to the oracle"""
    case = H.load_case(name)
    recs = [dict(r, name=r.get("name", "r%d" % i)) for i, r in enumerate(case["records"])]
    if any(r["end"] <= r["start"] and not r.get("flag", 0) & 4 for r in recs):
        pytest.skip("case has zero-length alignments a file cannot carry")
    path = str(tmp_path / "x.bam")
    write_bam(path, recs)
    monkeypatch.setitem(sys.modules, "pysam", None)
    monkeypatch.setenv("TEC_BAM_DECODER", decoder)
    mte = te_counter_b200.measureTE("test", case["qual"], device=0)
    mte.bind_genome(H.GOLD + "/" + case["glb"])
    mte.load_genome()
    log = CaptureLog()
    res = (mte.parse_bampe if case["paired"] else mte.parse_bamse)(path, log=log, loci=True)
    assert res == case["expected"]["result"]
    out = tmp_path / "o.tsv"
    mte.save_result_bulk(res, str(out), log=log)
    assert out.read_text() == case["expected"]["tsv"]
    idx = mte.genome
    _, _, want = LO.bulk_count_loci(H.oracle_index(idx), case["paired"], case["qual"],
                                    *[v.tolist() for v in H.pack_bulk(case, idx).values()])
    assert mte.locus_counts.tolist() == want
    if name == "bulk_se_appendixA":
        assert want == [3, 1, 1, 1, 0]
    mte.save_result_loci(str(tmp_path / "l.tsv"), log=log)
    assert len((tmp_path / "l.tsv").read_bytes().splitlines()) == idx.n_features + 1
    res2 = (mte.parse_bampe if case["paired"] else mte.parse_bamse)(path, log=log)
    assert res2 == res and mte.locus_counts is None


def _open(eng, path, idx):
    d = eng.bam_open(path)
    d.bind(reads.ChromMap(idx.chrom_keys))
    return d


def _whole(engine, path, idx, mode):
    engine.bulk_begin(mode != 0, 20, pairing="name" if mode == 4 else "index")
    d = _open(engine, path, idx)
    d.count(3 if mode == 4 else mode, 20)
    d.close()
    return engine.bulk_loci(), engine.bulk_finish()


@pytest.mark.parametrize("mode", [0, 1, 4])
def test_ranks_in_turn_sum_to_the_whole_file(tmp_path, mode):
    import torch
    idx = H.load_index(GLB)
    path = str(tmp_path / "x.bam")
    if mode == 4:
        _sorted_file(68, 3000, path, block=1500)
    else:
        write_bam(path, _records(6001, 69, False)[0], block=3000)
    size = os.path.getsize(path)
    worlds = (1, 2, 3, 8) if mode == 4 else (1, 2, 3, 37)          # the name exchange takes 1..8 ranks
    engs = []
    try:
        for _ in range(worlds[-1]):
            e = _lib.Engine(0)
            e.upload_index(idx)
            e.set_option("bulk_loci", 1)
            engs.append(e)
        whole_loci, whole = _whole(engs[0], path, idx, mode)
        assert whole_loci.sum() > 0
        for world in worlds:
            loci, counts, stats = 0, 0, 0
            if mode == 1:
                infos = []
                for r in range(world):
                    engs[r].bulk_begin(True, 20)
                    d = _open(engs[r], path, idx)
                    infos.append(d.count_range(1, 20, *shard.byte_range(size, r, world)))
                    d.close()
                plan = shard.pair_plan(infos)
            parts = []
            for r in range(world):
                e = engs[r]
                e.bulk_begin(mode != 0, 20, pairing="name" if mode == 4 else "index")
                d = _open(e, path, idx)
                d.count_range(mode, 20, *shard.byte_range(size, r, world))
                if mode == 1:
                    with pytest.raises(_lib.TecError) as ei:
                        e.bulk_loci()                              # the bank is not chosen yet
                    assert ei.value.status == -3
                    e.bulk_keep_bank(plan[r]["bank"])
                    if plan[r]["border"] is not None:
                        c = d.pair_columns(*plan[r]["border"], 20)
                        e.bulk_push(2, c["start"], c["end"], c["chrom"], c["mapq"], c["flag"])
                d.close()
                if mode == 4:
                    with pytest.raises(_lib.TecError) as ei:
                        e.bulk_loci()                              # rows wait for the partition
                    assert ei.value.status == -3
                    send, ptr = e.bulk_name_partition_dev(world)
                    src = torch.as_tensor(_DevBytes(ptr, sum(send) * 32), device="cuda:0") if sum(send) else \
                        torch.empty(0, dtype=torch.uint8, device="cuda:0")
                    parts.append(list(torch.split(src.clone(), [x * 32 for x in send])))
                else:
                    c_r, s_r = e.bulk_finish()
                    loci, counts, stats = loci + e.bulk_loci(), counts + c_r, stats + s_r
            if mode == 4:
                torch.cuda.synchronize()
                for o in range(world):
                    dst = torch.cat([parts[r][o] for r in range(world)])
                    torch.cuda.synchronize()
                    engs[o].bulk_name_import_dev(dst.numel() // 32, dst.data_ptr() if dst.numel() else None)
                    c_r, s_r = engs[o].bulk_finish()
                    loci, counts, stats = loci + engs[o].bulk_loci(), counts + c_r, stats + s_r
            assert np.array_equal(loci, whole_loci), world
            assert np.array_equal(counts, whole[0]) and np.array_equal(stats, whole[1]), world
    finally:
        for e in engs:
            e.close()


class _DevBytes:
    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "|u1", "data": (ptr, False), "version": 2}


def test_library_allreduce_carries_the_rows(engine, tmp_path):
    """tec_bulk_allreduce on a one-rank communicator sums the whole block: the rows come back unchanged"""
    idx = synth.synth_index(70, n_te=20000, n_exon=6000, n_gene=400, chrom_len=2_000_000, n_chrom=2)
    r = synth.synth_bulk_reads(71, idx, 40000, paired=False)
    e = _lib.Engine(0)
    try:
        e.upload_index(idx)
        e.comm_init(e.comm_unique_id(), 0, 1)
        e.set_option("bulk_loci", 1)
        e.bulk_begin(False, 20)
        assert e.get_info("bulk_counter_words") == idx.n_ensg + _lib.BULK_NSTATS + idx.n_features
        e.bulk_push(len(r["start"]), *[r[k] for k in COLS])
        e.bulk_allreduce()
        _, _, ol = oracle_rows(idx, False, 20, r)
        assert np.array_equal(e.bulk_loci(), ol)
    finally:
        e.close()


@pytest.mark.parametrize("mode,pairing,port", [("se", "index", 29710), ("pe", "index", 29720), ("pe", "name", 29730)])
def test_sharded_cli_writes_the_same_locus_tsv(tmp_path, mode, pairing, port):
    glb = os.path.join(H.GOLD, GLB)
    bam_path = str(tmp_path / "in.bam")
    if pairing == "name":
        _sorted_file(72, 8000, bam_path, block=1500)
    else:
        write_bam(bam_path, _records(30001, 73, False)[0], block=20000)
    args = ["--glb", glb, "--bam", bam_path, "--mode", mode, "--pairing", pairing]
    one = str(tmp_path / "one.loci.tsv")
    rc, log = _launch(1, 0, args + ["--loci", one, "-o", str(tmp_path / "one.tsv")])
    assert rc == 0, log[-3000:]
    lines = open(one, "rb").read().splitlines()
    assert lines[0] == b"ensg\tchrom\tleft\tright\tstrand\tcount\tcpm" and len(lines) == H.load_index(GLB).n_features + 1
    assert sum(int(x.split(b"\t")[5]) for x in lines[1:]) > 0
    for world in ((2, 3) if (mode, pairing) == ("pe", "index") else (2,)):
        out = str(tmp_path / ("w%d.loci.tsv" % world))
        rc, log = _launch(world, port + world, args + ["--loci", out, "-o", str(tmp_path / "w.tsv")])
        assert rc == 0, log[-3000:]
        assert "decoded by this rank" in log
        assert open(out, "rb").read() == open(one, "rb").read()
        assert open(str(tmp_path / "w.tsv"), "rb").read() == open(str(tmp_path / "one.tsv"), "rb").read()


def test_state_errors(engine):
    idx = synth.synth_index(74, n_te=2000, n_exon=600, n_gene=40, chrom_len=500_000, n_chrom=1)
    engine.upload_index(idx)
    with pytest.raises(_lib.TecError) as ei:
        engine.bulk_loci()                                    # no run begun
    assert ei.value.status == -3
    engine.bulk_begin(False, 20)
    with pytest.raises(_lib.TecError) as ei:
        engine.bulk_loci()                                    # begun without the option
    assert ei.value.status == -3
    with pytest.raises(_lib.TecError):
        engine.set_option("bulk_loci", 2)
    engine.set_option("bulk_loci", 1)
    engine.bulk_begin(False, 20)
    engine.set_option("bulk_loci", 0)                         # read at the begin: this run keeps its rows
    assert engine.bulk_loci().sum() == 0 and len(engine.bulk_loci()) == idx.n_features
