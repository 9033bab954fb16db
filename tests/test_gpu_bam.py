"""The device BAM decoder (tec_bam_*: BGZF inflate, record split and packing in CUDA kernels, one
thread per BGZF block) against the host decoder libtecbam on the same files -- identical counts and
statistics out of the same engine -- and golden cases file -> TSV with TEC_BAM_DECODER=gpu."""
import sys

import numpy as np
import pytest

import helpers as H
from bam_writer import write_bam
from oracle.ref_runner import CaptureLog
import te_counter_b200
from te_counter_b200 import _lib, fastbam, reads
from test_fastbam import _mixed_records

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    eng = _lib.Engine(0)
    yield eng
    eng.close()


def _host_run(eng, path, mode, idx, wl, qual):
    f = fastbam.NativeBam(path, threads=2)
    f.bind(reads.ChromMap(idx.chrom_keys), wl)
    b = reads.Batch(1 << 14, sc=mode == "sc", alloc=eng.pinned)
    if mode == "sc":
        eng.sc_begin(qual, True, len(wl))
    else:
        eng.bulk_begin(mode == "pe", qual)
    more = True
    while more:
        if mode == "sc":
            more = f.fill_sc(b, qual)
            eng.sc_push(b.n, b.start, b.end, b.chrom, b.mapq, b.flag, b.cell, b.umi)
        else:
            more = f.fill_bulk(b, mode == "pe", qual)
            eng.bulk_push(b.n, b.start, b.end, b.chrom, b.mapq, b.flag)
    f.close()
    return _finish(eng, mode)


def _finish(eng, mode):
    if mode == "sc":
        nt, nh = eng.sc_finalize(10 ** 7, 30, 1000)
        return [np.asarray(a).copy() for a in eng.sc_fetch(nt, nh)]
    counts, st = eng.bulk_finish()
    return [counts.copy(), st.copy()]


def _device_run(eng, path, mode, idx, wl, qual):
    d = eng.bam_open(path)
    d.bind(reads.ChromMap(idx.chrom_keys), wl)
    if mode == "sc":
        eng.sc_begin(qual, True, len(wl))
    else:
        eng.bulk_begin(mode == "pe", qual)
    n = d.count({"se": 0, "pe": 1, "sc": 2}[mode], qual)
    info = d.info()
    d.close()
    return n, info, _finish(eng, mode)


@pytest.mark.parametrize("mode", ["se", "pe", "sc"])
@pytest.mark.parametrize("block,window_blocks", [(3000, 32768), (700, 5), (65000, 1), (64, 13)])
def test_device_decoder_equals_host_decoder(engine, tmp_path, mode, block, window_blocks):
    recs, wl_list = _mixed_records(5000 + (mode == "pe"), 31 + block, mode == "sc")
    path = str(tmp_path / "x.bam")
    write_bam(path, recs, block=block)
    idx = H.load_index("idx_rand_a.glb")
    engine.upload_index(idx)
    wl = None
    if mode == "sc":
        wlf = tmp_path / "wl.txt"
        wlf.write_text("".join(w + "\n" for w in wl_list))
        wl = reads.Whitelist(str(wlf))
    want = _host_run(engine, path, mode, idx, wl, 20)
    engine.set_option("bam_window_blocks", window_blocks)
    try:
        n, info, got = _device_run(engine, path, mode, idx, wl, 20)
    finally:
        engine.set_option("bam_window_blocks", 32768)
    assert n == 5000 and info["host_inflated_blocks"] == 0
    assert len(want) == len(got)
    for a, b in zip(want, got):
        assert np.array_equal(a, b)


@pytest.mark.parametrize("name", ["bulk_pe_rand_b", "bulk_se_rand_b", "bulk_pe_odd"])
def test_bulk_golden_from_file_on_the_device(monkeypatch, tmp_path, name):
    case = H.load_case(name)
    recs = [dict(r, name=r.get("name", "r%d" % i)) for i, r in enumerate(case["records"])]
    if any(r["end"] <= r["start"] and not r.get("flag", 0) & 4 for r in recs):
        pytest.skip("case has zero-length alignments a file cannot carry")
    path = str(tmp_path / "x.bam")
    write_bam(path, recs)
    monkeypatch.setitem(sys.modules, "pysam", None)
    monkeypatch.setenv("TEC_BAM_DECODER", "gpu")
    mte = te_counter_b200.measureTE("test", case["qual"], device=0)
    mte.bind_genome(H.GOLD + "/" + case["glb"])
    mte.load_genome()
    log = CaptureLog()
    res = (mte.parse_bampe if case["paired"] else mte.parse_bamse)(path, strand=False, log=log)
    assert res == case["expected"]["result"] and mte.total_reads == case["expected"]["total_reads"]
    out = tmp_path / "o.tsv"
    mte.save_result_bulk(res, str(out), log=log)
    assert out.read_text() == case["expected"]["tsv"]


@pytest.mark.parametrize("name", ["sc_appendixA", "sc_rand_det_strand", "sc_rand_amb_bundles"])
def test_sc_golden_from_file_on_the_device(monkeypatch, tmp_path, name):
    case = H.load_case(name)
    path = str(tmp_path / "x.bam")
    write_bam(path, [dict(r, name=r.get("name", "r%d" % i)) for i, r in enumerate(case["records"])])
    wl = tmp_path / "wl.txt"
    wl.write_text("".join(w + "\n" for w in case["whitelist"]))
    monkeypatch.setitem(sys.modules, "pysam", None)
    monkeypatch.setenv("TEC_BAM_DECODER", "gpu")
    mte = te_counter_b200.measureTE("test", case["qual"], device=0)
    mte.bind_genome(H.GOLD + "/" + case["glb"])
    log = CaptureLog()
    res = mte.sc_parse_bamse(path, UMIS=True, whitelistfilename=str(wl), strand=case["strand"], log=log, label="l",
                             maxcells=case["maxcells"], _bundle_keys=case["bundle_keys"], _pad=case["pad"])
    assert {k: v for k, v in dict(res).items() if v} == case["expected"]["result"]
    out = tmp_path / "o.tsv"
    mte.sc_save_result(res, str(out), maxcells=case["maxcells"], log=log)
    assert out.read_text() == case["expected"]["tsv"]


def test_device_decoder_errors(engine, tmp_path):
    idx = H.load_index("idx_toy.glb")
    engine.upload_index(idx)
    ok = {"chrom": "chr1", "start": 1600, "end": 1650, "CB": "AAAA", "UB": "ACGT"}
    wlf = tmp_path / "wl.txt"
    wlf.write_text("AAAA\n")
    wl = reads.Whitelist(str(wlf))
    path = str(tmp_path / "x.bam")
    for bad, exc in ((dict(ok, CB=None), AssertionError), (dict(ok, UB=None), AssertionError), (dict(ok, UB="ACGX"), ValueError),
                     (dict(ok, end=1600), TypeError), (dict(ok, chrom="HLA:A"), ValueError)):
        write_bam(path, [ok] * 7 + [bad] + [ok] * 5, block=300)
        d = engine.bam_open(path)
        d.bind(reads.ChromMap(idx.chrom_keys), wl)
        engine.sc_begin(20, False, 1)
        with pytest.raises(exc):
            d.count(2, 20)
        d.close()
    write_bam(path, [dict(ok, end=1600)], block=300)
    d = engine.bam_open(path)
    d.bind(reads.ChromMap(idx.chrom_keys))
    engine.bulk_begin(False, 20)
    with pytest.raises(TypeError):
        d.count(0, 20)
    with pytest.raises(_lib.TecError):
        d.count(1, 20)                                       # the running count is single end
    d.close()
    # damaged file
    recs = [{"chrom": "chr1", "start": 100 + i, "end": 150 + i} for i in range(2000)]
    write_bam(path, recs, block=20000)
    raw = bytearray(open(path, "rb").read())
    raw[len(raw) // 2] ^= 0x55
    open(path, "wb").write(bytes(raw))
    d = engine.bam_open(path)
    d.bind(reads.ChromMap(idx.chrom_keys))
    engine.bulk_begin(False, 20)
    with pytest.raises(ValueError):
        d.count(0, 20)
    d.close()
    sam = tmp_path / "x.sam"
    sam.write_text("@HD\tVN:1.6\n")
    with pytest.raises(_lib.BamUnsupported):
        engine.bam_open(str(sam))


@pytest.mark.parametrize("name", ["htslib_eof_marker", "empty_blocks_inside", "stored_blocks", "tiny_fixed_huffman_blocks", "extra_subfields",
                                  "sq_order_and_comments"])
def test_htslib_shaped_files_on_the_device(engine, tmp_path, name):
    """The files of tests/test_bam_htslib_shapes.py (end-of-file marker, empty blocks inside, stored / fixed-Huffman blocks,
    extra gzip subfields, every optional-field type, CG placeholder CIGARs ...) through the kernels: counts and statistics
    equal those from the hand-computed columns pushed directly."""
    from oracle import te_oracle
    from test_bam_htslib_shapes import expected, write_variant
    path = str(tmp_path / (name + ".bam"))
    recs = write_variant(path, name)
    idx = H.load_index("idx_rand_a.glb")
    engine.upload_index(idx)
    want = expected(recs, idx)
    n, info, got = _device_run(engine, path, "se", idx, None, 20)
    assert n == len(recs)
    engine.bulk_begin(False, 20)
    engine.bulk_push(len(recs), want["start"], want["end"], want["chrom"], want["mapq"], want["flag"])
    counts, st = engine.bulk_finish()
    assert np.array_equal(got[0], counts) and np.array_equal(got[1], st)
    oc, _ = te_oracle.bulk_count(H.oracle_index(idx), False, 20, *[want[k].tolist() for k in ("start", "end", "chrom", "mapq", "flag")])
    assert counts.tolist() == oc and sum(oc) > 0


@pytest.fixture(scope="module")
def tenx():
    from test_bgzf_dev_cpu import tenx_whitelist
    return tenx_whitelist()


@pytest.mark.parametrize("window_blocks", [1, 5])
def test_device_decoder_10x_whitelist(engine, tmp_path, tenx, window_blocks):
    """The device whitelist table at 737 280 barcodes (16 bases + '-1'): probe chains that wrap past the last slot,
    absent barcodes that walk a full chain, one-base neighbours, prefixes and extensions (some of them with the home
    slot of the barcode they extend), against libtecbam."""
    from test_bgzf_dev_cpu import tenx_records
    wl_list, groups = tenx
    path = str(tmp_path / "x.bam")
    write_bam(path, tenx_records(wl_list, groups, 6000, 5), block=3000)
    wlf = tmp_path / "wl.txt"
    wlf.write_text("".join(w + "\n" for w in wl_list))
    wl = reads.Whitelist(str(wlf))
    idx = H.load_index("idx_rand_a.glb")
    engine.upload_index(idx)
    want = _host_run(engine, path, "sc", idx, wl, 20)
    engine.set_option("bam_window_blocks", window_blocks)
    try:
        n, info, got = _device_run(engine, path, "sc", idx, wl, 20)
    finally:
        engine.set_option("bam_window_blocks", 32768)
    assert n == 6000 and info["host_inflated_blocks"] == 0
    assert len(want) == len(got)
    for a, b in zip(want, got):
        assert np.array_equal(a, b)
    assert want[5][_lib.SS_INVALID_BARCODE] > 1000 and want[5][_lib.SS_VALID] > 1000
