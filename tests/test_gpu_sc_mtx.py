"""tec_sc_matrix_mtx and measureTE.sc_save_mtx on the device: the Matrix Market text must be byte for byte the host
formatter's (te_counter_b200/mtx.py, itself held against the dense TSV in test_sc_mtx_cpu.py) for the golden cases,
seeded runs with 5-digit counts and any column subset and order, and the production widths of test_gpu_sc_widths.py;
the ABI's edges; and the sharded CLI writes the same directory at 1, 2 and 3 ranks."""
import io
import os

import numpy as np
import pytest

import helpers as H
from oracle.ref_runner import CaptureLog
from te_counter_b200 import _lib, mtx, synth
from test_gpu_sc import COLS, _matrix_text, run_engine
from test_host_mirror import make_mte
from test_sc_mtx_cpu import check_dir_against_dense

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    eng = _lib.Engine(0)
    yield eng
    eng.close()


def device_mtx(engine, cells):
    nnz, n = engine.sc_matrix_mtx(cells)
    out = io.BytesIO()
    engine.sc_matrix_write(out, n, chunk=4096 + 7)            # several chunks, odd size
    assert out.tell() == n
    raw = out.getvalue()
    assert int(raw.split(b"\n", 2)[1].split()[2]) == nnz
    return raw


@pytest.mark.parametrize("name", H.case_names("sc"))
def test_golden_cases_through_mirror(monkeypatch, tmp_path, name):
    """Every single-cell golden case through measureTE on the device: the directory describes the dense TSV of the same
    run (the reference's bytes), and matrix.mtx is the host formatter's text of the same triples and cells."""
    import gzip
    case = H.load_case(name)
    mte = make_mte(monkeypatch, case, _lib.Engine, batch=1000)
    wl = tmp_path / "wl.txt"
    wl.write_text("".join(w + "\n" for w in case["whitelist"]))
    log = CaptureLog()
    res = mte.sc_parse_bamse("mem.bam", UMIS=True, whitelistfilename=str(wl), strand=case["strand"], log=log,
                             label="lbl", maxcells=case["maxcells"], _bundle_keys=case["bundle_keys"], _pad=case["pad"])
    out = tmp_path / "o.tsv"
    mte.sc_save_result(res, str(out), maxcells=case["maxcells"], log=log)
    assert out.read_text() == case["expected"]["tsv"]
    d = str(tmp_path / "mtx")
    mte.sc_save_mtx(res, d, maxcells=case["maxcells"], log=log)
    raw = check_dir_against_dense(d, case["expected"]["tsv"])
    sel = mte._engine_obj.sc_select(case["maxcells"], len(mte._sc_hit[0]))
    assert raw == mtx.mtx_text(len(res), res.ensg, res.cell, res.count, sel)
    assert gzip.decompress(open(os.path.join(d, "matrix.mtx.gz"), "rb").read()) == raw


def test_seeded_rows_any_subset_and_order(engine):
    """The shapes of test_gpu_sc.test_sc_matrix_text_rows: counts up to 5 digits, cells without entries, any column
    subset and order."""
    idx = synth.synth_index(3, n_te=3000, n_exon=800, n_gene=60, chrom_len=300_000, n_chrom=2)
    engine.upload_index(idx)
    n_wl = 40
    r = synth.synth_sc_reads(6, idx, 30000, n_whitelist=n_wl, n_cells=12, umis_per_cell=300)
    f = int(np.argmax(idx.R - idx.L))
    extra = {k: [] for k in COLS}
    for cellid, n_umi in ((3, 12346), (7, 151)):               # a 5-digit and a 3-digit count on one feature
        u = np.arange(n_umi, dtype=np.uint64)
        code = np.zeros(n_umi, dtype=np.uint64)
        for k in range(8):
            code = (code << np.uint64(3)) | ((u // np.uint64(5 ** (7 - k))) % np.uint64(5) + np.uint64(1))
        code <<= np.uint64(3 * (21 - 8))
        extra["start"].append(np.full(n_umi, idx.L[f] + 5, np.int32))
        extra["end"].append(np.full(n_umi, idx.L[f] + 6, np.int32))
        extra["chrom"].append(np.full(n_umi, idx.chrom_id[f], np.uint16))
        extra["mapq"].append(np.full(n_umi, 60, np.uint8))
        extra["flag"].append(np.zeros(n_umi, np.uint8))
        extra["cell"].append(np.full(n_umi, cellid, np.uint32))
        extra["umi"].append(code)
    r = {k: np.concatenate([np.asarray(r[k])] + extra[k]).astype(np.asarray(r[k]).dtype) for k in COLS}
    ensg, cell, count, hcell, hcount, st, sel = run_engine(engine, r, 20, False, n_wl, 10 ** 7, 30, 1000)
    assert count.max() >= 10000 and len(sel) >= 5
    no_hit = [c for c in range(n_wl) if c not in set(hcell.tolist())]
    rng = np.random.default_rng(9)
    for cells in (sel.tolist(), sel.tolist()[::-1][:4], [int(sel[0])], sel.tolist()[:3] + no_hit[:2], no_hit[:3],
                  rng.permutation(n_wl).tolist()):
        assert device_mtx(engine, cells) == mtx.mtx_text(idx.n_ensg, ensg, cell, count, cells)


def test_production_widths(engine):
    """2^23 + 1 whitelist ids (a rank array of that length), the cells near W - 1 without entries, the selection in
    both orders."""
    from test_gpu_sc_widths import V3, make_reads
    idx = synth.synth_index(11, n_te=30000, n_exon=9000, n_gene=600, chrom_len=3_000_000, n_chrom=3)
    engine.upload_index(idx)
    W = V3 + 1
    r = make_reads(idx, 70, W, 12)
    ensg, cell, count, hcell, hcount, st, sel = run_engine(engine, r, 20, True, W, 10 ** 7, 30, 1000)
    assert len(sel) >= 10 and W - 1 in set(hcell.tolist())
    hit = set(hcell.tolist())
    empty = [c for c in range(W - 1, W - 40, -1) if c not in hit][:5]
    for cells in (sel.tolist(), sel.tolist()[::-1], empty + sel.tolist()[:3], [W - 1], hcell.tolist()[::-1]):
        assert device_mtx(engine, cells) == mtx.mtx_text(idx.n_ensg, ensg, cell, count, cells)


def test_abi_edges(engine):
    idx = synth.synth_index(3, n_te=3000, n_exon=800, n_gene=60, chrom_len=300_000, n_chrom=2)
    fresh = _lib.Engine(0)
    try:
        fresh.upload_index(idx)
        with pytest.raises(_lib.TecError) as e:
            fresh.sc_matrix_mtx([0])                                       # no tec_sc_begin
        assert e.value.status == -3
        fresh.sc_begin(20, False, 10)
        with pytest.raises(_lib.TecError) as e:
            fresh.sc_matrix_mtx([0])                                       # begun, not finalized
        assert e.value.status == -3
    finally:
        fresh.close()
    engine.upload_index(idx)
    # a finalize without triples: columns without entries
    engine.sc_begin(20, False, 5)
    assert engine.sc_finalize(10 ** 7, 3, 1000)[0] == 0
    head = b"%%MatrixMarket matrix coordinate integer general\n"
    assert device_mtx(engine, [4, 1]) == head + b"%d 2 0\n" % idx.n_ensg
    assert device_mtx(engine, []) == head + b"%d 0 0\n" % idx.n_ensg     # zero columns: the header only
    # with triples
    r = synth.synth_sc_reads(6, idx, 20000, n_whitelist=40, n_cells=12, umis_per_cell=100)
    ensg, cell, count, hcell, hcount, st, sel = run_engine(engine, r, 20, False, 40, 10 ** 7, 30, 1000)
    assert len(ensg) > 0
    for bad in ([0, 0], [int(sel[0]), 3, int(sel[0])], [40], [2, 10 ** 6]):
        with pytest.raises(_lib.TecError) as e:
            engine.sc_matrix_mtx(bad)
        assert e.value.status == -2
    assert device_mtx(engine, []) == head + b"%d 0 0\n" % idx.n_ensg
    # the dense text, then the MTX text replaces it, then the dense text again unchanged
    names = ["bc%d" % c for c in sel.tolist()]
    dense = _matrix_text(engine, sel, names)
    want = mtx.mtx_text(idx.n_ensg, ensg, cell, count, sel)
    assert device_mtx(engine, sel) == want
    assert _matrix_text(engine, sel, names) == dense


def test_sharded_cli_one_two_three_ranks(tmp_path):
    """`sharded --mode sc --format mtx` at 1, 2 and 3 ranks writes byte-identical directories that describe the dense
    TSV of the one-rank run.  Ranks sharing one GPU go over gloo (host formatter on rank 0); with one GPU per rank the
    library's NCCL path keeps the job's triples on the device."""
    from bam_writer import write_bam
    from test_gpu_sharded_file import _records, _run
    recs, wl = _records(30000, 79, True)
    bam = str(tmp_path / "sc.bam")
    write_bam(bam, recs, block=20000)
    wlf = tmp_path / "wl.txt"
    wlf.write_text("".join(w + "\n" for w in wl))
    glb = os.path.join(H.GOLD, "idx_rand_a.glb")
    base = ["--glb", glb, "--bam", bam, "--mode", "sc", "--whitelist", str(wlf), "--maxcells", "40", "--strand"]
    tsv = str(tmp_path / "one.tsv")
    _run(1, 0, base + ["-o", tsv])
    files = ("matrix.mtx.gz", "features.tsv.gz", "barcodes.tsv.gz")
    got = {}
    for world in (1, 2, 3):
        d = str(tmp_path / ("w%d" % world))
        _run(world, 29640 + world, base + ["--format", "mtx", "-o", d])
        got[world] = [open(os.path.join(d, f), "rb").read() for f in files]
    assert got[2] == got[1] and got[3] == got[1]
    check_dir_against_dense(str(tmp_path / "w1"), open(tsv).read())
