"""The 10x-style Matrix Market directory of measureTE.sc_save_mtx on CPU: the host formatter (te_counter_b200/mtx.py)
against the dense rows of sc_save_result for the same triples and cells, the piecewise gzip writer, and the CLI switch.
The GPU tests (test_gpu_sc_mtx.py) hold the device text against the same formatter."""
import gzip
import io
import os

import numpy as np
import pytest
import scipy.io

import helpers as H
from oracle.ref_runner import CaptureLog
from oracle_engine import OracleEngine
from test_host_mirror import make_mte
import te_counter_b200
from te_counter_b200 import mtx, sharded
from te_counter_b200 import te_count as mirror


def parse_dense(text):
    """(feature names, barcodes, cells x features int64 array) of the dense TSV of sc_save_result"""
    lines = text.split("\n")
    assert lines[-1] == ""
    names = lines[0].split("\t")[1:]
    rows = [ln.split("\t") for ln in lines[1:-1]]
    m = np.array([[int(x) for x in r[1:]] for r in rows], dtype=np.int64).reshape(len(rows), len(names))
    return names, [r[0] for r in rows], m


def check_dir_against_dense(out_dir, dense_text):
    """out_dir describes exactly the matrix of the dense TSV: matrix.mtx.gz read by scipy is its transpose, the features
    are its header, the barcodes its rows.  Returns the decompressed matrix.mtx."""
    names, barcodes, m = parse_dense(dense_text)
    raw = gzip.decompress(open(os.path.join(out_dir, "matrix.mtx.gz"), "rb").read())
    a = scipy.io.mmread(os.path.join(out_dir, "matrix.mtx.gz"), spmatrix=False)
    a = a.toarray() if hasattr(a, "toarray") else np.asarray(a)
    assert a.shape == (len(names), len(barcodes))
    assert (a.astype(np.int64) == m.T).all()
    head = raw.split(b"\n", 2)
    assert head[0] == b"%%MatrixMarket matrix coordinate integer general"
    assert head[1] == b"%d %d %d" % (len(names), len(barcodes), int((m != 0).sum()))
    feats = gzip.decompress(open(os.path.join(out_dir, "features.tsv.gz"), "rb").read()).decode()
    assert feats == "".join("%s\t%s\tGene Expression\n" % (n, n) for n in names)
    bcs = gzip.decompress(open(os.path.join(out_dir, "barcodes.tsv.gz"), "rb").read()).decode()
    assert bcs == "".join(b + "\n" for b in barcodes)
    return raw


def reference_mtx(n_ensg, ensg, cell, count, cells):
    """The Matrix Market text restated line by line from its definition (include/tecount.h tec_sc_matrix_mtx)."""
    col = {int(c): k for k, c in enumerate(cells)}
    ent = sorted((col[int(c)], int(e), int(v)) for e, c, v in zip(ensg, cell, count) if int(c) in col)
    return (b"%%MatrixMarket matrix coordinate integer general\n" + b"%d %d %d\n" % (n_ensg, len(cells), len(ent)) +
            b"".join(b"%d %d %d\n" % (e + 1, k + 1, v) for k, e, v in ent))


class _SelectEngine:
    """The one engine call sc_save_mtx makes on the host path: sc_select over the given hit counts."""

    def __init__(self, hits):
        self.hits = hits

    def sc_select(self, maxcells, n_hit):
        order = sorted(self.hits.items(), key=lambda t: (-t[1], t[0]))[:maxcells]
        return np.array([c for c, _ in order], np.uint32)


def save_both(tmp_path, names, id_to_barcode, ensg, cell, count, maxcells, tag="x"):
    """sc_save_result and sc_save_mtx of one ScResult built from (ensg, cell, count) sorted by (ensg, cell), with a
    cell's hit count = its number of non-zeros; returns (dense TSV text, mtx directory, selected cells, triples)."""
    o = np.lexsort((cell, ensg))
    ensg, cell, count = (np.asarray(ensg, np.int32)[o], np.asarray(cell, np.uint32)[o], np.asarray(count, np.int64)[o])
    res = mirror.ScResult(names, id_to_barcode, ensg, cell, count)
    hits = {}
    for c in cell.tolist():
        hits[c] = hits.get(c, 0) + 1
    mte = te_counter_b200.measureTE("test", 20)
    mte._engine_obj = _SelectEngine(hits)
    mte._sc_hit = (np.array(sorted(hits), np.uint32), np.array([hits[c] for c in sorted(hits)], np.int64))
    mte.barcodes = {id_to_barcode[c]: h for c, h in sorted(hits.items())}
    log = CaptureLog()
    tsv = str(tmp_path / ("%s.tsv" % tag))
    mte.sc_save_result(res, tsv, maxcells=maxcells, log=log)
    d = str(tmp_path / ("%s_mtx" % tag))
    mte.sc_save_mtx(res, d, maxcells=maxcells, log=log)
    sel = _SelectEngine(hits).sc_select(maxcells, len(hits))
    return open(tsv).read(), d, sel, (ensg, cell, count)


def test_hand_made_triples(tmp_path):
    """Counts from 1 to 2^63 - 1, a feature with no entry (the last), an empty barcode string, a cell whose only entry is
    in the last feature that has one."""
    names = ["ENSG%02d" % i for i in range(6)]
    wl = ["AAAC", "AAAG", "", "CCCT", "GGGA"]
    tri = [(0, 0, 1), (1, 0, 22), (4, 0, 10 ** 18), (2, 1, 2 ** 63 - 1), (3, 1, 999), (0, 2, 5), (1, 2, 10),
           (4, 3, 123456789012345678)]
    e, c, v = zip(*tri)
    dense, d, sel, tri = save_both(tmp_path, names, wl, e, c, v, maxcells=10)
    assert len(sel) == 4
    raw = check_dir_against_dense(d, dense)
    assert raw == reference_mtx(len(names), *tri, sel)
    assert raw == mtx.mtx_text(len(names), *tri, sel)


def test_counts_of_every_width_from_1_to_19_digits():
    v = np.array([10 ** k for k in range(19)] + [10 ** (k + 1) - 1 for k in range(18)] + [2 ** 63 - 1], np.int64)
    assert {len(str(int(x))) for x in v} == set(range(1, 20))
    n = len(v)
    ensg, cell = np.arange(n) % 7, np.arange(n) // 7
    cells = list(range(cell.max() + 1))[::-1]
    assert mtx.mtx_text(7, ensg, cell, v, cells) == reference_mtx(7, ensg, cell, v, cells)


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_seeded_triples(tmp_path, seed):
    """Random triples over 300 whitelist ids and 200 features; maxcells below and above the number of hit cells,
    one selection with cells that have no entry (columns of zeros) and the zero-column directory."""
    rng = np.random.default_rng(seed)
    n_wl, n_ensg = 300, 200
    names = ["G%04d" % i for i in range(n_ensg)]
    wl = ["%016x-1" % rng.integers(1 << 60) for _ in range(n_wl)]
    pairs = np.unique(rng.integers(0, n_ensg, 4000) * n_wl + rng.integers(0, 80, 4000))
    e, c = pairs // n_wl, pairs % n_wl
    v = np.where(rng.random(len(pairs)) < 0.9, rng.integers(1, 10, len(pairs)), rng.integers(1, 10 ** 6, len(pairs)))
    for maxcells in (1, 17, 80, 500):
        dense, d, sel, tri = save_both(tmp_path, names, wl, e, c, v, maxcells, tag="m%d" % maxcells)
        raw = check_dir_against_dense(d, dense)
        assert raw == reference_mtx(n_ensg, *tri, sel)
    # columns with no entry, in any order, and no columns at all
    cells = [299, 5, 150, 3, 298]
    assert mtx.mtx_text(n_ensg, *tri, cells) == reference_mtx(n_ensg, *tri, cells)
    assert mtx.mtx_text(n_ensg, *tri, []) == b"%%MatrixMarket matrix coordinate integer general\n200 0 0\n"


def test_zero_columns_directory(tmp_path):
    """No hit cell at all: a valid file with the two header lines, an empty barcodes file."""
    names = ["A", "B", "C"]
    dense, d, sel, tri = save_both(tmp_path, names, ["x", "y"], [], [], [], maxcells=5)
    assert len(sel) == 0
    raw = check_dir_against_dense(d, dense)
    assert raw == b"%%MatrixMarket matrix coordinate integer general\n3 0 0\n"


@pytest.mark.parametrize("name", H.case_names("sc"))
def test_golden_cases_through_mirror(monkeypatch, tmp_path, name):
    """Every single-cell golden case through measureTE with the CPU oracle as the engine: the directory describes the
    dense TSV of the same run, which is the reference's."""
    case = H.load_case(name)
    mte = make_mte(monkeypatch, case, OracleEngine, batch=1000)
    wl = tmp_path / "wl.txt"
    wl.write_text("".join(w + "\n" for w in case["whitelist"]))
    log = CaptureLog()
    res = mte.sc_parse_bamse("mem.bam", UMIS=True, whitelistfilename=str(wl), strand=case["strand"], log=log,
                             label="lbl", maxcells=case["maxcells"], _bundle_keys=case["bundle_keys"], _pad=case["pad"])
    mte.sc_save_mtx(res, str(tmp_path / "mtx"), maxcells=case["maxcells"], log=log)
    raw = check_dir_against_dense(str(tmp_path / "mtx"), case["expected"]["tsv"])
    sel = mte._engine_obj.sc_select(case["maxcells"], 0)
    assert raw == reference_mtx(len(res), res.ensg, res.cell, res.count, sel)
    assert any("Saving the sparse matrix" in m for _, m in log.lines)


def test_rejects_anything_but_sc_result(tmp_path):
    mte = te_counter_b200.measureTE("test", 20)
    with pytest.raises(TypeError):
        mte.sc_save_mtx({"ENSG1": {"AAAC": 1}}, str(tmp_path / "d"), maxcells=3, log=CaptureLog())


def _gz(text, threads, step=None):
    out = io.BytesIO()
    with mtx.ThreadPoolExecutor(max_workers=threads) as pool:
        gz = mtx.GzipPieces(out, pool, 2 * threads)
        for a in range(0, len(text), step or max(1, len(text))):
            gz.write(text[a:a + (step or len(text))])
        gz.close()
    return out.getvalue()


@pytest.mark.parametrize("size", [0, 1000, mtx.PIECE - 1, mtx.PIECE, mtx.PIECE + 1, 2 * mtx.PIECE + 12345])
def test_gzip_pieces_do_not_depend_on_threads(size):
    """Texts shorter than, equal to and longer than one piece: the same bytes at 1 and 8 threads and for any write
    sizes; gzip.decompress gives the text back; one member per started piece."""
    rng = np.random.default_rng(size)
    words = np.array([b"%d %d %d\n" % (i % 977 + 1, i % 31 + 1, i % 13 + 1) for i in range(4096)], dtype=object)
    text = b"".join(words[rng.integers(0, 4096, size // 8 + 1)].tolist())[:size]
    one = _gz(text, 1)
    assert _gz(text, 8) == one
    assert _gz(text, 8, step=(1 << 22) + 7) == one
    assert gzip.decompress(one) == text
    members = one.count(b"\x1f\x8b\x08")
    assert members >= max(1, -(-size // mtx.PIECE))


def test_write_gzip_file(tmp_path):
    p = str(tmp_path / "t.gz")
    mtx.write_gzip(p, lambda fh: fh.write(b"abc\n" * 1000), 3)
    assert gzip.open(p).read() == b"abc\n" * 1000


@pytest.mark.parametrize("mode", ["se", "pe"])
def test_cli_rejects_mtx_outside_single_cell(mode, capsys):
    with pytest.raises(SystemExit) as e:
        sharded.main(["--glb", "x.glb", "--bam", "x.bam", "--mode", mode, "--format", "mtx", "-o", "out"])
    assert e.value.code == 2
    assert "--format mtx" in capsys.readouterr().err
