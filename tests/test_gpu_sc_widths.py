"""The single-cell path at production key widths: whitelists of 2 to 2^23 + 1 barcodes (1 to 24 cell bits), UMIs of 1 to
21 characters and chromosome ids up to 0xFFEF, so that the (cell, UMI, chrom:strand) key of the packed sort reaches
bit 63, and inputs on both sides of the 64-bit line where tec_sc_finalize leaves the packed key for the library sorts.
Every case is held against the oracle with the checks of test_gpu_sc.check_against_oracle and asserts, through
tec_get_info("sc_last_sort" / "sc_last_sort_passes"), the sort route it was written for."""
import numpy as np
import pytest

import helpers as H
from oracle import te_oracle, te_oracle_c
from te_counter_b200 import _lib, reads, synth
from test_gpu_sc import COLS, _matrix_text, _text_from_triples, check_against_oracle, run_engine

pytestmark = pytest.mark.gpu

PACKED, LIB2, LIB3 = 1, 2, 3          # sc_last_sort: packed key + radix.cuh, library sorts on 2-bit / 3-bit UMI keys
INVALID = 0xFFFFFFFF
V2, V3 = 737_280, 1 << 23             # 10x v2 whitelist; 2^23 ids (a v3 whitelist needs 23 bits)


def cell_bits(W):
    return max(1, (W - 1).bit_length())


@pytest.fixture(scope="module")
def idx():
    return synth.synth_index(11, n_te=30000, n_exon=9000, n_gene=600, chrom_len=3_000_000, n_chrom=3)


@pytest.fixture(scope="module")
def engine(idx):
    eng = _lib.Engine(0)
    eng.upload_index(idx)
    yield eng
    eng.close()


def pinned_cells(W):
    """0, W - 1 and the ids 2^k - 1, 2^k below W: every cell bit set and cleared on its own."""
    p = {0, W - 1}
    for k in range(1, cell_bits(W) + 1):
        p |= {c for c in ((1 << k) - 1, 1 << k) if c < W}
    return sorted(p)


def make_reads(idx, seed, W, L, max_chrom=None, n=20000, n_wl=300):
    """synth_sc_reads over `n_wl` barcodes, the barcodes then spread over [0, W) with the pinned ids first.  Every 7th
    read moves to a chromosome outside the index (ids n_index .. max_chrom); the first reads are survivors that carry
    the pinned cells and max_chrom itself."""
    rng = np.random.default_rng(seed)
    n_wl = min(n_wl, W)
    r = synth.synth_sc_reads(seed, idx, n, n_whitelist=n_wl, n_cells=min(60, n_wl), umis_per_cell=40, umi_len=L)
    pins = pinned_cells(W)
    rest = np.setdiff1d(rng.choice(W, size=min(W, 2 * n_wl + len(pins)), replace=False), pins)
    ids = np.concatenate([pins, rng.permutation(rest)])[:n_wl].astype(np.uint32)
    cell = r["cell"]
    r["cell"] = np.where(cell == INVALID, cell, ids[np.minimum(cell, n_wl - 1)]).astype(np.uint32)
    n_index = int(idx.chrom_id.max()) + 1
    if max_chrom is not None and max_chrom >= n_index:
        far = np.arange(3, n, 7)
        r["chrom"][far] = rng.integers(n_index, max_chrom + 1, len(far)).astype(np.uint16)
        r["chrom"][far[0]] = max_chrom
    head = np.arange(len(pins) + 1)
    f = int(np.argmax(idx.R - idx.L))                   # the pinned cells' reads lie inside one long feature
    r["start"][head] = idx.L[f] + 5 + head
    r["end"][head] = idx.L[f] + 6 + head
    r["chrom"][head] = idx.chrom_id[f]
    r["cell"][head[:-1]] = pins
    r["cell"][head[-1]] = ids[0]
    r["mapq"][head] = 60
    r["flag"][head] &= ~np.uint8(te_oracle.F_UNMAPPED | te_oracle.F_DUP | te_oracle.F_QCFAIL)
    if max_chrom is not None and max_chrom >= n_index:
        r["chrom"][head[-1]] = max_chrom
    return r


def key_bits(r, W, L, strand, qual=20):
    """cell bits + 2 L + bits of the OR of the survivors' chrom:strand words: the width of the packed key."""
    f = r["flag"]
    surv = ((f & (te_oracle.F_UNMAPPED | te_oracle.F_DUP | te_oracle.F_QCFAIL)) == 0) & (r["mapq"] >= qual) & (r["cell"] != INVALID) & \
        (r["chrom"] != reads.CHROM_SC_SKIP)
    sc = np.where(f & te_oracle.F_REVERSE, 1, 0) if strand else np.full(len(f), 2)
    cs = (r["chrom"].astype(np.int64) << 2) | sc
    return cell_bits(W) + 2 * L + int(np.bitwise_or.reduce(cs[surv])).bit_length()


def check(engine, idx, r, W, L, strand, route, bundle_keys=10 ** 7, maxcells=50, pad=1000):
    out = check_against_oracle(engine, idx, r, 20, strand, W, bundle_keys, maxcells, pad)
    assert engine.get_info("sc_last_sort") == route
    want_passes = -(-(cell_bits(W) + 2 * L) // 11) if route == PACKED else 0
    assert engine.get_info("sc_last_sort_passes") == want_passes
    assert out["stats"]["assigned"] > 0
    return out


@pytest.mark.parametrize("W", [2, 1 << 10, V2, V3, V3 + 1])
def test_whitelist_sizes(engine, idx, W):
    """1, 10, 20, 23 and 24 cell bits: packed sorts of 3, 4, 4, 5 and 5 passes; the triple sort's cell pass takes
    1 to 3 digits.  Both strand settings (strand code 2 sets bit 1 of the chrom:strand word)."""
    r = make_reads(idx, 20 + W % 97, W, 12)
    for strand in (False, True):
        check(engine, idx, r, W, 12, strand, PACKED)
    if W <= V2:
        check(engine, idx, r, W, 12, True, PACKED, bundle_keys=700)


@pytest.mark.parametrize("W,L,max_chrom,strand,bits,route", [
    (V3, 12, (1 << 14) - 1, True, 63, PACKED),
    (V3, 12, (1 << 15) - 1, False, 64, PACKED),
    (V3, 12, 1 << 15, True, 65, LIB2),
    (1 << 20, 16, (1 << 10) - 1, False, 64, PACKED),
    (1 << 20, 16, 1 << 10, True, 65, LIB2),
    (V2, 12, 0xFFEF, False, 62, PACKED),
    (V3 + 1, 12, 0xFFEF, True, 66, LIB2),
])
def test_packing_boundary(engine, idx, W, L, max_chrom, strand, bits, route):
    """cell bits + 2 L + chrom:strand bits of 63 and 64 take the packed key (bit 63 is a key bit), 65 and more the
    library sorts; chromosome ids up to the largest one a file may carry (0xFFEF), most of them outside the index."""
    r = make_reads(idx, 30 + bits, W, L, max_chrom)
    assert key_bits(r, W, L, strand) == bits
    check(engine, idx, r, W, L, strand, route)


@pytest.mark.parametrize("L", [1, 2, 11, 16, 17, 21])
def test_umi_lengths(engine, idx, L):
    """L = 1: four UMIs in all, heavy key duplication; 17 and 21 characters do not fit 2 bits per character in 32 bits
    and take the 3-bit codes."""
    route = PACKED if L <= 16 else LIB3
    r = make_reads(idx, 40 + L, V2, L, max_chrom=200)
    for strand in (False, True):
        check(engine, idx, r, V2, L, strand, route)
    engine.set_option("sc_sort", 0)
    try:
        check(engine, idx, r, V2, L, True, LIB2 if L <= 16 else LIB3, bundle_keys=900)
    finally:
        engine.set_option("sc_sort", 1)


def test_packed_pass_counts(engine, idx):
    """1, 2 and 6 passes: two cells and one-character UMIs (3 key bits), 1024 cells and two-character UMIs (14 bits),
    2^23 + 1 cells and 16-character UMIs (56 bits)."""
    for W, L, passes in ((2, 1, 1), (1 << 10, 2, 2), (V3 + 1, 16, 6)):
        r = make_reads(idx, 50 + W % 97, W, L)
        assert key_bits(r, W, L, True) <= 64
        check(engine, idx, r, W, L, True, PACKED)
        assert engine.get_info("sc_last_sort_passes") == passes


@pytest.mark.parametrize("shape", ["v3+1", "64-bit"])
def test_sort_routes(engine, idx, shape):
    """The four ways to group the survivors on one input: packed key with prev[] stored in place, packed key with prev[]
    through a radix pass and three tiles per chunk, library sorts on 2-bit and on 3-bit UMI keys."""
    W, max_chrom = (V3 + 1, 2) if shape == "v3+1" else (V3, (1 << 15) - 1)
    r = make_reads(idx, 60 + len(shape), W, 12, max_chrom)
    try:
        for sort, pack, prev, chunk, route in ((1, 1, 0, 1, PACKED), (1, 1, 2, 3, PACKED), (0, 1, 0, 1, LIB2), (0, 0, 0, 1, LIB3)):
            engine.set_option("sc_sort", sort)
            engine.set_option("sc_pack_umi", pack)
            engine.set_option("sc_prev_partition", prev)
            engine.set_option("sc_sort_chunk", chunk)
            check(engine, idx, r, W, 12, True, route)
            check(engine, idx, r, W, 12, False, route, bundle_keys=1500)
    finally:
        engine.set_option("sc_sort", 1)
        engine.set_option("sc_pack_umi", 1)
        engine.set_option("sc_prev_partition", 0)
        engine.set_option("sc_sort_chunk", 1)


def tie_reads(idx, seed, W, n_cells):
    """n_cells cells spread over [0, W), each with 2 to 4 reads of distinct UMIs inside one long feature."""
    rng = np.random.default_rng(seed)
    cells = np.sort(rng.choice(W, size=n_cells, replace=False)).astype(np.uint32)
    cells[-1] = W - 1
    reps = rng.integers(2, 5, n_cells)                  # the first read of a cell only opens its line (Part 2)
    cell = np.repeat(cells, reps)
    k = np.arange(len(cell)) - np.repeat(np.cumsum(reps) - reps, reps)
    n = len(cell)
    f = int(np.argmax(idx.R - idx.L))
    start = np.full(n, idx.L[f] + 5, np.int32)
    umi = np.array([1, 2, 3, 5], np.uint64)[k] << np.uint64(3 * 20)              # 'A', 'C', 'G', 'T': one-character UMIs
    return {"start": start, "end": start + 1, "chrom": np.full(n, idx.chrom_id[f], np.uint16), "mapq": np.full(n, 60, np.uint8),
            "flag": np.zeros(n, np.uint8), "cell": cell, "umi": umi}


def test_select_many_ties(engine, idx):
    """tec_sc_select over 120 000 hit cells in 2^23 ids with 1 to 3 hits each: the 10 000 cells with the most hits,
    ties by the lower id, against sorted(cell_hits, key=(-hits, cell)) and the C++ oracle."""
    W, maxcells = V3, 10_000
    r = tie_reads(idx, 7, W, 120_000)
    engine.sc_begin(20, False, W)
    engine.sc_push(len(r["start"]), *[r[k] for k in COLS])
    nt, nh = engine.sc_finalize(10 ** 7, maxcells, 200_000)          # every cell is a to-do cell of Part 2
    ensg, cell, count, hcell, hcount, st = engine.sc_fetch(nt, nh)
    sel = engine.sc_select(maxcells, nh)
    out = te_oracle_c.sc_count((idx.chrom_id, idx.L, idx.R, idx.ensg_id, idx.type_code, idx.strand_code),
                               int(idx.chrom_id.max()) + 1, idx.bucket_size, 20, False, 10 ** 7, maxcells, 200_000, *[r[k] for k in COLS])
    assert list(zip(hcell.tolist(), hcount.tolist())) == sorted(out["cell_hits"])
    assert {(int(e), int(c)): int(v) for e, c, v in zip(ensg, cell, count)} == out["triples"]
    assert nh >= 100_000 and set(hcount.tolist()) == {1, 2, 3}
    want = [c for c, _ in sorted(zip(hcell.tolist(), hcount.tolist()), key=lambda t: (-t[1], t[0]))[:maxcells]]
    assert sel.tolist() == want
    assert engine.get_info("sc_last_sort") == PACKED


def test_matrix_text_at_v3_plus_one(engine, idx):
    """tec_sc_matrix_text after a finalize over 2^23 + 1 ids (a rank array of that length): the selected cells' rows and
    rows of cells near W - 1 that have no entry."""
    W = V3 + 1
    r = make_reads(idx, 70, W, 12)
    check(engine, idx, r, W, 12, True, PACKED, maxcells=30)
    ensg, cell, count, hcell, hcount, st, sel = run_engine(engine, r, 20, True, W, 10 ** 7, 30, 1000)
    assert len(sel) >= 10 and W - 1 in set(hcell.tolist())
    hit = set(hcell.tolist())
    empty = [c for c in range(W - 1, W - 40, -1) if c not in hit][:5]
    for cells in (sel.tolist(), empty + sel.tolist()[:3], [W - 1]):
        names = ["%016x-1" % c for c in cells]
        assert _matrix_text(engine, cells, names) == _text_from_triples(idx.n_ensg, ensg, cell, count, cells, names)


@pytest.fixture(scope="module")
def comm_engine(idx):
    eng = _lib.Engine(0)
    try:
        eng.comm_init(eng.comm_unique_id(), 0, 1)
    except _lib.TecError as e:
        eng.close()
        pytest.skip("NCCL not available: %s" % e)
    eng.upload_index(idx)
    yield eng
    eng.close()


def test_exchange_single_rank_at_v3_plus_one(comm_engine, idx):
    """tec_sc_exchange + tec_sc_allgather_triples on one rank over 2^23 + 1 ids: the gathered triples are sorted again
    by their cell bits (sc_comm.cuh) and must equal the oracle's, ascending in (ensg, cell)."""
    W = V3 + 1
    r = make_reads(idx, 80, W, 12, max_chrom=40)
    eng = comm_engine
    for strand in (False, True):
        eng.sc_begin(20, strand, W)
        eng.sc_push(len(r["start"]), *[r[k] for k in COLS])
        assert eng.sc_exchange() == eng.sc_survivors()
        nt, nh = eng.sc_finalize(10 ** 7, 50, 1000)
        assert eng.sc_allgather_triples() == nt
        assert eng.get_info("sc_last_sort") == PACKED
        ensg, cell, count, hcell, hcount, st = eng.sc_fetch(nt, nh)
        out = te_oracle.sc_count(H.oracle_index(idx), 20, strand, 10 ** 7, 50, 1000, *[r[k].tolist() for k in COLS])
        assert {(int(e), int(c)): int(v) for e, c, v in zip(ensg, cell, count)} == out["triples"]
        key = ensg.astype(np.int64) << 32 | cell.astype(np.int64)
        assert (np.diff(key) > 0).all() and cell.max() == W - 1
        assert list(zip(hcell.tolist(), hcount.tolist())) == sorted(out["cell_hits"])
