"""bench.py --dump-outputs: the seeded sample of the single-cell triples and the size limit of the written arrays."""
import argparse

import numpy as np
import pytest

import bench


def _triples(n, seed):
    rng = np.random.default_rng(seed)
    key = np.unique(rng.integers(0, 1 << 40, size=n, dtype=np.uint64))
    return (key >> np.uint64(32)).astype(np.int32), (key & np.uint64(0xFFFFFFFF)).astype(np.uint32), \
        rng.integers(1, 1000, size=len(key)).astype(np.int64)


def test_sample_depends_on_the_set_not_the_order():
    ensg, cell, count = _triples(50_000, 1)
    a = bench.sample_triples(ensg, cell, count, 1000)
    perm = np.random.default_rng(2).permutation(len(ensg))
    b = bench.sample_triples(ensg[perm], cell[perm], count[perm], 1000)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    key = a[0].astype(np.int64) << 32 | a[1].astype(np.int64)
    assert len(key) == 1000 and (np.diff(key) > 0).all()
    # every kept triple carries its own count
    src = dict(zip((ensg.astype(np.int64) << 32 | cell.astype(np.int64)).tolist(), count.tolist()))
    assert [src[k] for k in key.tolist()] == a[2].tolist()
    # a smaller sample is a subset of a larger one
    small = bench.sample_triples(ensg, cell, count, 100)
    assert set(zip(small[0].tolist(), small[1].tolist())) <= set(zip(a[0].tolist(), a[1].tolist()))


def test_sample_keeps_everything_below_the_cap():
    ensg, cell, count = _triples(500, 3)
    perm = np.random.default_rng(4).permutation(len(ensg))
    e, c, n = bench.sample_triples(ensg[perm], cell[perm], count[perm], 10_000)
    assert np.array_equal(e, ensg) and np.array_equal(c, cell) and np.array_equal(n, count)
    assert all(len(x) == 0 for x in bench.sample_triples(ensg, cell, count, 0))


def _ctx(dump_outputs, rank=0):
    """A bench.Ctx with only what keep_outputs needs (no engine, no device)."""
    C = bench.Ctx.__new__(bench.Ctx)
    C.args, C.rank, C.outputs = argparse.Namespace(dump_outputs=dump_outputs), rank, {}
    return C


def test_legs_fill_the_outputs_within_the_budget(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 200_000)
    C = _ctx(str(tmp_path / "out"))
    for leg in ("bulk_pe", "bulk_se"):
        C.keep_outputs(leg, counts=np.arange(2000, dtype=np.int64), stats=np.arange(8, dtype=np.int64))
    ensg, cell, count = _triples(50_000, 5)
    C.keep_sc_outputs(ensg, cell, count, np.arange(300, dtype=np.uint32), np.ones(300, dtype=np.int64),
                      np.zeros(16, dtype=np.int64), np.arange(100, dtype=np.uint32), len(ensg))
    assert sorted(C.outputs) == sorted(["bulk_pe_counts", "bulk_pe_stats", "bulk_se_counts", "bulk_se_stats", "sc_stats",
                                        "sc_hit_cell", "sc_hit_count", "sc_selected", "sc_n_triples", "sc_ensg",
                                        "sc_cell", "sc_count"])
    assert all(a.dtype == np.float64 and a.ndim == 1 for a in C.outputs.values())
    assert C.outputs["sc_n_triples"].tolist() == [len(ensg)]
    # the triples take what is left of the budget after every other array, in whole triples
    rest = bench.DUMP_BYTES - sum(a.nbytes for k, a in C.outputs.items() if k not in ("sc_ensg", "sc_cell", "sc_count"))
    assert len(C.outputs["sc_ensg"]) == rest // 24 < len(ensg)
    info = bench.write_outputs(C.args.dump_outputs, C.outputs)
    assert info["arrays"] == 12 and info["bytes"] <= bench.DUMP_BYTES
    assert np.load(tmp_path / "out" / "bulk_se_counts.npy").tolist() == list(range(2000))


def test_outputs_kept_only_when_asked_and_on_rank_0():
    for C in (_ctx(None), _ctx("out", rank=1)):
        C.keep_outputs("bulk_pe", counts=np.arange(3))
        C.keep_sc_outputs(*_triples(10, 6), np.arange(2), np.arange(2), np.zeros(16), np.arange(1), 10)
        assert C.outputs == {}


def test_write_outputs(tmp_path, monkeypatch):
    arrays = {"bulk_pe_counts": np.arange(10, dtype=np.float64), "sc_stats": np.zeros(16)}
    info = bench.write_outputs(str(tmp_path / "out"), arrays)
    assert info["arrays"] == 2 and info["bytes"] == 208
    got = np.load(tmp_path / "out" / "bulk_pe_counts.npy")
    assert got.dtype == np.float64 and got.tolist() == list(range(10))
    monkeypatch.setattr(bench, "DUMP_BYTES", 200)
    with pytest.raises(SystemExit):
        bench.write_outputs(str(tmp_path / "over"), arrays)
    assert not (tmp_path / "over").exists()
