"""Paired-end BAM split over ranks by global record parity (tec_bam_count_range mode 1, tec_bulk_keep_bank,
tec_bam_pair_columns; te_counter_b200/shard.py pair_plan).  In one process: ranks run one after another on one GPU and
their summed counters equal the whole-file decode and the C oracle.  Through torch.distributed.run: the TSV of the
sharded run is byte for byte the one-rank TSV, and the name-mismatch crash of a pair across a range border is raised
the same way."""
import os
import subprocess
import sys

import numpy as np
import pytest

import helpers as H
from bam_writer import write_bam
from oracle import te_oracle_c
from te_counter_b200 import _lib, fastbam, reads, shard
from test_fastbam import _mixed_records
from test_gpu_sharded_file import _records

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def engine():
    eng = _lib.Engine(0)
    yield eng
    eng.close()


def _host_columns(path, idx, qual):
    f = fastbam.NativeBam(path, threads=2)
    f.bind(reads.ChromMap(idx.chrom_keys))
    b = reads.Batch(1 << 14)
    parts, more = [], True
    while more:
        more = f.fill_bulk(b, True, qual)
        parts.append({k: getattr(b, k)[:b.n].copy() for k in ("start", "end", "chrom", "mapq", "flag")})
    f.close()
    return {k: np.concatenate([p[k] for p in parts]) for k in parts[0]}


def _open(eng, path, idx):
    d = eng.bam_open(path)
    d.bind(reads.ChromMap(idx.chrom_keys))
    return d


@pytest.mark.parametrize("block,window_blocks", [(3000, 32768), (700, 5), (65000, 2)])
def test_ranks_in_turn_sum_to_the_whole_file(engine, tmp_path, block, window_blocks):
    n = 6001
    recs = _mixed_records(n, 41 + block, False)[0]
    path = str(tmp_path / "x.bam")
    write_bam(path, recs, block=block)
    idx = H.load_index("idx_rand_a.glb")
    engine.upload_index(idx)
    engine.set_option("bam_window_blocks", window_blocks)
    try:
        d = _open(engine, path, idx)
        engine.bulk_begin(True, 20)
        assert d.count(1, 20) == n - 1
        d.close()
        whole = [a.copy() for a in engine.bulk_finish()]
        cols = _host_columns(path, idx, 20)
        oc = te_oracle_c.Index(idx.chrom_id, idx.L, idx.R, idx.ensg_id, idx.type_code, idx.n_chrom, idx.n_ensg, idx.bucket_size)
        o_counts, o_stats = te_oracle_c.bulk_count(oc, True, 20, cols["start"], cols["end"], cols["chrom"], cols["mapq"], cols["flag"])
        assert np.array_equal(whole[0], o_counts) and np.array_equal(whole[1][:7], o_stats)
        size = os.path.getsize(path)
        n_border = 0
        for world in (1, 2, 3, 8, 37):
            infos = []
            for rank in range(world):                      # pass 1: the range infos every rank would gather
                d = _open(engine, path, idx)
                engine.bulk_begin(True, 20)
                infos.append(d.count_range(1, 20, *shard.byte_range(size, rank, world)))
                d.close()
            assert shard.chain_is_consistent(infos), world
            plan = shard.pair_plan(infos)
            counts, stats = np.zeros_like(whole[0]), np.zeros_like(whole[1])
            for rank in range(world):                      # pass 2: count, keep the bank, push the border pair
                d = _open(engine, path, idx)
                engine.bulk_begin(True, 20)
                d.count_range(1, 20, *shard.byte_range(size, rank, world))
                with pytest.raises(_lib.TecError):
                    engine.bulk_finish()                   # the bank is not chosen yet
                engine.bulk_keep_bank(plan[rank]["bank"])
                if plan[rank]["border"] is not None:
                    c = d.pair_columns(*plan[rank]["border"], 20)
                    engine.bulk_push(2, c["start"], c["end"], c["chrom"], c["mapq"], c["flag"])
                    n_border += 1
                d.close()
                c_r, s_r = engine.bulk_finish()
                counts += c_r
                stats += s_r
            assert np.array_equal(counts, whole[0]), world
            assert np.array_equal(stats, whole[1]), world
            assert stats[_lib.BS_UNITS] == n // 2
        assert n_border > 0
    finally:
        engine.set_option("bam_window_blocks", 65536)


def _launch(world, port, args, extra_env=None):
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""), TEC_INDEX_CACHE="0")
    env.update(extra_env or {})
    if world == 1:
        cmd = [sys.executable, "-m", "te_counter_b200.sharded"] + args
    else:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
               "--master-port", str(port), "-m", "te_counter_b200.sharded"] + args
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    return p.returncode, p.stdout + p.stderr


def test_pe_file_split_over_ranks(tmp_path):
    recs, _ = _records(30001, 81, False)
    bam = str(tmp_path / "pe.bam")
    write_bam(bam, recs, block=20000)
    glb = os.path.join(H.GOLD, "idx_rand_a.glb")
    one = str(tmp_path / "one.tsv")
    rc, log = _launch(1, 0, ["--glb", glb, "--bam", bam, "--mode", "pe", "-o", one])
    assert rc == 0, log[-3000:]
    for world in (2, 3):
        out = str(tmp_path / ("w%d.tsv" % world))
        rc, log = _launch(world, 29640 + world, ["--glb", glb, "--bam", bam, "--mode", "pe", "-o", out])
        assert rc == 0, log[-3000:]
        assert open(out, "rb").read() == open(one, "rb").read()
        assert "decoded by this rank" in log                              # the ranges were used, not the fallback
    out = str(tmp_path / "fallback.tsv")
    rc, log = _launch(2, 29650, ["--glb", glb, "--bam", bam, "--mode", "pe", "-o", out], {"TEC_TEST_SHARD_REFUSE": "1"})
    assert rc == 0, log[-3000:]
    assert "decoded by this rank" not in log
    assert open(out, "rb").read() == open(one, "rb").read()


def _first_record_of_rank1(path, idx):
    """index of rank 1's first record when two ranks split the file (range decode on the device, single end)"""
    eng = _lib.Engine(0)
    try:
        eng.upload_index(idx)
        d = _open(eng, path, idx)
        eng.bulk_begin(False, 0)
        n0 = d.count_range(0, 0, *shard.byte_range(os.path.getsize(path), 0, 2))["n"]
        d.close()
        return n0
    finally:
        eng.close()


def test_name_mismatch_across_the_border_crashes_like_one_rank(tmp_path):
    """The only pair whose mate names differ is (read1 = last record of rank 0, read2 = first record of rank 1).
    Stored (level 0) blocks and equal-length names keep the file's layout when one name changes."""
    idx = H.load_index("idx_rand_a.glb")
    glb = os.path.join(H.GOLD, "idx_rand_a.glb")
    bam = str(tmp_path / "pe.bam")
    for n in range(4001, 4401, 2):
        recs = [{"chrom": "chr1", "start": 1000 + 7 * i, "end": 1100 + 7 * i, "mapq": 60, "name": "p%06d/%d" % (i // 2, i % 2 + 1)}
                for i in range(n)]
        write_bam(bam, recs, block=5000, level=0)
        first = _first_record_of_rank1(bam, idx)
        if first % 2:
            break
    assert first % 2
    recs[first]["name"] = "z%06d/2" % (first // 2)
    write_bam(bam, recs, block=5000, level=0)
    assert _first_record_of_rank1(bam, idx) == first
    for world, port in ((1, 0), (2, 29660)):
        rc, log = _launch(world, port, ["--glb", glb, "--bam", bam, "--mode", "pe", "-o", str(tmp_path / "o.tsv")])
        assert rc != 0
        assert "AttributeError: module 'sys' has no attribute 'quit'" in log, log[-3000:]
        if world == 2:
            assert "decoded by this rank" in log
