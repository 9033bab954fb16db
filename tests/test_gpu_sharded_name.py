"""Paired end by read name with one file split over ranks (tec_bam_count_range mode 4, tec_bulk_name_partition_dev,
tec_bulk_name_import_dev, tec_bulk_name_exchange; dist.bulk_name_exchange).  In one process: ranks run one after another
on one GPU, Python routes the packed records by owner, and the summed counters equal the whole-file mode-3 decode and the
oracle.  Through torch.distributed.run: the TSV and rank 0's log are those of a one-rank run."""
import os

import numpy as np
import pytest

import helpers as H
from te_counter_b200 import _lib, reads, shard
from test_gpu_pair_name import EXTRA, GLB, _device, _oracle, _sorted_file
from test_gpu_sharded_pe import _launch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engines():
    idx = H.load_index(GLB)
    engs = []
    for _ in range(8):
        e = _lib.Engine(0)
        e.upload_index(idx)
        engs.append(e)
    yield engs
    for e in engs:
        e.close()


def _open(eng, path):
    d = eng.bam_open(path)
    d.bind(reads.ChromMap(H.load_index(GLB).chrom_keys))
    return d


def _ranges_in_turn(engs, path, world, window_blocks):
    """every rank's range, partition, routing by owner in Python, import and finish; (summed counts, stats, excluded,
    records per owner)"""
    import torch
    size = os.path.getsize(path)
    infos, parts = [], []
    for r in range(world):
        e = engs[r]
        e.set_option("bam_window_blocks", window_blocks)
        e.bulk_begin(True, 20, pairing="name")
        d = _open(e, path)
        infos.append(d.count_range(4, 20, *shard.byte_range(size, r, world)))
        d.close()
        e.set_option("bam_window_blocks", 65536)
        send, ptr = e.bulk_name_partition_dev(world)
        src = torch.as_tensor(_DevBytes(ptr, sum(send) * 32), device="cuda:0") if sum(send) else torch.empty(0, dtype=torch.uint8, device="cuda:0")
        parts.append(list(torch.split(src.clone(), [x * 32 for x in send])))          # copies: the owners import later
    assert shard.chain_is_consistent(infos), infos
    torch.cuda.synchronize()
    counts, stats, excluded, owned = 0, 0, 0, []
    for o in range(world):
        dst = torch.cat([parts[r][o] for r in range(world)])                          # laid out by source rank
        torch.cuda.synchronize()
        engs[o].bulk_name_import_dev(dst.numel() // 32, dst.data_ptr() if dst.numel() else None)
        c, s = engs[o].bulk_finish()
        counts, stats = counts + c, stats + s
        excluded += engs[o].get_info("bulk_name_excluded")
        owned.append(dst.numel() // 32)
    return counts, stats, excluded, owned


class _DevBytes:
    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "|u1", "data": (ptr, False), "version": 2}


@pytest.mark.parametrize("seed", [21, 22])
def test_ranks_in_turn_sum_to_the_whole_file(engines, tmp_path, seed):
    path = str(tmp_path / "s.bam")
    recs = _sorted_file(seed, 6000, path, block=1500)
    o_counts, o_st, excl, no_mate = _oracle(path)
    n, w_counts, w_st = _device(engines[0], path)
    assert n == len(recs) and np.array_equal(w_counts, o_counts) and np.array_equal(w_st[:7], o_st)
    for window_blocks in (1, 7, 65536):
        for world in (1, 2, 3, 8):
            counts, st, e, owned = _ranges_in_turn(engines, path, world, window_blocks)
            assert np.array_equal(counts, w_counts), (world, window_blocks)
            assert np.array_equal(st, w_st), (world, window_blocks)
            assert e == excl and st[_lib.BS_NO_MATE] == excl + no_mate
            assert sum(owned) == len(recs) - excl and (world == 1 or min(owned) > 0)


def test_library_exchange_on_a_one_rank_communicator(engines, tmp_path):
    """tec_bulk_name_exchange over NCCL (rank 0 sends to itself) gives the counters of the whole-file decode"""
    path = str(tmp_path / "s.bam")
    recs = _sorted_file(23, 4000, path, block=1500)
    _, w_counts, w_st = _device(engines[0], path, 7)
    e = _lib.Engine(0)
    try:
        e.upload_index(H.load_index(GLB))
        e.comm_init(e.comm_unique_id(), 0, 1)
        for window_blocks in (7, 65536):
            e.set_option("bam_window_blocks", window_blocks)
            e.bulk_begin(True, 20, pairing="name")
            d = _open(e, path)
            info = d.count_range(4, 20, 0, os.path.getsize(path))
            d.close()
            assert info["n"] == len(recs)
            n = e.bulk_name_exchange()
            assert n == len(recs) - e.get_info("bulk_name_excluded")
            e.bulk_allreduce()
            counts, st = e.bulk_finish()
            assert np.array_equal(counts, w_counts) and np.array_equal(st, w_st), window_blocks
    finally:
        e.close()


def test_abi_edges(engines, tmp_path):
    path = str(tmp_path / "s.bam")
    _sorted_file(24, 500, path)
    e = engines[0]
    d = _open(e, path)
    size = os.path.getsize(path)
    e.bulk_begin(True, 20)                                       # mode 4 needs the name-pairing begin
    with pytest.raises(_lib.TecError) as x:
        d.count_range(4, 20, 0, size)
    assert x.value.status == -3
    e.bulk_begin(True, 20, pairing="name")
    with pytest.raises(_lib.TecError) as x:
        e.bulk_name_partition_dev(2)                             # nothing held yet
    assert x.value.status == -3
    info = d.count_range(4, 20, 0, size)
    assert info["n"] > 0
    for call in (e.bulk_finish, lambda: e.bulk_name_import_dev(0, None), lambda: d.count(3, 20)):
        with pytest.raises(_lib.TecError) as x:                  # held rows wait for the partition
            call()
        assert x.value.status == -3
    # a new begin drops the held rows: nothing is counted
    e.bulk_begin(True, 20, pairing="name")
    counts, st = e.bulk_finish()
    assert not counts.any() and not st.any()
    # a range with no records: the partition sends nothing, the import takes nothing, the counters stay zero
    e.bulk_begin(True, 20, pairing="name")
    info = d.count_range(4, 20, size, size)
    assert info["n"] == 0
    send, _ = e.bulk_name_partition_dev(3)
    assert send == [0, 0, 0]
    e.bulk_name_import_dev(0, None)
    counts, st = e.bulk_finish()
    assert not counts.any() and not st.any()
    d.close()


def _log_lines(log):
    return [ln for ln in log.splitlines() if ln.startswith("INFO")]


def test_sharded_cli_by_name_same_tsv_and_log(tmp_path):
    path = str(tmp_path / "s.bam")
    _sorted_file(25, 20000, path, block=20000)
    glb = os.path.join(H.GOLD, GLB)
    args = ["--glb", glb, "--bam", path, "--mode", "pe", "--pairing", "name"]
    one = str(tmp_path / "one.tsv")
    rc, log1 = _launch(1, 0, args + ["-o", one])
    assert rc == 0, log1[-3000:]
    assert EXTRA in log1
    want = [ln.replace(one, "OUT") for ln in _log_lines(log1)]
    for world in (2, 3):
        out = str(tmp_path / ("w%d.tsv" % world))
        rc, log = _launch(world, 29690 + world, args + ["-o", out])
        assert rc == 0, log[-3000:]
        assert open(out, "rb").read() == open(one, "rb").read()
        assert "decoded by this rank" in log                     # the ranges were used, not the fallback
        got = [ln.replace(out, "OUT") for ln in _log_lines(log) if "decoded by this rank" not in ln]
        assert got == want, (world, got, want)
    out = str(tmp_path / "refused.tsv")
    rc, log = _launch(2, 29699, args + ["-o", out], {"TEC_TEST_SHARD_REFUSE": "1"})
    assert rc == 0, log[-3000:]
    assert open(out, "rb").read() == open(one, "rb").read()
    assert "decoded by this rank" not in log


def test_two_gpus_over_nccl_same_tsv(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs: the library exchange over NCCL between two devices")
    path = str(tmp_path / "s.bam")
    _sorted_file(26, 20000, path, block=20000)
    args = ["--glb", os.path.join(H.GOLD, GLB), "--bam", path, "--mode", "pe", "--pairing", "name"]
    one, two = str(tmp_path / "one.tsv"), str(tmp_path / "two.tsv")
    rc, log = _launch(1, 0, args + ["-o", one])
    assert rc == 0, log[-3000:]
    rc, log = _launch(2, 29701, args + ["-o", two])
    assert rc == 0, log[-3000:]
    assert "decoded by this rank" in log and open(two, "rb").read() == open(one, "rb").read()
