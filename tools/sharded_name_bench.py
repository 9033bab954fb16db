"""Paired end by read name with the file split over the GPUs of one node (te_counter_b200/shard.py: byte ranges, mode 4;
dist.bulk_name_exchange: the rows meet at the rank that owns their read name).  Writes a coordinate-sorted synthetic
paired-end BAM (te_counter_b200.synth_bam, sorted_pe=True), then for each rank count runs one process per GPU under
torch.distributed.run.  Every rank reports:
  - parse_bampe(pairing='name') end to end: the best of --repeat calls, host clock around the call, which ends in a
    device synchronise (tec_bulk_finish); the engine and the index upload are made before the clock starts;
  - the same steps one at a time, each behind a device synchronise and a barrier: the range decode (tec_bam_count_range
    mode 4), the exchange with the bytes this rank sends and receives (32 per record), and the device time of the
    pairing pass over the received records (tec_get_info "bulk_name_ms").
World 1 runs the whole-file decode (mode 3) end to end, and the range path over one range for the breakdown.  World sizes
above the number of GPUs are not measured: ranks sharing a GPU over gloo show correctness, not scaling (the tests cover
them).  Also reported: whether each TSV equals the world-1 TSV, and the name and power limit of the GPUs, read in the same
run.  Needs GPUs; prints one JSON line and writes it to --out-dir.

    python tools/sharded_name_bench.py --records 16000000 --worlds 1,2,4,8 --out-dir profiles/
"""
import argparse
import json
import logging
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _steps(mte, eng, bam, world, rank, device):
    """the steps of the sharded path one at a time; returns this rank's numbers"""
    import torch
    import torch.distributed as dist
    from te_counter_b200 import dist as tdist, reads, shard

    def barrier():
        eng.sync()
        if world > 1:
            dist.barrier()
        return time.perf_counter()

    eng.bulk_begin(True, 20, pairing="name")
    dev = eng.bam_open(bam)
    dev.bind(reads.ChromMap(mte.genome.chrom_keys))
    t0 = barrier()
    info = dev.count_range(4, 20, *shard.byte_range(os.path.getsize(bam), rank, world))
    eng.sync()
    t1 = time.perf_counter()
    dev.close()
    t2 = barrier()
    if world > 1:
        received = tdist.bulk_name_exchange(eng, torch.device("cuda", device))
    else:
        send, ptr = eng.bulk_name_partition_dev(1)
        eng.bulk_name_import_dev(send[0], ptr)
        received = send[0]
    eng.sync()
    t3 = time.perf_counter()
    excluded = eng.get_info("bulk_name_excluded")
    return {"rank": rank, "records_decoded": info["n"], "range_decode_s": t1 - t0, "exchange_s": t3 - t2,
            "bytes_sent": 32 * (info["n"] - excluded), "bytes_received": 32 * received,
            "bulk_name_ms": eng.get_info("bulk_name_ms")}


def worker(a):
    import torch
    import torch.distributed as dist
    import te_counter_b200
    from te_counter_b200 import synth
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    device = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(device)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", device))
    log = logging.getLogger("sharded_name_bench")
    log.addHandler(logging.NullHandler())
    log.propagate = False
    idx = synth.synth_index()
    mte = te_counter_b200.measureTE("sharded_name_bench", 20, device=device)
    mte.genome = idx
    mte.all_feature_names = idx.names
    eng = mte._engine()                                 # engine + index upload before the clock
    times = []
    for _ in range(a.repeat):
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        res = mte.parse_bampe(a.bam, log=log, pairing="name")
        times.append(time.perf_counter() - t0)
    if rank == 0:
        mte.save_result_bulk(res, a.tsv, log=log)
    mine = dict(_steps(mte, eng, a.bam, world, rank, device), parse_bampe_best_s=min(times), parse_bampe_s=times)
    ranks = [mine]
    if world > 1:
        ranks = [None] * world
        dist.all_gather_object(ranks, mine)
    if rank == 0:
        with open(a.json, "w") as fh:
            json.dump({"world": world, "seconds": max(r["parse_bampe_best_s"] for r in ranks), "paired_records": 2 * (mte.total_reads - 1),
                       "backend": "nccl" if world > 1 else "none", "ranks": ranks}, fh)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=16000000)
    ap.add_argument("--worlds", default="1,2,4,8")
    ap.add_argument("--repeat", type=int, default=3)
    ap.add_argument("--out-dir", default=".")
    ap.add_argument("--dir", default=None, help="where the BAM is written (default: a temporary directory)")
    ap.add_argument("--worker", action="store_true")
    ap.add_argument("--bam")
    ap.add_argument("--tsv")
    ap.add_argument("--json")
    a = ap.parse_args()
    if a.worker:
        return worker(a)
    import torch
    n_gpu = torch.cuda.device_count()
    if not n_gpu:
        raise SystemExit("no GPU: nothing to measure")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    work = a.dir or tempfile.mkdtemp(prefix="sharded_name_bench_")
    bam = os.path.join(work, "sorted.bam")
    from te_counter_b200 import synth_bam
    size = synth_bam.write(bam, records=a.records, mode="pe", sorted_pe=True)
    out = {"records_in_file": a.records, "file_bytes": size, "gpus_on_node": n_gpu, "gpus": smi.strip().splitlines(), "runs": []}
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""), TEC_INDEX_CACHE="0")
    one_tsv = None
    for world in [int(w) for w in a.worlds.split(",")]:
        if world > n_gpu:
            out["runs"].append({"world": world, "not_measured": "more ranks than GPUs on the node"})
            continue
        tsv, js = os.path.join(work, "w%d.tsv" % world), os.path.join(work, "w%d.json" % world)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
               "--master-port", str(29760 + world), os.path.abspath(__file__), "--worker", "--bam", bam, "--tsv", tsv, "--json", js,
               "--repeat", str(a.repeat)]
        subprocess.run(cmd, check=True, cwd=ROOT, env=env)
        r = json.load(open(js))
        r["records_per_s"] = a.records / r["seconds"]
        if one_tsv is None and world == 1:
            one_tsv = open(tsv, "rb").read()
        r["tsv_equals_one_rank"] = None if one_tsv is None else open(tsv, "rb").read() == one_tsv
        out["runs"].append(r)
    line = json.dumps(out)
    print(line)
    os.makedirs(a.out_dir, exist_ok=True)
    with open(os.path.join(a.out_dir, "sharded_name_bench.json"), "w") as fh:
        fh.write(line + "\n")


if __name__ == "__main__":
    main()
