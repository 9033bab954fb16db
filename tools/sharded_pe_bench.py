"""Paired-end file -> counts with the file split over the GPUs of one node (te_counter_b200/shard.py: byte ranges, global
record parity, counter banks).  Writes a synthetic paired-end BAM (te_counter_b200.synth_bam), then for each rank count
runs parse_bampe under torch.distributed.run, one process per GPU.  On every rank the host clock is taken around
parse_bampe, which ends in a device synchronise (tec_bulk_finish); the engine and the index upload are made before the
clock starts, and process start and index load stay outside it.  Reported: the maximum over ranks of the best of
--repeat calls, records per second, and whether the TSV equals the one-rank TSV.  World sizes above the number of
GPUs are skipped.  Needs GPUs; prints one JSON line and writes it to --out-dir.

    python tools/sharded_pe_bench.py --records 16000000 --worlds 1,2,4,8 --out-dir profiles/
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


def worker(a):
    import torch
    import torch.distributed as dist
    import te_counter_b200
    from te_counter_b200 import synth
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    n_gpu = torch.cuda.device_count()
    device = int(os.environ.get("LOCAL_RANK", "0")) % max(1, n_gpu)
    torch.cuda.set_device(device)
    if world > 1:
        if n_gpu >= world:
            dist.init_process_group("nccl", device_id=torch.device("cuda", device))
        else:
            dist.init_process_group("gloo")
    log = logging.getLogger("sharded_pe_bench")
    log.addHandler(logging.NullHandler())
    log.propagate = False
    idx = synth.synth_index()
    mte = te_counter_b200.measureTE("sharded_pe_bench", 20, device=device)
    mte.genome = idx
    mte.all_feature_names = idx.names
    mte._engine()                                       # engine + index upload before the clock
    times = []
    for _ in range(a.repeat):
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        res = mte.parse_bampe(a.bam, log=log)
        times.append(time.perf_counter() - t0)
    best = min(times)
    worst_rank = [best]
    if world > 1:
        worst_rank = [None] * world
        dist.all_gather_object(worst_rank, best)
    if rank == 0:
        mte.save_result_bulk(res, a.tsv, log=log)
        with open(a.json, "w") as fh:
            json.dump({"world": world, "seconds": max(worst_rank), "per_rank_best_s": worst_rank,
                       "records": 2 * (mte.total_reads - 1), "backend": "nccl" if world > 1 and n_gpu >= world else "gloo" if world > 1 else "none"}, fh)
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
    work = a.dir or tempfile.mkdtemp(prefix="sharded_pe_bench_")
    bam = os.path.join(work, "pe.bam")
    from te_counter_b200 import synth_bam
    size = synth_bam.write(bam, records=a.records, mode="pe")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    out = {"records_in_file": a.records, "file_bytes": size, "gpus_on_node": n_gpu, "gpus": smi.strip().splitlines(), "runs": []}
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""), TEC_INDEX_CACHE="0")
    one_tsv = None
    for world in [int(w) for w in a.worlds.split(",")]:
        if world > n_gpu:
            out["runs"].append({"world": world, "skipped": "more ranks than GPUs"})
            continue
        tsv, js = os.path.join(work, "w%d.tsv" % world), os.path.join(work, "w%d.json" % world)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
               "--master-port", str(29700 + world), os.path.abspath(__file__), "--worker", "--bam", bam, "--tsv", tsv, "--json", js,
               "--repeat", str(a.repeat)]
        subprocess.run(cmd, check=True, cwd=ROOT, env=env)
        r = json.load(open(js))
        r["records_per_s"] = r["records"] / r["seconds"]
        if one_tsv is None and world == 1:
            one_tsv = open(tsv, "rb").read()
        r["tsv_equals_one_rank"] = None if one_tsv is None else open(tsv, "rb").read() == one_tsv
        out["runs"].append(r)
    line = json.dumps(out)
    print(line)
    os.makedirs(a.out_dir, exist_ok=True)
    with open(os.path.join(a.out_dir, "sharded_pe_bench.json"), "w") as fh:
        fh.write(line + "\n")


if __name__ == "__main__":
    main()
