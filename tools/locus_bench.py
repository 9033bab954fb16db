"""Counts per index row (bulk locus mode, tec_set_option "bulk_loci") on one GPU, against the same runs without it.

1. Device-resident arrays: bench.py's bulk shapes (500 M records, synth.synth_bulk_reads on the hg38-like
   synth.synth_index), single end and paired end.  One step = tec_bulk_begin + tec_bulk_push_dev, timed with CUDA events
   around each step; reported as the median of --steps steps after --warmup, with loci off (the default kernels) and on
   (the exact search kernel with the row tally).  Checked in the same run: per-name counts and statistics identical,
   the rows equal to the C oracle (tests/locus_oracle_c.c) bit for bit, and the row sums per name at least the counts.
2. From a file: a --file-records paired-end synthetic BAM (synth_bam) through parse_bampe with and without loci=True,
   host clock around each call (it ends in a device synchronise); counts must be equal.
3. Writer: time and bytes of save_result_loci on the hg38-like index.

Needs a GPU; prints one JSON line and writes it to --out-dir.

    python tools/locus_bench.py --out-dir profiles/
"""
import argparse
import json
import logging
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))                 # tests/locus_oracle.py: the checker
T0 = time.perf_counter()
COLS = ("start", "end", "chrom", "mapq", "flag")


def log(msg):
    print("[locus_bench %.0f s] %s" % (time.perf_counter() - T0, msg), file=sys.stderr, flush=True)


def device_arm(eng, idx, paired, n_rec, steps, warmup):
    import torch
    import locus_oracle
    from te_counter_b200 import synth
    reads = synth.synth_bulk_reads(synth.SEED, idx, n_rec, paired=paired, device="cuda:0", as_numpy=False)
    ptrs = [reads[k].data_ptr() for k in COLS]
    torch.cuda.synchronize()
    out, res = {}, {}
    # loci off on the default kernels, on the exact search kernel alone (bulk_algo 0: the kernel locus mode runs
    # on, without the row tally), and loci on
    for arm, loci, algo in (("loci_off", 0, -1), ("exact_loci_off", 0, 0), ("loci_on", 1, -1)):
        eng.set_option("bulk_loci", loci)
        eng.set_option("bulk_algo", algo)
        times = []
        for s in range(warmup + steps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(torch.cuda.ExternalStream(eng.stream))
            eng.bulk_begin(paired, 20)
            eng.bulk_push_dev(n_rec, *ptrs)
            e1.record(torch.cuda.ExternalStream(eng.stream))
            e1.synchronize()
            if s >= warmup:
                times.append(e0.elapsed_time(e1))
        counts, st = eng.bulk_finish()
        res[arm] = (counts, st, eng.bulk_loci() if loci else None)
        ms = float(np.median(times))
        out[arm] = {"median_ms": ms, "times_ms": times, "records_per_s": n_rec / (ms * 1e-3)}
        log("%s %s: %.2f ms" % ("pe" if paired else "se", arm, ms))
    eng.set_option("bulk_loci", 0)
    eng.set_option("bulk_algo", -1)
    out["identical_counts_and_stats"] = all(np.array_equal(res["loci_off"][i], res[k][i]) for k in ("exact_loci_off", "loci_on")
                                            for i in (0, 1))
    host = {k: reads[k].cpu().numpy() for k in COLS}
    del reads
    t = time.perf_counter()
    oc, ost, ol = locus_oracle.c_bulk_count_loci(locus_oracle.CIndex(idx), paired, 20, *[host[k] for k in COLS])
    out["oracle_s"] = time.perf_counter() - t
    order = idx.sorted_layout()["order"]
    counts, st, loci = res["loci_on"]
    out["oracle_counts_equal"] = bool(np.array_equal(counts, oc) and np.array_equal(st[:7], ost))
    out["oracle_loci_equal"] = bool(np.array_equal(loci, ol[order]))
    per_name = np.bincount(idx.sorted_layout()["ensg_id"], weights=loci, minlength=idx.n_ensg)
    out["sum_identity"] = bool((per_name >= counts).all())
    out["rows_hit"] = int((loci > 0).sum())
    out["row_count_sum"], out["name_count_sum"] = int(loci.sum()), int(counts.sum())
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=500_000_000)
    ap.add_argument("--file-records", type=int, default=16_000_000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out-dir", default=".")
    a = ap.parse_args()
    import torch
    if not torch.cuda.device_count():
        raise SystemExit("no GPU: nothing to measure")
    import te_counter_b200
    from te_counter_b200 import _lib, synth, synth_bam
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    idx = synth.synth_index()
    out = {"gpus": smi.strip().splitlines(), "records": a.records, "file_records": a.file_records, "steps": a.steps,
           "warmup": a.warmup, "n_features": idx.n_features, "n_ensg": idx.n_ensg, "host_cpus": os.cpu_count()}
    eng = _lib.Engine(0)
    eng.upload_index(idx)
    for paired in (False, True):
        out["device_pe" if paired else "device_se"] = device_arm(eng, idx, paired, a.records - (a.records & 1), a.steps, a.warmup)
    eng.close()
    torch.cuda.empty_cache()

    work = tempfile.mkdtemp(prefix="locus_bench_")
    path = os.path.join(work, "pe.bam")
    size = synth_bam.write(path, records=a.file_records, mode="pe")
    log("wrote %s (%d bytes)" % (path, size))
    quiet = logging.getLogger("locus_bench")
    quiet.addHandler(logging.NullHandler())
    quiet.propagate = False
    mte = te_counter_b200.measureTE("locus_bench", 20, device=0)
    mte.genome = idx
    mte.all_feature_names = idx.names
    mte._engine()
    os.environ["TEC_BAM_DECODER"] = "gpu"
    f = {"file_bytes": size}
    res = {}
    for rep in range(a.warmup + a.steps):
        for loci in (False, True):                              # alternated, so both arms see the same machine state
            t = time.perf_counter()
            r = mte.parse_bampe(path, log=quiet, loci=loci)
            dt = time.perf_counter() - t
            if rep >= a.warmup:
                f.setdefault("loci_on_s" if loci else "loci_off_s", []).append(dt)
            res[loci] = r
    for k in ("loci_off_s", "loci_on_s"):
        f[k.replace("_s", "_median_s")] = float(np.median(f[k]))
    f["identical_counts"] = res[False] == res[True]
    f["bam_info_us"] = getattr(mte, "_bam_info", None)
    out["file_pe"] = f
    t = time.perf_counter()
    tsv = os.path.join(work, "loci.tsv")
    mte.save_result_loci(tsv)
    out["writer"] = {"s": time.perf_counter() - t, "bytes": os.path.getsize(tsv), "rows": idx.n_features}
    os.unlink(tsv)
    os.unlink(path)
    os.rmdir(work)
    line = json.dumps(out)
    print(line)
    os.makedirs(a.out_dir, exist_ok=True)
    with open(os.path.join(a.out_dir, "r03_locus_bench.json"), "w") as fh:
        fh.write(line + "\n")
    ok = all(out[k][c] for k in ("device_se", "device_pe")
             for c in ("identical_counts_and_stats", "oracle_counts_equal", "oracle_loci_equal", "sum_identity"))
    if not (ok and f["identical_counts"]):
        raise SystemExit("a check failed")


if __name__ == "__main__":
    main()
