#!/usr/bin/env python3
"""
bench.py -- reads/sec of the counting hot path on B200 (BASELINE.json metric), ONE JSON line.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # all three workloads, see below
    python bench.py --workload bulk_pe|bulk_se|sc ...               # one workload as the headline
    python bench.py --impl reference ...                            # the unmodified reference on the host cores
    python bench.py --dump-outputs DIR ...                          # also save the last timed step's results

The headline of the line is BASELINE.json configs[3] (synthetic 500 M-record paired-end bulk on an hg38-like
genes_tes index, SURVEY.md 8d): a "step" is one pass of filter -> overlap -> tally (+ cross-GPU merge) over the
whole workload.  The same line carries two more objects measured the same way in the same process:
  "bulk_se"  the configs[3] reads taken as single-end records (short leg),
  "sc"       BASELINE.json configs[4], 10x-style single cell: 1 B records at N = 1, 250 M per GPU at N > 1
             (UMI collapse, Part-2 rule, overlap, tally, selection; NCCL exchange by cell at N > 1).
Every leg reports `value` (inputs resident in HBM, CUDA events on the library's stream, max over ranks),
`roofline` (algorithmic bytes / kernel time against the measured HBM peak), `e2e` (through the host-buffer
C ABI with pinned host arrays, H2D / D2H inside the timed region) and parity against the oracle.
Inputs (>= 6 GB per step) are far larger than the 126 MB L2, so no explicit flush is needed between steps.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BYTES_PER_RECORD = {"bulk_pe": 12, "bulk_se": 12, "sc": 24}        # SURVEY.md 8(d)
INDEX_BYTES_PER_FEATURE = 16
CONFIG_RECORDS = {"bulk_pe": 500_000_000, "bulk_se": 500_000_000, "sc": 1_000_000_000}
SC_RECORDS_MULTI = 250_000_000                                      # per GPU at N > 1
DUMP_BYTES = 64_000_000                                             # --dump-outputs: 64 MB for all arrays together
DUMP_TRIPLES = 2_000_000                                            # single-cell triples kept by the sample
DUMP_SEED = 20261018


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="all", choices=["all", "bulk_pe", "bulk_se", "sc"])
    ap.add_argument("--records", type=int, default=0, help="records per GPU (default: the config's size)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--index-scale", type=float, default=1.0)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--cpu-sample", type=int, default=600_000, help="records of the CPU-baseline sample")
    ap.add_argument("--ref-sample", type=int, default=300_000, help="reference arm: records per step")
    ap.add_argument("--sorted", action="store_true", help="coordinate-sorted arrival order (bulk_se)")
    ap.add_argument("--sc-parity-records", type=int, default=30_000_000,
                    help="sc: records of the large parity check against the C++ oracle (0 = skip)")
    ap.add_argument("--sc-e2e-records", type=int, default=250_000_000, help="sc: records of the host-buffer leg")
    ap.add_argument("--file-records", type=int, default=8_000_000,
                    help="records of the synthetic BAM file of the from_file leg (0 = skip)")
    ap.add_argument("--opt", action="append", default=[], help="engine tuning knob key=value (tec_set_option)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what each timed leg returned in its last step to DIR/<leg>_<name>.npy (float64, "
                         "at most 64 MB in all; the single-cell triples are a fixed, seeded sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs saves the results of --impl ours")
    return args


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def make_index(scale):
    from te_counter_b200 import synth
    if scale == 1.0:
        return synth.synth_index()
    return synth.synth_index(n_te=int(4_600_000 * scale), n_exon=int(1_300_000 * scale),
                             n_gene=max(10, int(38_000 * scale)), n_te_names=max(10, int(1200 * min(1.0, scale * 4))))


WORKLOAD_NAMES = {
    "bulk_pe": "BASELINE.json configs[3]: synthetic paired-end bulk RNA-seq, hg38-like genes_tes index "
               "(5.9 M features, 39.2 k ensg), name-collated random arrival order",
    "bulk_se": "synthetic single-end bulk RNA-seq (configs[3] reads taken as SE), hg38-like genes_tes index",
    "sc": "BASELINE.json configs[4]: synthetic 10x-style single cell, 100 k barcodes, --maxcells 10000"}


def workload_config(args, wl, n_rec_per_gpu, world):
    return {"workload": WORKLOAD_NAMES[wl], "records_per_gpu": int(n_rec_per_gpu), "records_total": int(n_rec_per_gpu * world),
            "sharding": "genomic coordinate range per GPU, index replicated" if world > 1 else "single GPU",
            "index_scale": args.index_scale, "l2_policy": "inputs >> L2 (no flush needed)",
            "bytes_per_record": BYTES_PER_RECORD[wl]}


# ------------------------------------------------------------------------------ --dump-outputs
def sample_triples(ensg, cell, count, k, seed=DUMP_SEED):
    """The k triples whose (ensg, cell) key has the lowest seeded splitmix64 hash, in ascending key order.  The hash is
    a bijection of the key, so which triples are kept depends on the set of triples alone, not on their order."""
    key = ensg.astype(np.uint64) << np.uint64(32) | cell.astype(np.uint64)
    keep = np.arange(len(key))
    if len(key) > k:
        z = key ^ np.uint64(seed)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z ^= z >> np.uint64(31)
        keep = np.argpartition(z, k - 1)[:k] if k > 0 else keep[:0]
    keep = keep[np.argsort(key[keep], kind="stable")]
    return ensg[keep], cell[keep], count[keep]


def write_outputs(path, arrays):
    """Every array as path/<name>.npy; refuses to write more than DUMP_BYTES."""
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:
        raise SystemExit("--dump-outputs: %d bytes of results exceed the limit of %d" % (total, DUMP_BYTES))
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)
    return {"dir": os.path.abspath(path), "arrays": len(arrays), "bytes": int(total)}


# ------------------------------------------------------------------------------ clocks sampler
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown," \
        "clocks_event_reasons.sw_power_cap,power.draw"

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [l for (t, l) in self.lines if t0 - 0.05 <= t <= t1 + 0.15] or [l for _, l in self.lines[-3:]]
        for l in rows:
            f = [x.strip() for x in l.split(",")]
            try:
                sm.append(float(f[0]))
                smax = max(smax, float(f[1]))
                for nm, v in zip(names, f[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        if not sm:
            return None
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------ reference arm
def reference_setup(args):
    """The unmodified reference from baseline/_ref (baseline/ref_arm.py) with its index object for the benchmark
    index; None when baseline/_ref is absent."""
    from baseline import ref_arm
    if not ref_arm.available():
        return None
    idx = make_index(args.index_scale)
    t = time.perf_counter()
    mod = ref_arm.load()
    gl = ref_arm.make_genelist(mod, idx)
    return {"mod": mod, "gl": gl, "idx": idx, "ref_arm": ref_arm, "index_seconds": time.perf_counter() - t}


def reference_time_bulk(R, paired, arrays):
    """One call of the reference's measureTE.parse_bampe / parse_bamse on in-memory reads; returns (seconds, result,
    total_reads).  The read objects are built before the clock starts (BAM decode excluded)."""
    ra = R["ref_arm"]
    mte = ra.new_measure(R["mod"], R["gl"], R["idx"].names)
    reads = ra.bulk_reads(R["idx"], *arrays)
    t = time.perf_counter()
    res = ra.run_bulk(mte, reads, paired)
    return time.perf_counter() - t, res, mte.total_reads


def reference_time_sc(R, arrays, n_wl, strand, maxcells):
    import shutil
    import tempfile
    ra = R["ref_arm"]
    mte = ra.new_measure(R["mod"], R["gl"], R["idx"].names)
    wl = ["%016d" % i for i in range(n_wl)]
    tmp = tempfile.mkdtemp(prefix="tec_ref_sc_")
    try:
        wlf = os.path.join(tmp, "wl.txt")
        with open(wlf, "w") as oh:
            oh.write("\n".join(wl) + "\n")
        reads = ra.sc_reads(R["idx"], wl, *arrays)
        t = time.perf_counter()
        res = ra.run_sc(mte, reads, wlf, strand, maxcells, tmp)
        dt = time.perf_counter() - t
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    return dt, res, mte


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the path on the box's host cores.  The
    reference is single-threaded Python (its only thread writes spill files, te_count.py:384), so it runs on one
    core; every step is one call of parse_bampe on a bounded sample of the same synthetic workload."""
    from te_counter_b200 import synth
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = "bulk_pe" if args.workload == "all" else args.workload
    R = None if args.no_cpu else reference_setup(args)
    if R is None:
        return run_reference_port(args, wl)
    idx = R["idx"]
    n = args.ref_sample & ~1
    K, W = args.steps, args.warmup
    legs = {}

    def bulk(paired, steps, warm, n_rec):
        r = synth.synth_bulk_reads(synth.SEED, idx, n_rec, paired=paired, sort=args.sorted)
        arrays = [r[k] for k in ("start", "end", "chrom", "mapq", "flag")]
        times = []
        for i in range(warm + steps):
            dt, res, total = reference_time_bulk(R, paired, arrays)
            if i >= warm:
                times.append(dt)
        # the per-call set-up of the reference (loc_lookups over all features, te_count.py:70-73) is inside every
        # step; one call on twice the sample separates it from the marginal cost per record
        r2 = synth.synth_bulk_reads(synth.SEED + 1, idx, 2 * n_rec, paired=paired, sort=args.sorted)
        dt2, _, _ = reference_time_bulk(R, paired, [r2[k] for k in ("start", "end", "chrom", "mapq", "flag")])
        ms = 1e3 * float(np.mean(times))
        extra = dt2 - float(np.mean(times))
        marg = n_rec / extra if extra > 0.05 * float(np.mean(times)) else None
        return {"value": n_rec / (ms / 1e3), "unit": "records/s", "ms_per_step": ms, "steps": steps, "warmup": warm,
                "records_per_step": n_rec, "marginal_records_per_s": marg,
                "per_call_setup_s": None if marg is None else max(float(np.mean(times)) - n_rec / marg, 0.0),
                "counts_sum": int(sum(res.values())), "total_reads": int(total)}

    head = bulk(wl == "bulk_pe", K, W, n) if wl in ("bulk_pe", "bulk_se") else None
    if args.workload == "all":
        legs["bulk_se"] = bulk(False, K, W, n)
    if args.workload in ("all", "sc"):
        n_sc = max(1000, n // 3)
        r = synth.synth_sc_reads(synth.SEED, idx, n_sc, n_whitelist=100_000)
        arrays = [r[k] for k in ("start", "end", "chrom", "mapq", "flag", "cell", "umi")]
        ts = []
        for _ in range(W + K):
            dt, res, mte = reference_time_sc(R, arrays, 100_000, True, 10_000)
            ts.append(dt)
        ts = ts[W:]
        sc = {"value": n_sc / float(np.mean(ts)), "unit": "records/s", "ms_per_step": 1e3 * float(np.mean(ts)), "steps": len(ts),
              "records_per_step": n_sc, "what": "measureTE.sc_parse_bamse(strand=True, maxcells=10000), 100 k-barcode whitelist; "
              "load_genome bound to a no-op on the instance (index object already in place)"}
        if args.workload == "sc":
            head = sc
        else:
            legs["sc"] = sc
    value = head["value"]
    line = {"impl": "reference", "metric": "reads_per_sec", "value": value, "unit": "records/s",
            "n_gpus": args.gpus, "steps": K, "warmup": W, "ms_per_step": head["ms_per_step"],
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "int32" if wl != "sc" else "int64",
            "data": "synthetic", "gpu_launches": 0,
            "config": workload_config(args, wl, head["records_per_step"], 1),
            "cpu_baseline": {"value": value, "unit": "records/s", "cores": 1, "kind": "reference",
                             "host_cores_available": os.cpu_count(),
                             "sample": "%d-record sample of the same synthetic workload per step; the UNMODIFIED reference "
                                       "(baseline/_ref, te_count.py measureTE.parse_bam*) under a stub pysam that yields prebuilt "
                                       "read objects (BAM decode excluded), 1 process, 1 thread -- the reference has no "
                                       "parallelism; index object filled directly (baseline/ref_arm.py), %.1f s outside the "
                                       "timed region" % (head["records_per_step"], R["index_seconds"])},
            "e2e": {"value": value, "unit": "records/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "detail": head}
    line.update(legs)
    print(json.dumps(line))


_W = {}


def _port_worker(a_b):
    a, b = a_b
    from oracle import te_oracle
    c, st = te_oracle.bulk_count(_W["oidx"], _W["paired"], 20, *[x[a:b] for x in _W["cols"]])
    return st["assigned"]


def run_reference_port(args, wl):
    """Fallback of the reference arm when baseline/_ref is absent: the pure-Python port (oracle/te_oracle.py),
    bulk units split over worker processes."""
    import multiprocessing as mp
    from te_counter_b200 import synth
    from oracle import te_oracle
    paired = wl == "bulk_pe"
    cores = os.cpu_count() or 1
    idx = make_index(args.index_scale)
    oidx = te_oracle.Index(idx.chrom_id, idx.L, idx.R, idx.ensg_id, idx.type_code, idx.strand_code, idx.n_ensg, idx.bucket_size)
    n = (args.ref_sample * 4) & ~1
    if wl == "sc":
        r = synth.synth_sc_reads(synth.SEED, idx, n)
        cols = [r[k].tolist() for k in ("start", "end", "chrom", "mapq", "flag", "cell", "umi")]
        cores = 1
    else:
        r = synth.synth_bulk_reads(synth.SEED, idx, n, paired=paired, sort=args.sorted)
        cols = [r[k].tolist() for k in ("start", "end", "chrom", "mapq", "flag")]
    _W.update(cols=cols, oidx=oidx, paired=paired)
    chunk = (n // cores) & ~1
    tasks = [(i * chunk, (i + 1) * chunk if i < cores - 1 else n) for i in range(cores)]
    pool = mp.get_context("fork").Pool(cores) if cores > 1 else None
    times = []
    for i in range(args.warmup + args.steps):
        t = time.perf_counter()
        if wl == "sc":
            te_oracle.sc_count(oidx, 20, True, 10_000_000, 10_000, 1000, *cols)
        elif pool is None:
            _port_worker(tasks[0])
        else:
            pool.map(_port_worker, tasks)
        if i >= args.warmup:
            times.append(time.perf_counter() - t)
    if pool:
        pool.close()
    ms = 1e3 * float(np.mean(times))
    value = n / (ms / 1e3)
    print(json.dumps({"impl": "reference", "metric": "reads_per_sec", "value": value, "unit": "records/s", "n_gpus": args.gpus,
                      "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": args.scaling,
                      "vs_baseline": None, "dtype": "int32", "data": "synthetic", "gpu_launches": 0,
                      "config": workload_config(args, wl, n, 1),
                      "cpu_baseline": {"value": value, "unit": "records/s", "cores": cores, "kind": "port",
                                       "sample": "%d-record sample per step over %d worker process(es); pure-Python restatement "
                                                 "(oracle/te_oracle.py) because baseline/_ref is absent" % (n, cores)},
                      "e2e": {"value": value, "unit": "records/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


# ------------------------------------------------------------------------------ our arm
class Ctx:
    """What every leg needs: ranks, device, engine, index."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.args = args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        from te_counter_b200 import _lib
        self.idx = make_index(args.index_scale)
        self.eng = _lib.Engine(self.local)
        for kv in args.opt:
            k, v = kv.split("=")
            self.eng.set_option(k, int(v))
        self.eng.upload_index(self.idx)
        if self.world > 1:
            from te_counter_b200 import dist as tdist
            tdist.comm_init(self.eng)          # the library's own NCCL communicator: its collectives run inside the library
        self.ext = torch.cuda.ExternalStream(self.eng.stream, device=self.dev)
        self.peak, self.peak_src = load_peaks()
        self._ref = None
        self.outputs = {}

    def keep_outputs(self, leg, **arrays):
        """--dump-outputs: results of a leg's last timed step, as float64 (exact for these integers, all below 2**53)."""
        if self.args.dump_outputs and self.rank == 0:
            for name, a in arrays.items():
                self.outputs[leg + "_" + name] = np.asarray(a, dtype=np.float64).reshape(-1)

    def keep_sc_outputs(self, ensg, cell, count, hit_cell, hit_count, stats, selected, n_triples):
        """The single-cell results; the triples as a sample of at most DUMP_TRIPLES that fits what is left of
        DUMP_BYTES after every other array (3 float64 columns, 24 bytes per triple)."""
        if not (self.args.dump_outputs and self.rank == 0):
            return
        self.keep_outputs("sc", stats=stats, hit_cell=hit_cell, hit_count=hit_count, selected=selected, n_triples=[n_triples])
        used = sum(a.nbytes for a in self.outputs.values())
        k = max(0, min(DUMP_TRIPLES, (DUMP_BYTES - used) // 24))
        self.keep_outputs("sc", **dict(zip(("ensg", "cell", "count"), sample_triples(ensg, cell, count, k))))

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.eng.sync()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        if self.world == 1:
            return float(x)
        t = self.torch.tensor([x], device=self.dev, dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def reference(self):
        if self._ref is None:
            self._ref = reference_setup(self.args) or False
        return self._ref or None


def bulk_leg(C, wl, headline):
    """One bulk workload: device-resident timing, host-buffer e2e, parity.  headline: the long version (full-size
    parity against the C oracle, the reference timed beside it, the file leg)."""
    torch, dist, args, eng, idx = C.torch, C.dist, C.args, C.eng, C.idx
    from te_counter_b200 import _lib, synth
    from te_counter_b200 import dist as tdist
    rank, world, dev = C.rank, C.world, C.dev
    paired = wl == "bulk_pe"
    n_cfg = args.records or CONFIG_RECORDS[wl]
    n_rec = n_cfg if args.scaling == "weak" else n_cfg // world
    n_rec -= n_rec & 1
    reads = synth.synth_bulk_reads(synth.SEED + rank, idx, n_rec, paired=paired, device=dev, as_numpy=False,
                                   shard=(rank, world), sort=args.sorted)
    cols = [reads[k] for k in ("start", "end", "chrom", "mapq", "flag")]
    ptrs = [t.data_ptr() for t in cols]
    torch.cuda.synchronize()
    ext = C.ext
    counts_t = tdist.counts_tensor(eng, idx.n_ensg, dev)

    def step():
        eng.bulk_begin(paired, 20)
        eng.bulk_push_dev(n_rec, *ptrs)
        if world > 1:
            eng.bulk_allreduce()               # ncclAllReduce of the counter block, issued by the library on its stream

    W = max(3, args.warmup)
    for _ in range(W):
        step()
    C.barrier()
    K = args.steps
    k0 = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    k1 = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(C.local)
    sampler.start()
    time.sleep(0.3)
    l0 = eng.launch_count()
    C.barrier()
    t0 = time.time()
    e0.record(ext)
    for k in range(K):
        eng.bulk_begin(paired, 20)
        k0[k].record(ext)
        eng.bulk_push_dev(n_rec, *ptrs)
        k1[k].record(ext)
        if world > 1:
            eng.bulk_allreduce()
    e1.record(ext)
    C.barrier()
    t1 = time.time()
    clocks = sampler.stop(t0, t1)
    launches = eng.launch_count() - l0
    deferred, slow = eng.get_info("last_deferred_units"), eng.get_info("last_slow_units")
    left = eng.get_info("last_left_units")
    kern_ms = float(np.mean([a.elapsed_time(b) for a, b in zip(k0, k1)]))
    ms_step = C.max_over_ranks(e0.elapsed_time(e1)) / K
    value = n_rec * world / (ms_step / 1e3)
    counts, st = eng.bulk_finish()
    C.keep_outputs(wl, counts=counts, stats=st)

    # ---- end to end through the host-buffer ABI (pinned host arrays, H2D + D2H in the timed region)
    parity_full = None
    e2e = None
    host = None
    if not args.no_e2e:
        host = [eng.pinned(n_rec, dt) for dt in (np.int32, np.int32, np.uint16, np.uint8, np.uint8)]
        for h, t in zip(host, cols):
            torch.from_numpy(h.view(np.int16) if h.dtype == np.uint16 else h).copy_(
                t.view(torch.int16) if t.dtype == torch.uint16 else t)
        torch.cuda.synchronize()

        def e2e_step():
            eng.bulk_begin(paired, 20)
            eng.bulk_push(n_rec, *host)
            return eng.bulk_finish()

        for _ in range(2):
            c2, s2 = e2e_step()
        C.barrier()
        Ke = K
        ta = time.perf_counter()
        for _ in range(Ke):
            c2, s2 = e2e_step()
        dt = C.max_over_ranks((time.perf_counter() - ta) / Ke)
        e2e = {"value": n_rec * world / dt, "unit": "records/s", "h2d_bytes_per_step": int(n_rec) * (8 if paired else 12),
               "d2h_bytes_per_step": (idx.n_ensg + _lib.BULK_NSTATS) * 8, "ms_per_step": dt * 1e3, "steps": Ke,
               "api": "tec_bulk_begin + tec_bulk_push(host SoA, pinned) + tec_bulk_finish"}
        if world == 1:
            assert (c2 == counts).all(), "e2e counts differ from the device-resident run"
        # ---- full-size parity: the whole workload against the C restatement of the reference's loop
        #      (oracle/te_oracle_c.c, the checker), all host cores
        if rank == 0 and world == 1 and not args.no_cpu:
            from oracle import te_oracle_c
            tc0 = time.perf_counter()
            cidx = te_oracle_c.Index(idx.chrom_id, idx.L, idx.R, idx.ensg_id, idx.type_code, idx.n_chrom, idx.n_ensg,
                                     idx.bucket_size)
            fc, fs = te_oracle_c.bulk_count(cidx, paired, 20, *host)
            tc1 = time.perf_counter()
            full_ok = bool((fc == counts).all() and fs[:5].tolist() == [int(x) for x in st[:5]])
            parity_full = {"records": int(n_rec), "bit_exact": full_ok, "seconds": tc1 - tc0, "threads": os.cpu_count(),
                           "c_port_records_per_s": n_rec / (tc1 - tc0),
                           "checker": "oracle/te_oracle_c.c (C restatement of te_count.py's bulk loop, pinned through "
                                      "oracle/te_oracle.py and tests/golden)"}
            assert full_ok, "full-size counts differ from the C oracle"
    del host

    # ---- CPU baseline + parity on a bounded prefix (rank 0, N = 1): the unmodified reference (baseline/_ref) beside
    #      the pure-Python port; the CUDA result of the same prefix must equal both
    cpu = None
    parity = None
    if rank == 0 and world == 1 and not args.no_cpu:
        from oracle import te_oracle
        ns = min(n_rec, args.cpu_sample if headline else args.cpu_sample // 3) & ~1
        sample = [t[:ns].cpu().numpy() for t in cols]
        sample[2] = sample[2].view(np.uint16)
        sample = [np.ascontiguousarray(a) for a in sample]
        eng.bulk_begin(paired, 20)
        eng.bulk_push(ns, *sample)
        gc, gs = eng.bulk_finish()
        oidx = te_oracle.Index(idx.chrom_id, idx.L, idx.R, idx.ensg_id, idx.type_code, idx.strand_code,
                               idx.n_ensg, idx.bucket_size)
        np_ = min(ns, 200_000) & ~1
        lists = [a[:np_].tolist() for a in sample]
        ta = time.perf_counter()
        oc, os_ = te_oracle.bulk_count(oidx, paired, 20, *lists)
        tb = time.perf_counter()
        port = {"value": np_ / (tb - ta), "unit": "records/s", "cores": 1, "kind": "port", "sample_records": np_,
                "what": "oracle/te_oracle.py, pure-Python restatement of te_count.py's loop"}
        if np_ < ns:
            eng.bulk_begin(paired, 20)
            eng.bulk_push(np_, *[np.ascontiguousarray(a[:np_]) for a in sample])
            pc, ps = eng.bulk_finish()
        else:
            pc, ps = gc, gs
        ok = (pc.tolist() == oc and int(ps[_lib.BS_UNITS]) + 1 == os_["total_reads"]
              and int(ps[_lib.BS_ASSIGNED]) == os_["assigned"] and int(ps[_lib.BS_LOWQ]) == os_["lowq"]
              and int(ps[_lib.BS_BADCHROM]) == os_["badchrom"] and int(ps[_lib.BS_QCFAIL]) == os_["qcfail"])
        parity = {"sample_records": np_, "bit_exact": bool(ok), "checker": "oracle/te_oracle.py"}
        assert ok, "counts differ from the oracle on the sample"
        R = C.reference()
        if R is not None:
            dt, res, total = reference_time_bulk(R, paired, sample)
            ref_ok = [res[n] for n in idx.names] == gc.tolist() and total == int(gs[_lib.BS_UNITS]) + 1
            parity["reference_sample_records"] = ns
            parity["reference_bit_exact"] = bool(ref_ok)
            assert ref_ok, "counts differ from the unmodified reference on the sample"
            cpu = {"value": ns / dt, "unit": "records/s", "cores": 1, "kind": "reference",
                   "host_cores_available": os.cpu_count(),
                   "sample": "first %d records of this workload through the UNMODIFIED reference (baseline/_ref: "
                             "measureTE.%s under a stub pysam, read objects prebuilt, BAM decode excluded), 1 process, "
                             "1 thread as the reference is; index object filled directly in %.1f s outside the timed "
                             "region" % (ns, "parse_bampe" if paired else "parse_bamse", R["index_seconds"]),
                   "port_python": port,
                   "port_c_threads": None if not parity_full else {"value": parity_full["c_port_records_per_s"], "unit": "records/s",
                                                                   "cores": os.cpu_count(), "kind": "port",
                                                                   "what": "oracle/te_oracle_c.c on the full workload (the parity_full run)"}}
        else:
            cpu = dict(port, host_cores_available=os.cpu_count(),
                       sample="first %d records of this workload; baseline/_ref absent, so the pure-Python restatement "
                              "(oracle/te_oracle.py, pinned to the unmodified reference by tests/golden), single thread" % np_)

    bpr = BYTES_PER_RECORD[wl] + INDEX_BYTES_PER_FEATURE * idx.n_features / float(n_rec)
    achieved = n_rec * bpr / (kern_ms / 1e3) / 1e9
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "r02_bulk_ncu_traffic.json")
    if os.path.exists(tp):
        t = json.load(open(tp))
        if paired:
            traffic = (t["dram_bytes_read"] + t["dram_bytes_write"]) / t["records_per_launch"] * n_rec
            traffic_src = t.get("source")
        elif "bulk_se" in t:
            traffic = (t["bulk_se"]["dram_bytes_read"] + t["bulk_se"]["dram_bytes_write"]) / t["bulk_se"]["records_per_step"] * n_rec
            traffic_src = t["bulk_se"].get("source")
    leg = {"value": value, "unit": "records/s", "ms_per_step": ms_step, "steps": K, "warmup": W,
           "config": workload_config(args, wl, n_rec, world), "gpu_launches": int(launches), "dtype": "int32",
           "roofline": {"bound": "hbm", "achieved": achieved, "peak": C.peak, "unit": "GB/s",
                        "frac": achieved / C.peak, "traffic": traffic, "peak_source": C.peak_src, "traffic_source": traffic_src,
                        "kernel": "bulk2_fast_kernel<%s> + bulk2_pair_kernel / bulk2_second_kernel (deferred units) + bulk_slow_kernel (exact search)"
                                  % ("paired" if paired else "single"),
                        "cell_table_bytes": eng.get_info("stab_bytes"), "deferred_units_per_launch": deferred,
                        "left_units_per_launch": left,
                        "slow_units_per_launch": slow, "kernel_ms": kern_ms, "algorithmic_bytes_per_record": bpr},
           "cpu_baseline": cpu, "e2e": e2e, "clocks": clocks, "parity": parity, "parity_full": parity_full,
           "stats": {"units": int(st[0]), "assigned": int(st[1]), "lowq": int(st[2]), "badchrom": int(st[3]),
                     "qcfail": int(st[4]), "counts_sum": int(counts.sum())}}
    # ---- the same count from a BAM FILE on disk through the public call (measureTE.parse_bampe / parse_bamse)
    if headline and rank == 0 and world == 1 and not args.no_e2e and args.file_records > 0:
        try:
            leg["from_file"] = file_leg(eng, idx, paired, args.file_records)
        except Exception as e:                          # noqa: BLE001 -- an extra leg: report, do not lose the bench line
            leg["from_file"] = {"error": "%s: %s" % (type(e).__name__, e)}
    del reads, cols
    torch.cuda.empty_cache()
    return leg


def sc_leg(C, headline):
    """BASELINE.json configs[4]: one step = tec_sc_begin + tec_sc_push_dev (filter, whitelist, compaction)
    [+ exchange by cell over NCCL] + tec_sc_finalize (UMI collapse, Part-2 rule, overlap, tally) + tec_sc_select."""
    torch, dist, args, eng, idx = C.torch, C.dist, C.args, C.eng, C.idx
    from te_counter_b200 import _lib, synth
    from te_counter_b200 import dist as tdist
    rank, world, dev = C.rank, C.world, C.dev
    n_cfg = args.records or (CONFIG_RECORDS["sc"] if world == 1 else SC_RECORDS_MULTI)
    n_rec = n_cfg if args.scaling == "weak" else n_cfg // world
    n_wl, maxcells, pad, bundle_keys = 100_000, 10_000, 1000, 10_000_000
    # this rank's slice of the coordinate-sorted file: `parts` consecutive genome slices
    parts = max(1, (n_rec + 124_999_999) // 125_000_000)
    names = ("start", "end", "chrom", "mapq", "flag", "cell", "umi")
    chunks = {k: [] for k in names}
    for p in range(parts):
        n_p = n_rec // parts + (1 if p < n_rec % parts else 0)
        r = synth.synth_sc_reads(synth.SEED, idx, n_p, n_whitelist=n_wl, device=dev, as_numpy=False,
                                 part=(rank * parts + p, parts * world))
        for k in names:
            chunks[k].append(r[k])
        del r
    cols = [torch.cat(chunks[k]) if parts > 1 else chunks[k][0] for k in names]
    del chunks
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    ptrs = [t.data_ptr() for t in cols]
    ext = C.ext
    strand = True
    phase = {}

    def step():
        ta = time.perf_counter()
        eng.sc_begin(20, strand, n_wl)
        eng.sc_push_dev(n_rec, *ptrs)
        if os.environ.get("TEC_DIST_TIMING"):
            eng.sync()
        tb = time.perf_counter()
        if world > 1:
            tdist.sc_exchange_by_cell(eng, dev)             # all-to-all by cell over NCCL
        tc = time.perf_counter()
        nt, nh = eng.sc_finalize(bundle_keys, maxcells, pad)
        if world > 1:
            nt = eng.sc_allgather_triples()                 # every rank ends with the job's triples (NCCL inside the library)
        sel = eng.sc_select(maxcells, nh)
        td = time.perf_counter()
        phase.update(push=tb - ta, exchange=tc - tb, finalize=td - tc)
        return nt, nh, sel

    W = max(3, args.warmup) if headline else 3
    K = args.steps
    for _ in range(W):
        step()
    C.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(C.local)
    sampler.start()
    time.sleep(0.3)
    l0 = eng.launch_count()
    C.barrier()
    t0 = time.time()
    e0.record(ext)
    for _ in range(K):
        nt, nh, sel = step()
    e1.record(ext)
    C.barrier()
    t1 = time.time()
    clocks = sampler.stop(t0, t1)
    launches = eng.launch_count() - l0
    ms_step = e0.elapsed_time(e1) / K
    if world > 1:
        # the exchange runs on torch's stream and the step has host synchronisation points: take the wall clock
        # of the timed region (barrier + synchronize on both sides), max over ranks
        ms_step = C.max_over_ranks(max(ms_step, (t1 - t0) * 1e3 / K))
    value = n_rec * world / (ms_step / 1e3)
    ensg, cell, count, hcell, hcount, st = eng.sc_fetch(nt, nh)
    C.keep_sc_outputs(ensg, cell, count, hcell, hcount, st, sel, nt)
    # dense matrix rows of sc_save_result formatted on the device (te_count.py:744-754): size and rate
    matrix_text = None
    if world == 1 and len(sel) and headline:
        bcs = ["%016d-1" % int(c) for c in sel.tolist()]
        eng.sc_matrix_text(sel, bcs)                                    # warm (allocations)
        ta = time.perf_counter()
        n_text = eng.sc_matrix_text(sel, bcs)
        tb = time.perf_counter()
        matrix_text = {"rows": int(len(sel)), "columns": int(idx.n_ensg), "bytes": int(n_text), "ms": (tb - ta) * 1e3,
                       "GBps_written": n_text / (tb - ta) / 1e9,
                       "what": "tec_sc_matrix_text, wall clock around the call (sort of the triples by row + text kernel)"}
    no_e2e = args.no_e2e or world > 1
    no_cpu = args.no_cpu or world > 1

    e2e = None
    if not no_e2e:
        ne = min(n_rec, args.sc_e2e_records)
        dts = (np.int32, np.int32, np.uint16, np.uint8, np.uint8, np.uint32, np.uint64)
        host = [eng.pinned(ne, dt) for dt in dts]
        for h, t in zip(host, cols):
            hv = h.view(np.int16) if h.dtype == np.uint16 else h.view(np.int32) if h.dtype == np.uint32 else \
                h.view(np.int64) if h.dtype == np.uint64 else h
            tv = t.view(torch.int16) if t.dtype == torch.uint16 else t.view(torch.int32) if t.dtype == torch.uint32 else \
                t.view(torch.int64) if t.dtype == torch.uint64 else t
            torch.from_numpy(hv).copy_(tv[:ne])
        torch.cuda.synchronize()

        def e2e_step():
            eng.sc_begin(20, strand, n_wl)
            eng.sc_push(ne, *host)
            a, b = eng.sc_finalize(bundle_keys, maxcells, pad)
            out = eng.sc_fetch(a, b, pinned=True)
            return out, eng.sc_select(maxcells, b)

        e2e_step()
        Ke = K
        ta = time.perf_counter()
        for _ in range(Ke):
            out2, sel2 = e2e_step()
        dt = (time.perf_counter() - ta) / Ke
        e2e = {"value": ne / dt, "unit": "records/s", "h2d_bytes_per_step": int(ne) * 24,
               "d2h_bytes_per_step": int(len(out2[0]) * 16 + len(out2[3]) * 12 + _lib.SC_NSTATS * 8 + len(sel2) * 4),
               "ms_per_step": dt * 1e3, "steps": Ke, "records": int(ne),
               "note": None if ne == n_rec else "host-buffer leg on the first %d records of the workload (pinned host memory: "
                                                "24 B per record)" % ne,
               "api": "tec_sc_begin + tec_sc_push(host SoA, pinned) + tec_sc_finalize + tec_sc_fetch + tec_sc_select"}
        if ne == n_rec:
            assert (out2[0] == ensg).all() and (out2[2] == count).all(), "e2e triples differ from the device-resident run"
        del host

    cpu = None
    parity = None
    if not no_cpu and rank == 0:
        from oracle import te_oracle
        ns = min(n_rec, (args.cpu_sample if headline else args.cpu_sample // 3))
        sample = [t[:ns].cpu().numpy() for t in cols]
        sample[2] = sample[2].view(np.uint16)
        sample[5] = sample[5].view(np.uint32)
        sample[6] = sample[6].view(np.uint64)
        sample = [np.ascontiguousarray(a) for a in sample]
        eng.sc_begin(20, strand, n_wl)
        eng.sc_push(ns, *sample)
        a, b = eng.sc_finalize(bundle_keys, maxcells, pad)
        g_ensg, g_cell, g_count, g_hc, g_hn, g_st = eng.sc_fetch(a, b)
        oidx = te_oracle.Index(idx.chrom_id, idx.L, idx.R, idx.ensg_id, idx.type_code, idx.strand_code,
                               idx.n_ensg, idx.bucket_size)
        lists = [x.tolist() for x in sample]
        ta = time.perf_counter()
        out = te_oracle.sc_count(oidx, 20, strand, bundle_keys, maxcells, pad, *lists)
        tb = time.perf_counter()
        got = {(int(e), int(c)): int(v) for e, c, v in zip(g_ensg, g_cell, g_count)}
        ok = got == out["triples"] and list(zip(g_hc.tolist(), g_hn.tolist())) == sorted(out["cell_hits"]) and \
            int(g_st[_lib.SS_VALID]) == out["stats"]["valid"] and int(g_st[_lib.SS_ASSIGNED]) == out["stats"]["assigned"]
        parity = {"sample_records": ns, "bit_exact": bool(ok), "checker": "oracle/te_oracle.py"}
        assert ok, "single-cell result differs from the oracle on the sample"
        port = {"value": ns / (tb - ta), "unit": "records/s", "cores": 1, "kind": "port", "sample_records": ns,
                "what": "oracle/te_oracle.py, pure-Python restatement of sc_parse_bamse"}
        R = C.reference()
        if R is not None:
            nr = min(ns, 200_000)
            dt, res, mte = reference_time_sc(R, [a[:nr] for a in sample], n_wl, strand, maxcells)
            cpu = {"value": nr / dt, "unit": "records/s", "cores": 1, "kind": "reference", "host_cores_available": os.cpu_count(),
                   "sample": "first %d records of this workload through the UNMODIFIED reference (baseline/_ref: "
                             "measureTE.sc_parse_bamse under a stub pysam, read objects prebuilt, load_genome bound to a no-op on "
                             "the instance), 1 process, 1 thread" % nr,
                   "port_python": port}
        else:
            cpu = dict(port, host_cores_available=os.cpu_count(),
                       sample="first %d records; baseline/_ref absent, so the pure-Python restatement" % ns)

    # ---- large parity check: real 1e7-key bundles, against the C++ restatement (oracle/te_oracle_sc.cpp)
    parity_full = None
    if not no_cpu and rank == 0 and args.sc_parity_records > 0:
        from oracle import te_oracle_c
        nb = min(n_rec, args.sc_parity_records)
        # a whole-genome file of its own (a prefix of the timed, coordinate-sorted workload would cover one corner of the
        # genome and too few distinct keys for a second bundle)
        rp = synth.synth_sc_reads(synth.SEED + 1, idx, nb, n_whitelist=n_wl, device=dev, as_numpy=False)
        big = [rp[k].cpu().numpy() for k in names]
        del rp
        big[2] = big[2].view(np.uint16)
        big[5] = big[5].view(np.uint32)
        big[6] = big[6].view(np.uint64)
        big = [np.ascontiguousarray(a) for a in big]
        eng.sc_begin(20, strand, n_wl)
        for a0 in range(0, nb, 1 << 24):
            eng.sc_push(min(nb, a0 + (1 << 24)) - a0, *[a[a0:a0 + (1 << 24)] for a in big])
        a, b = eng.sc_finalize(bundle_keys, maxcells, pad)
        g_ensg, g_cell, g_count, g_hc, g_hn, g_st = eng.sc_fetch(a, b)
        ta = time.perf_counter()
        out = te_oracle_c.sc_count((idx.chrom_id, idx.L, idx.R, idx.ensg_id, idx.type_code, idx.strand_code), idx.n_chrom,
                                   idx.bucket_size, 20, strand, bundle_keys, maxcells, pad, *big)
        tb = time.perf_counter()
        o_ensg, o_cell, o_count = out["triples_arrays"]
        ok = (len(o_ensg) == len(g_ensg) and (o_ensg == g_ensg).all() and (o_cell == g_cell).all() and (o_count == g_count).all()
              and sorted(out["cell_hits"]) == list(zip(g_hc.tolist(), g_hn.tolist()))
              and all(int(g_st[k]) == out["stats"][f] for k, f in (
                  (_lib.SS_INVALID_BARCODE, "invalid_barcode"), (_lib.SS_ALREADY_SEEN, "already_seen"), (_lib.SS_LOWQ, "lowq"),
                  (_lib.SS_QCFAIL, "qcfail"), (_lib.SS_VALID, "valid"), (_lib.SS_ASSIGNED, "assigned"),
                  (_lib.SS_RAW_BARCODES, "raw_barcodes"), (_lib.SS_BUNDLES, "n_bundles"))))
        parity_full = {"records": int(nb), "bundles": out["stats"]["n_bundles"], "triples": int(len(o_ensg)), "bit_exact": bool(ok),
                       "seconds": tb - ta, "c_port_records_per_s": nb / (tb - ta),
                       "checker": "oracle/te_oracle_sc.cpp (C++ restatement of sc_parse_bamse, checked against "
                                  "oracle/te_oracle.py and tests/golden)"}
        assert ok, "single-cell result differs from the C++ oracle"
        del big

    bpr = BYTES_PER_RECORD["sc"] + INDEX_BYTES_PER_FEATURE * idx.n_features / float(n_rec)
    achieved = n_rec * bpr / (ms_step / 1e3) / 1e9
    if world > 1:
        dist.barrier()
    leg = {"value": value, "unit": "records/s", "ms_per_step": ms_step, "steps": K, "warmup": W, "dtype": "int64",
           "config": dict(workload_config(args, "sc", n_rec, world), n_whitelist=n_wl, maxcells=maxcells, strand=strand,
                          bundle_keys=bundle_keys),
           "gpu_launches": int(launches),
           "roofline": {"bound": "hbm", "achieved": achieved, "peak": C.peak, "unit": "GB/s", "frac": achieved / C.peak,
                        "traffic": None, "peak_source": C.peak_src,
                        "kernel": "whole sc step (sort passes dominate; see profiles/)", "kernel_ms": ms_step,
                        "sc_cell_table": bool(eng.get_info("has_sc_stab")), "sc_cell_table_bytes": eng.get_info("sc_stab_bytes"),
                        "algorithmic_bytes_per_record": bpr},
           "cpu_baseline": cpu, "e2e": e2e, "clocks": clocks, "parity": parity, "parity_full": parity_full,
           "matrix_text": matrix_text,
           "collective": None if world == 1 else "issued by the library over its own NCCL communicator: tec_sc_exchange (all-to-all of the survivors by cell, grouped send / receive), "
                                                   "all-reduces inside tec_sc_finalize, tec_sc_allgather_triples; all inside the timed step",
           "stats": {"units": int(st[_lib.SS_UNITS]), "survivors": int(st[_lib.SS_SURVIVORS]),
                     "segments": int(st[_lib.SS_SEGMENTS]), "bundles": int(st[_lib.SS_BUNDLES]),
                     "valid": int(st[_lib.SS_VALID]), "assigned": int(st[_lib.SS_ASSIGNED]),
                     "triples": int(nt), "hit_cells": int(nh), "selected": int(len(sel))}}
    if os.environ.get("TEC_DIST_TIMING"):
        leg["phase_s_last_step"] = phase
        leg["exchange_s_total"] = dict(tdist.TIMING)
    del cols
    torch.cuda.empty_cache()
    eng.trim()
    return leg


def run_ours(args):
    C = Ctx(args)
    wl = args.workload
    t_start = time.time()
    if wl == "sc":
        head = sc_leg(C, True)
        legs = {}
    else:
        head = bulk_leg(C, "bulk_pe" if wl == "all" else wl, True)
        legs = {}
        if wl == "all":
            legs["bulk_se"] = bulk_leg(C, "bulk_se", False)
            legs["sc"] = sc_leg(C, False)
    line = {"metric": "reads_per_sec", "value": head["value"], "unit": "records/s", "n_gpus": C.world, "steps": head["steps"],
            "warmup": head["warmup"], "ms_per_step": head["ms_per_step"], "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": head["dtype"], "data": "synthetic"}
    for k in ("config", "gpu_launches", "roofline", "cpu_baseline", "e2e", "clocks", "parity", "parity_full", "stats",
              "from_file", "matrix_text", "collective"):
        if k in head:
            line[k] = head[k]
    line.update(legs)
    line["bench_seconds"] = time.time() - t_start
    if args.dump_outputs and C.rank == 0:
        line["dump_outputs"] = write_outputs(args.dump_outputs, C.outputs)
    if C.rank == 0:
        print(json.dumps(line))
    C.eng.close()
    if C.world > 1:
        C.dist.destroy_process_group()


def file_leg(eng, idx, paired, n_records, sc=None):
    """BAM file on disk -> counts through measureTE (wall clock around the public call, best of 3), per decoder.
    sc = dict(strand, maxcells) for the single-cell call."""
    import logging
    import tempfile
    import te_counter_b200
    from te_counter_b200 import bam as pybam, reads as treads, synth_bam
    log = logging.getLogger("bench.file_leg")
    log.addHandler(logging.NullHandler())
    log.propagate = False
    tmp = tempfile.mkdtemp(prefix="tec_bench_")
    path = os.path.join(tmp, "synth.bam")
    try:
        wlf = os.path.join(tmp, "whitelist.txt")
        size = synth_bam.write(path, n_records & ~1, "sc" if sc else "pe" if paired else "se", whitelist=wlf)
        mte = te_counter_b200.measureTE("bench", 20)
        mte.genome = idx
        mte.all_feature_names = idx.names
        mte._engine_obj = eng
        mte._index_on_device = True
        mte.load_genome = lambda: None                  # (sc_parse_bamse reloads the .glb; the synthetic index has none)
        out = {"records": n_records & ~1, "file_bytes": size, "host_cores": os.cpu_count(),
               "api": "measureTE.sc_parse_bamse(file)" if sc else "measureTE.parse_bampe(file)" if paired else "measureTE.parse_bamse(file)"}
        results = {}
        old = os.environ.get("TEC_BAM_DECODER")
        try:
            for dec, key in (("gpu", "device_decoder"), ("native", "host_decoder")):
                os.environ["TEC_BAM_DECODER"] = dec
                best = None
                for _ in range(3):
                    ta = time.perf_counter()
                    if sc:
                        r = mte.sc_parse_bamse(path, whitelistfilename=wlf, strand=sc["strand"], log=log, label="bench",
                                               maxcells=sc["maxcells"])
                        res = (r.ensg.tolist(), r.cell.tolist(), r.count.tolist(), dict(mte.barcodes))
                    else:
                        res = (mte.parse_bampe if paired else mte.parse_bamse)(path, log=log)
                    dt = time.perf_counter() - ta
                    best = dt if best is None else min(best, dt)
                results[dec] = res
                out[key] = {"records_per_s": (n_records & ~1) / best, "seconds": best}
        finally:
            if old is None:
                os.environ.pop("TEC_BAM_DECODER", None)
            else:
                os.environ["TEC_BAM_DECODER"] = old
        out["decoders_agree"] = results["gpu"] == results["native"]
        assert out["decoders_agree"], "device and host BAM decoders disagree"
        f = pybam.AlignmentFile(path, "r")
        b = treads.Batch(200000, sc=bool(sc))
        ta = time.perf_counter()
        if sc:
            treads.fill_sc(b, f, treads.ChromMap(idx.chrom_keys), treads.Whitelist(wlf), 20)
        else:
            treads.fill_bulk(b, f, treads.ChromMap(idx.chrom_keys), paired, 20)
        out["python_packing"] = {"records_per_s": b.n / (time.perf_counter() - ta), "sample_records": b.n, "cores": 1,
                                 "what": "bam.py + reads.fill_*, the stand-in for the reference's pysam loop"}
        f.close()
        return out
    finally:
        import shutil
        shutil.rmtree(tmp, ignore_errors=True)


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
