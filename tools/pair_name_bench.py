"""Paired end by read name on one GPU: a coordinate-sorted synthetic BAM (te_counter_b200.synth_bam --sorted) through
parse_bampe(pairing='name'), and a name-collated copy of the same pairs through parse_bampe(pairing='index').

The collated copy is made on the host from the sorted file: every synthetic record has the same size, so the records
are inflated, paired by their QNAME with numpy (same rule: primary, exactly one of 0x40 / 0x80) and written read1, read2
in pair order.  The host clock is taken around each parse_bampe, which ends in a device synchronise (tec_bulk_finish);
the engine and the index upload are made before the clock starts.  Reported: the median of --steps timed calls after
--warmup calls for each arm, the pairing stage's device time (tec_get_info "bulk_name_ms") and pending peak of the
last call, and whether both arms give identical counts and statistics.  Needs a GPU; prints one JSON line and writes it
to --out-dir.

    python tools/pair_name_bench.py --records 16000000 --out-dir profiles/
"""
import argparse
import json
import logging
import multiprocessing
import os
import struct
import subprocess
import sys
import tempfile
import time
import zlib
from concurrent.futures import ProcessPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
T0 = time.perf_counter()


def inflate_bgzf(path):
    """the inflated bytes of a BGZF file, block by block (BSIZE of each header gives the next block)"""
    raw = memoryview(open(path, "rb").read())
    out, p = [], 0
    while p < len(raw):
        xlen = struct.unpack_from("<H", raw, p + 10)[0]
        bsize = struct.unpack_from("<H", raw, p + 16)[0] + 1               # the BC subfield comes first (synth_bam._bgzf)
        out.append(zlib.decompress(raw[p + 12 + xlen:p + bsize - 8], -15))
        p += bsize
    return b"".join(out)


def log(msg):
    print("[pair_name_bench %.0f s] %s" % (time.perf_counter() - T0, msg), file=sys.stderr, flush=True)


def collated_copy(src, dst):
    """The pairs of the coordinate-sorted synthetic file src, each written read1 then read2, into dst.  Returns the
    number of pairs."""
    from te_counter_b200 import synth_bam
    data = inflate_bgzf(src)
    head = len(synth_bam.header_bytes(synth_bam.HG38))
    size = 4 + struct.unpack_from("<i", data, head)[0]
    m = np.frombuffer(data, dtype=np.uint8, offset=head).reshape(-1, size)
    flag = m[:, 18].astype(np.uint16) | (m[:, 19].astype(np.uint16) << 8)
    digits = m[:, 44:59].astype(np.int64) - 48
    ids = digits @ (10 ** np.arange(14, -1, -1, dtype=np.int64))
    role = np.where((flag & 1) & ((flag & 0x900) == 0), np.where((flag & 0xC0) == 0x40, 1, np.where((flag & 0xC0) == 0x80, 2, 0)), 0)
    keep = np.flatnonzero(role > 0)
    order = keep[np.lexsort((role[keep], ids[keep]))]
    i_ = ids[order]
    first = np.flatnonzero((i_[:-1] == i_[1:]) & (role[order[:-1]] == 1) & (role[order[1:]] == 2))
    rows = np.empty(2 * len(first), dtype=np.int64)
    rows[0::2], rows[1::2] = order[first], order[first + 1]
    body = m[rows]
    per = max(1, (64 << 20) // size)                                        # records per deflate job
    pieces = [body[i:i + per].tobytes() for i in range(0, len(body), per)]
    log("collated %d pairs; deflating" % len(first))
    ctx = multiprocessing.get_context("forkserver")
    with open(dst, "wb") as fh, ProcessPoolExecutor(os.cpu_count() or 1, mp_context=ctx) as ex:
        fh.write(synth_bam._bgzf(synth_bam.header_bytes(synth_bam.HG38)))
        for comp in ex.map(synth_bam._deflate_chunk, pieces):
            fh.write(comp)
        fh.write(synth_bam._bgzf(b""))
    return len(first)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=16000000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out-dir", default=".")
    ap.add_argument("--dir", default=None, help="where the BAMs are written (default: a temporary directory)")
    a = ap.parse_args()
    import torch
    if not torch.cuda.device_count():
        raise SystemExit("no GPU: nothing to measure")
    import te_counter_b200
    from te_counter_b200 import _lib, synth, synth_bam
    work = a.dir or tempfile.mkdtemp(prefix="pair_name_bench_")
    sorted_bam, collated_bam = os.path.join(work, "sorted.bam"), os.path.join(work, "collated.bam")
    t0 = time.perf_counter()
    size = synth_bam.write(sorted_bam, records=a.records, mode="pe", sorted_pe=True)
    log("wrote %s (%d bytes)" % (sorted_bam, size))
    pairs = collated_copy(sorted_bam, collated_bam)
    log("wrote %s" % collated_bam)
    prep_s = time.perf_counter() - t0
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    quiet = logging.getLogger("pair_name_bench")
    quiet.addHandler(logging.NullHandler())
    quiet.propagate = False
    idx = synth.synth_index()
    mte = te_counter_b200.measureTE("pair_name_bench", 20, device=0)
    mte.genome = idx
    mte.all_feature_names = idx.names
    eng = mte._engine()
    os.environ["TEC_BAM_DECODER"] = "gpu"
    out = {"records_in_file": a.records, "file_bytes": size, "collated_pairs": pairs, "gpus": smi.strip().splitlines(),
           "steps": a.steps, "warmup": a.warmup, "prep_s": prep_s}
    results = {}
    for arm, path, pairing in (("name", sorted_bam, "name"), ("index_collated", collated_bam, "index")):
        times = []
        for step in range(a.warmup + a.steps):
            t0 = time.perf_counter()
            res = mte.parse_bampe(path, log=quiet, pairing=pairing)
            if step >= a.warmup:
                times.append(time.perf_counter() - t0)
            log("%s step %d: %.3f s" % (arm, step, time.perf_counter() - t0))
        _, st = eng.bulk_finish()
        results[arm] = (res, st.tolist(), mte.total_reads)
        out[arm] = {"median_s": float(np.median(times)), "times_s": times, "total_reads": mte.total_reads}
        if pairing == "name":
            out[arm]["bulk_name_ms"] = eng.get_info("bulk_name_ms")
            out[arm]["pending_peak"] = eng.get_info("bulk_name_pending_peak")
            out[arm]["excluded"] = eng.get_info("bulk_name_excluded")
            out[arm]["no_mate"] = int(st[_lib.BS_NO_MATE]) - out[arm]["excluded"]
            out[arm]["bam_info_us"] = getattr(mte, "_bam_info", None)
    n, c = results["name"], results["index_collated"]
    out["identical_counts"] = n[0] == c[0]
    out["identical_stats"] = n[1][:7] == c[1][:7] and n[2] == c[2]
    line = json.dumps(out)
    print(line)
    os.makedirs(a.out_dir, exist_ok=True)
    with open(os.path.join(a.out_dir, "pair_name_bench.json"), "w") as fh:
        fh.write(line + "\n")
    if not (out["identical_counts"] and out["identical_stats"]):
        raise SystemExit("the two arms differ")


if __name__ == "__main__":
    main()
