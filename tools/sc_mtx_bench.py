"""Times the 10x-style Matrix Market output of the single-cell path (measureTE.sc_save_mtx) on one GPU:

    python tools/sc_mtx_bench.py [--records 200000000] [--threads N] [--json out.json]

One seeded run of the shape of bench.py's single-cell workload (hg38-like index, 100 k-barcode whitelist, --maxcells
10000, strand on), then, on the same triples and the same 10 000 selected cells:
  * tec_sc_matrix_mtx: host clock around the call, which ends in a device synchronise, after a warm-up call;
  * the text's non-zeros and bytes, and the device-to-host streaming of it (tec_sc_matrix_read in 16 MiB pieces);
  * gzip of that text at the thread count used (te_counter_b200/mtx.py);
  * sc_save_mtx and sc_save_result wall time, each writing to a temporary directory;
  * the device text against the host formatter (mtx.mtx_text) on the same triples, byte for byte;
  * the GPU's name and power limit, read in the same process.
Outputs go to a temporary directory that is removed at the end; the JSON goes to stdout and to --json.
"""
import argparse
import io
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


class _Log:
    def info(self, *a):
        pass

    warning = info


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        name, power = [x.strip() for x in out.split(",")[:2]]
        return {"gpu": name, "power_limit": power}
    except Exception as e:                                     # report, do not guess
        return {"gpu": None, "power_limit": None, "nvidia_smi_error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=200_000_000)
    ap.add_argument("--threads", type=int, default=0)
    ap.add_argument("--json")
    args = ap.parse_args()
    import numpy as np
    import torch
    from te_counter_b200 import _lib, mtx, synth
    from te_counter_b200.te_count import ScResult, measureTE

    threads = args.threads or mtx.default_threads()
    n_wl, maxcells, pad, bundle_keys = 100_000, 10_000, 1000, 10_000_000
    dev = torch.device("cuda", 0)
    idx = synth.synth_index()
    eng = _lib.Engine(0)
    eng.upload_index(idx)
    parts = max(1, (args.records + 124_999_999) // 125_000_000)       # bench.py's genome slices
    names = ("start", "end", "chrom", "mapq", "flag", "cell", "umi")
    chunks = {k: [] for k in names}
    for p in range(parts):
        n_p = args.records // parts + (1 if p < args.records % parts else 0)
        r = synth.synth_sc_reads(synth.SEED, idx, n_p, n_whitelist=n_wl, device=dev, as_numpy=False, part=(p, parts))
        for k in names:
            chunks[k].append(r[k])
        del r
    cols = [torch.cat(chunks[k]) if parts > 1 else chunks[k][0] for k in names]
    del chunks
    torch.cuda.synchronize()
    eng.sc_begin(20, True, n_wl)
    eng.sc_push_dev(args.records, *[t.data_ptr() for t in cols])
    nt, nh = eng.sc_finalize(bundle_keys, maxcells, pad)
    ensg, cell, count, hcell, hcount, st = eng.sc_fetch(nt, nh)
    sel = eng.sc_select(maxcells, nh)
    del cols
    torch.cuda.empty_cache()

    eng.sc_matrix_mtx(sel)                                             # warm (allocations, sort temporaries)
    t0 = time.perf_counter()
    nnz, n_bytes = eng.sc_matrix_mtx(sel)
    t_dev = time.perf_counter() - t0
    buf = io.BytesIO()
    t0 = time.perf_counter()
    eng.sc_matrix_write(buf, n_bytes, chunk=mtx.PIECE)
    t_d2h = time.perf_counter() - t0
    text = buf.getvalue()
    del buf
    tmp = tempfile.mkdtemp(prefix="sc_mtx_bench_")
    try:
        gz = os.path.join(tmp, "m.gz")
        t0 = time.perf_counter()
        mtx.write_gzip(gz, lambda fh: fh.write(text), threads)
        t_gz = time.perf_counter() - t0
        gz_bytes = os.path.getsize(gz)
        os.unlink(gz)
        t0 = time.perf_counter()
        host = mtx.mtx_text(idx.n_ensg, ensg, cell, count, sel)
        t_host = time.perf_counter() - t0
        same = host == text
        del host

        barcodes = ["%016d-1" % i for i in range(n_wl)]
        res = ScResult(idx.names, barcodes, ensg, cell, count)
        mte = measureTE(tmp, 20, device=0)
        mte._engine_obj = eng
        mte._sc_hit = (hcell, hcount)
        mte.barcodes = {barcodes[c]: h for c, h in zip(hcell.tolist(), hcount.tolist())}
        t0 = time.perf_counter()
        mte.sc_save_mtx(res, os.path.join(tmp, "mtx"), maxcells, log=_Log(), threads=threads)
        t_mtx = time.perf_counter() - t0
        mtx_dir_bytes = sum(os.path.getsize(os.path.join(tmp, "mtx", f)) for f in os.listdir(os.path.join(tmp, "mtx")))
        t0 = time.perf_counter()
        mte.sc_save_result(res, os.path.join(tmp, "dense.tsv"), maxcells, log=_Log())
        t_tsv = time.perf_counter() - t0
        tsv_bytes = os.path.getsize(os.path.join(tmp, "dense.tsv"))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    out = {
        "what": "10x-style Matrix Market directory of the single-cell matrix (measureTE.sc_save_mtx) vs the dense TSV "
                "(sc_save_result), one seeded run",
        "config": {"records": args.records, "n_whitelist": n_wl, "maxcells": maxcells, "strand": True,
                   "index": "synth_index() (hg38-like, %d ensg)" % idx.n_ensg, "n_triples": int(nt), "n_hit_cells": int(nh),
                   "selected_cells": int(len(sel))},
        **gpu_info(),
        "host_cores": len(os.sched_getaffinity(0)),
        "nnz": int(nnz), "text_bytes": int(n_bytes), "bytes_per_line": (n_bytes / nnz) if nnz else None,
        "tec_sc_matrix_mtx_ms": t_dev * 1e3,
        "d2h_stream_ms": t_d2h * 1e3, "d2h_GBps": n_bytes / t_d2h / 1e9,
        "gzip_ms": t_gz * 1e3, "gzip_threads": threads, "gzip_level": mtx.LEVEL, "gzip_bytes": gz_bytes,
        "sc_save_mtx_ms": t_mtx * 1e3, "mtx_dir_bytes": mtx_dir_bytes,
        "sc_save_result_ms": t_tsv * 1e3, "tsv_bytes": tsv_bytes,
        "host_formatter_ms": t_host * 1e3, "device_text_equals_host_formatter": bool(same),
    }
    line = json.dumps(out)
    print(line)
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as fh:
            fh.write(line + "\n")
    return 0 if same else 1


if __name__ == "__main__":
    sys.exit(main())
