"""
One BAM counted by all GPUs of a node:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29500 \\
        -m te_counter_b200.sharded --glb genes_tes.glb --bam in.bam --mode se -o out.tsv
    ... --mode pe -o out.tsv
    ... --mode pe --pairing name -o out.tsv      (coordinate-sorted BAM: mates paired by read name)
    ... --mode se|pe --loci loci.tsv -o out.tsv   (also the counts per index row; measureTE.save_result_loci)
    ... --mode sc --whitelist 3M-february-2018.txt --maxcells 10000 [--strand] -o out.tsv
    ... --mode sc --format mtx ... -o out_dir      (matrix.mtx.gz, features.tsv.gz, barcodes.tsv.gz; measureTE.sc_save_mtx)

Every rank builds the same `measureTE` the reference's bin/te_count builds (bin/te_count:77-120) and calls the same
method; inside, the ranks split the file by byte ranges (shard.py; paired end pairs records by their global index, so
each rank keeps the counter bank of its record parity and counts the pair across its front border; with --pairing name
each rank sends the records of its range to the rank that owns their read name, which pairs them).  Rank 0 writes the
outputs, which are byte for byte those of a one-GPU run.  With fewer GPUs than ranks the ranks share GPUs and talk over gloo (tests).
"""
import argparse
import logging
import os
import sys


def main(argv=None):
    ap = argparse.ArgumentParser(prog="python -m te_counter_b200.sharded")
    ap.add_argument("--glb", required=True)
    ap.add_argument("--bam", required=True)
    ap.add_argument("--mode", choices=["se", "pe", "sc"], default="se")
    ap.add_argument("-q", "--qual", type=int, default=20)
    ap.add_argument("--whitelist")
    ap.add_argument("--maxcells", type=int, default=10000)
    ap.add_argument("--strand", action="store_true")
    ap.add_argument("--format", choices=["tsv", "mtx"], default="tsv",
                    help="single cell: the reference's dense TSV (default) or a 10x-style Matrix Market directory at -o")
    ap.add_argument("--pairing", choices=["index", "name"], default="index",
                    help="paired end: record 2i with 2i+1 as the reference (default), or mates by read name (measureTE.parse_bampe; "
                         "every rank decodes its byte range and the records meet by name)")
    ap.add_argument("--loci", metavar="PATH",
                    help="bulk: also count per index row and write them to PATH (measureTE.save_result_loci)")
    ap.add_argument("-o", "--out", required=True)
    args = ap.parse_args(argv)
    if args.format == "mtx" and args.mode != "sc":
        ap.error("--format mtx needs --mode sc")
    if args.pairing == "name" and args.mode != "pe":
        ap.error("--pairing name needs --mode pe")
    if args.loci and args.mode == "sc":
        ap.error("--loci needs --mode se or pe")
    import torch
    import torch.distributed as dist
    from . import measureTE
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    n_gpu = torch.cuda.device_count()
    device = local % max(1, n_gpu)
    torch.cuda.set_device(device)
    if world > 1:
        if n_gpu >= world:
            dist.init_process_group("nccl", device_id=torch.device("cuda", device))
        else:
            dist.init_process_group("gloo")
    logging.basicConfig(level=logging.INFO if rank == 0 else logging.WARNING, format="%(levelname)-8s: %(message)s")
    log = logging.getLogger("te_count")
    mte = measureTE(sys.path[0], args.qual, device=device)
    mte.bind_genome(args.glb)
    if args.mode == "sc":
        res = mte.sc_parse_bamse(args.bam, UMIS=True, whitelistfilename=args.whitelist, strand=args.strand, log=log,
                                 label=os.path.basename(args.out), maxcells=args.maxcells)
        if rank == 0 and args.format == "mtx":
            mte.sc_save_mtx(res, args.out, maxcells=args.maxcells, log=log)
        elif rank == 0:
            mte.sc_save_result(res, args.out, maxcells=args.maxcells, log=log)
    else:
        mte.load_genome()
        if args.mode == "pe":
            res = mte.parse_bampe(args.bam, log=log, pairing=args.pairing, loci=bool(args.loci))
        else:
            res = mte.parse_bamse(args.bam, log=log, loci=bool(args.loci))
        if rank == 0:
            mte.save_result_bulk(res, args.out, log=log)
            if args.loci:
                mte.save_result_loci(args.loci, log=log)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
