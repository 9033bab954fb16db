"""Synthetic workload, file form: writes a BGZF-compressed BAM of fixed-layout records, fast (numpy
builds the record bytes, a process pool deflates the blocks), for measuring the BAM decoders
(tools/bam_bench.py), file-to-result runs of measureTE (tools/file_e2e.py) and the `from_file` leg
of bench.py.  Records look like 10x / bulk RNA-seq alignments: 100 bp reads, CIGAR 40M<gap>N60M,
4-bit packed random sequence, skewed qualities, NH/AS/CB/UB tags.

    python -m te_counter_b200.synth_bam out.bam --records 4000000 --mode sc --whitelist wl.txt
    python -m te_counter_b200.synth_bam out.bam --records 16000000 --mode pe --sorted

--sorted (paired end): coordinate-sorted like `samtools sort` output, one unique QNAME per pair, mates 50 to 400 bp
apart and a fraction (--cross, default 2 %) of the pairs with the mate on another chromosome.  Every writer chunk
owns one slice of the genome; the cross-chromosome mates are planned up front and handed to the chunk whose slice
holds them.
"""
import argparse
import multiprocessing
import os
import struct
import zlib
from concurrent.futures import ProcessPoolExecutor

import numpy as np

HG38 = [("chr%s" % c, n) for c, n in zip(
    list(range(1, 23)) + ["X", "Y", "M"],
    [248956422, 242193529, 198295559, 190214555, 181538259, 170805979, 159345973, 145138636, 138394717, 133797422,
     135086622, 133275309, 114364328, 107043718, 101991189, 90338345, 83257441, 80373285, 58617616, 64444167,
     46709983, 50818468, 156040895, 57227415, 16569])]
BLOCK = 65280


def _bgzf(data):
    co = zlib.compressobj(4, zlib.DEFLATED, -15)
    comp = co.compress(data) + co.flush()
    head = struct.pack("<BBBBIBBHBBHH", 0x1f, 0x8b, 8, 4, 0, 0, 0xff, 6, 66, 67, 2, len(comp) + 25)
    return head + comp + struct.pack("<II", zlib.crc32(data) & 0xffffffff, len(data))


def _deflate_chunk(raw):
    return b"".join(_bgzf(raw[o:o + BLOCK]) for o in range(0, len(raw), BLOCK))


def header_bytes(contigs):
    text = "@HD\tVN:1.6\tSO:unsorted\n" + "".join("@SQ\tSN:%s\tLN:%d\n" % c for c in contigs)
    raw = b"BAM\1" + struct.pack("<i", len(text)) + text.encode() + struct.pack("<i", len(contigs))
    for name, ln in contigs:
        raw += struct.pack("<i", len(name) + 1) + name.encode() + b"\0" + struct.pack("<i", ln)
    return raw


def records_bytes(rng, n, contigs, mode, barcodes, first_id, layout=None):
    """n records as one uint8 matrix [n, rec_size] (every record has the same size).  layout: (ref, pos, flag, name id)
    arrays that replace the random placement (sorted paired end)."""
    sc = mode == "sc"
    name_len = 24                                           # with the NUL
    n_cig, l_seq = 3, 100
    aux = 4 + 7 + ((3 + 18 + 1) + (3 + 12 + 1) if sc else 0)    # NH:C, AS:i, CB:Z (16 + "-1"), UB:Z (12)
    body = 32 + name_len + 4 * n_cig + (l_seq + 1) // 2 + l_seq + aux
    m = np.zeros((n, 4 + body), dtype=np.uint8)

    def put(off, arr, dt):
        m[:, off:off + np.dtype(dt).itemsize] = np.ascontiguousarray(arr.astype(dt)).view(np.uint8).reshape(n, -1)

    lens = np.array([c[1] for c in contigs], dtype=np.float64)
    if layout is not None:
        rng.random(n)                                       # keeps the draws below independent of the layout
    ref = rng.choice(len(contigs), size=n, p=lens / lens.sum())
    pos = (rng.random(n) * np.maximum(lens[ref] - 200000, 1000)).astype(np.int64)
    flag = np.where(rng.random(n) < 0.5, 16, 0)
    flag |= np.where(rng.random(n) < 0.02, 0x400, 0) | np.where(rng.random(n) < 0.005, 0x200, 0)
    unm = rng.random(n) < 0.01
    flag |= np.where(unm, 4, 0)
    if mode == "pe":
        ids = first_id + np.arange(n)
        flag |= np.where(ids % 2 == 0, 0x41, 0x81)
        mate = np.roll(pos, 1)
        pos = np.where(ids % 2 == 1, np.clip(mate + rng.integers(50, 400, n), 0, None), pos)
        ref = np.where(ids % 2 == 1, np.roll(ref, 1), ref)
    if layout is not None:
        ref, pos, flag, name_ids = layout
    u = rng.random(n)
    mapq = np.where(u < 0.8, 255, np.where(u < 0.9, rng.integers(20, 60, n), rng.integers(0, 20, n)))
    put(0, np.full(n, body), "<i4")
    put(4, ref, "<i4")
    put(8, pos, "<i4")
    m[:, 12] = name_len
    m[:, 13] = mapq
    put(14, np.full(n, 4680), "<u2")
    put(16, np.full(n, n_cig), "<u2")
    put(18, flag, "<u2")
    put(20, np.full(n, l_seq), "<i4")
    put(24, np.full(n, -1), "<i4")
    put(28, np.full(n, -1), "<i4")
    put(32, np.zeros(n), "<i4")
    o = 36
    ids = first_id + np.arange(n)
    if mode == "pe":
        ids = ids // 2
    if layout is not None:
        ids = name_ids
    digits = np.array([(ids // 10 ** k) % 10 for k in range(14, -1, -1)], dtype=np.uint8).T + 48
    m[:, o:o + 8] = np.frombuffer(b"NB5012:7", dtype=np.uint8)
    m[:, o + 8:o + 23] = digits
    o += name_len
    gap = np.where(rng.random(n) < 0.15, rng.lognormal(7, 1, n).astype(np.int64) + 1, 0)
    put(o, np.full(n, 40 << 4 | 0), "<u4")
    put(o + 4, gap << 4 | 3, "<u4")
    put(o + 8, np.full(n, 60 << 4 | 0), "<u4")
    o += 12
    m[:, o:o + 50] = np.array([0x11, 0x12, 0x14, 0x18, 0x21, 0x22, 0x24, 0x28, 0x41, 0x42, 0x44, 0x48, 0x81, 0x82, 0x84,
                               0x88], dtype=np.uint8)[rng.integers(0, 16, (n, 50))]
    o += 50
    m[:, o:o + 100] = np.array([37, 37, 37, 37, 37, 32, 32, 25, 14, 2], dtype=np.uint8)[rng.integers(0, 10, (n, 100))]
    o += 100
    m[:, o:o + 4] = np.frombuffer(b"NHC\1", dtype=np.uint8)
    m[:, o + 4:o + 7] = np.frombuffer(b"ASi", dtype=np.uint8)
    put(o + 7, rng.integers(60, 99, n), "<i4")
    o += 11
    if sc:
        u = rng.random(n)
        n_real = max(1, len(barcodes) // 10)
        cell = np.where(u < 0.9, rng.integers(0, n_real, n), rng.integers(0, len(barcodes), n))
        bc = barcodes[cell].copy()
        bad = rng.random(n) < 0.02
        bc[bad, 0] = ord("N")
        m[:, o:o + 3] = np.frombuffer(b"CBZ", dtype=np.uint8)
        m[:, o + 3:o + 19] = bc
        m[:, o + 19:o + 21] = np.frombuffer(b"-1", dtype=np.uint8)
        o += 22
        m[:, o:o + 3] = np.frombuffer(b"UBZ", dtype=np.uint8)
        m[:, o + 3:o + 15] = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, (n, 12))]
        o += 16
    assert o == 4 + body
    return m


def _chunk(job):
    seed, i, n, mode, barcodes = job
    rng = np.random.default_rng([seed, i])
    return _deflate_chunk(records_bytes(rng, n, HG38, mode, barcodes, i * 250000).tobytes())


SORTED_CHUNK_PAIRS = 125000


def _pe_flags(rng, n, read1):
    """SAM flags of paired-end mates: 0x1, 0x40 or 0x80, strand, and a few duplicates, QC fails, unmapped and
    secondary records"""
    f = np.where(read1, 0x41, 0x81) | np.where(rng.random(n) < 0.5, 16, 0)
    f |= np.where(rng.random(n) < 0.02, 0x400, 0) | np.where(rng.random(n) < 0.005, 0x200, 0)
    f |= np.where(rng.random(n) < 0.01, 4, 0) | np.where(rng.random(n) < 0.005, 0x100, 0)
    return f


def _sorted_chunk(job):
    """Chunk i of a coordinate-sorted paired-end file: its pairs within its slice [lo, hi) of the concatenated genome,
    plus the cross-chromosome mates planned into the slice, in (reference, position) order."""
    seed, i, n_pairs, lo, hi, foreign = job
    rng = np.random.default_rng([seed, 1, i])
    starts = np.cumsum([0] + [c[1] for c in HG38])
    g = np.sort(rng.integers(lo, max(lo + 1, hi - 1000), n_pairs))
    ref = np.searchsorted(starts, g, side="right") - 1
    pos = g - starts[ref]
    pos = np.minimum(pos, np.array([c[1] for c in HG38])[ref] - 1000)
    d = rng.integers(50, 401, n_pairs)
    ids = (np.int64(i) * SORTED_CHUNK_PAIRS + np.arange(n_pairs)).astype(np.int64)
    f_ref, f_pos, f_id, f_r1 = foreign
    refs = np.concatenate([ref, ref, f_ref])
    poss = np.concatenate([pos, pos + d, f_pos])
    read1 = np.concatenate([np.ones(n_pairs, bool), np.zeros(n_pairs, bool), f_r1])
    names = np.concatenate([ids, ids, f_id])
    order = np.lexsort((poss, refs))
    refs, poss, read1, names = refs[order], poss[order], read1[order], names[order]
    n = len(refs)
    lay = (refs, poss, _pe_flags(rng, n, read1), names)
    return _deflate_chunk(records_bytes(rng, n, HG38, "pe", None, 0, layout=lay).tobytes())


def _sorted_jobs(records, seed, cross):
    """Jobs of _sorted_chunk: equal genome slices; the cross-chromosome pairs are placed here, both mates at random
    positions of two different chromosomes, and each mate goes to the job whose slice holds it."""
    rng = np.random.default_rng([seed, 2])
    pairs = records // 2
    n_cross = int(round(pairs * cross))
    n_local = pairs - n_cross
    n_jobs = max(1, (n_local + SORTED_CHUNK_PAIRS - 1) // SORTED_CHUNK_PAIRS)
    lens = np.array([c[1] for c in HG38], dtype=np.int64)
    starts = np.concatenate([[0], np.cumsum(lens)])
    edges = np.linspace(0, starts[-1], n_jobs + 1).astype(np.int64)
    r1 = rng.choice(len(HG38), n_cross, p=lens / lens.sum())
    r2 = (r1 + rng.integers(1, len(HG38), n_cross)) % len(HG38)
    p1 = (rng.random(n_cross) * (lens[r1] - 1000)).astype(np.int64)
    p2 = (rng.random(n_cross) * (lens[r2] - 1000)).astype(np.int64)
    cid = n_jobs * SORTED_CHUNK_PAIRS + np.arange(n_cross)
    f_ref = np.concatenate([r1, r2])
    f_pos = np.concatenate([p1, p2])
    f_id = np.concatenate([cid, cid])
    f_r1 = np.concatenate([np.ones(n_cross, bool), np.zeros(n_cross, bool)])
    f_job = np.searchsorted(edges, starts[f_ref] + f_pos, side="right") - 1
    jobs = []
    for j in range(n_jobs):
        k = f_job == j
        n = min(SORTED_CHUNK_PAIRS, n_local - j * SORTED_CHUNK_PAIRS)
        jobs.append((seed, j, n, int(edges[j]), int(edges[j + 1]), (f_ref[k], f_pos[k], f_id[k], f_r1[k])))
    return jobs


def write(out, records=4000000, mode="pe", whitelist=None, n_barcodes=100000, seed=20261018, procs=None, sorted_pe=False,
          cross=0.02):
    """Writes the file; returns its size in bytes.  sorted_pe: coordinate-sorted paired end (module header)."""
    rng = np.random.default_rng(seed)
    barcodes = None
    if mode == "sc":
        barcodes = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, (n_barcodes, 16))]
        barcodes = np.unique(barcodes, axis=0)
        if whitelist:
            with open(whitelist, "w") as fh:
                fh.write("".join(bytes(b).decode() + "-1\n" for b in barcodes))
    chunk = 250000
    jobs = [(seed, i, min(chunk, records - i * chunk), mode, barcodes) for i in range((records + chunk - 1) // chunk)]
    fn = _chunk
    if sorted_pe:
        if mode != "pe":
            raise ValueError("sorted_pe needs mode 'pe'")
        jobs, fn = _sorted_jobs(records, seed, cross), _sorted_chunk
    # worker processes come from a fork server: the caller may be a multi-threaded process with a CUDA context
    # (bench.py), which must not be forked
    ctx = multiprocessing.get_context("forkserver")
    with open(out, "wb") as fh, ProcessPoolExecutor(procs or os.cpu_count() or 1, mp_context=ctx) as ex:
        fh.write(_bgzf(header_bytes(HG38)))
        for comp in ex.map(fn, jobs):                   # records straddle blocks inside a chunk
            fh.write(comp)
        fh.write(_bgzf(b""))
    return os.path.getsize(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--records", type=int, default=4000000)
    ap.add_argument("--mode", choices=["se", "pe", "sc"], default="pe")
    ap.add_argument("--whitelist", help="sc: file to write the barcode whitelist to (barcodes end in -1)")
    ap.add_argument("--barcodes", type=int, default=100000)
    ap.add_argument("--seed", type=int, default=20261018)
    ap.add_argument("--procs", type=int, default=os.cpu_count() or 1)
    ap.add_argument("--sorted", action="store_true", help="pe: coordinate-sorted, mates paired by read name")
    ap.add_argument("--cross", type=float, default=0.02, help="--sorted: fraction of pairs whose mates are on two chromosomes")
    a = ap.parse_args()
    if a.sorted and a.mode != "pe":
        ap.error("--sorted needs --mode pe")
    size = write(a.out, a.records, a.mode, a.whitelist, a.barcodes, a.seed, a.procs, sorted_pe=a.sorted, cross=a.cross)
    print(a.out, size, "bytes,", a.records, "records")


if __name__ == "__main__":
    main()
