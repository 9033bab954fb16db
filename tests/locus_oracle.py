"""TEST INFRASTRUCTURE -- counts per index row (bulk locus mode, include/tecount.h tec_bulk_loci; the reference has
no such output).  Same rules as oracle/: only tests and tools/locus_bench.py use it, as the checker.

Rule: filters, mate merge, candidate rule, point tests, type rule and statistics are the reference's.  A unit whose
`result` the tally counts (its hit rows include a gene, TE or snRNA type) adds 1 to every row in `result`, once per
row; any other unit adds nothing.  Under the bulk --strand rule (oracle/te_oracle_ext.py) the rows the strand filter
removes are not hits.

bulk_count_loci is oracle/te_oracle.bulk_count's loop, literally, with the rows tallied from the same `result`;
CIndex / c_bulk_count_loci run tests/locus_oracle_c.c (the C loop of oracle/te_oracle_c.c with the same additions,
multi-threaded) for full-size results.  The C library is compiled into a temporary directory on first use."""
import ctypes
import os
import subprocess
import tempfile

import numpy as np

from oracle import te_oracle
from oracle.te_oracle import F_REVERSE

HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def bulk_count_loci(idx, paired, qual, start, end, chrom, mapq, flag, candidate=None):
    """Counts per index row (tec_set_option "bulk_loci"; the reference has no such output).
    Rule: a unit whose `result` the tally counts (its hit rows include a gene, TE or snRNA type) adds 1 to every
    row in `result`, once per row; any other unit adds nothing.  This is te_oracle.bulk_count's loop, literally
    (bucket hash, `result` list, _bulk_tally), with the rows tallied from the same `result`.
    Returns (counts, stats, loci) with loci a list[n_features] in linearData order."""
    counts = [0] * idx.n_ensg
    loci = [0] * len(idx.L)
    bs = idx.bs
    assigned = lowq = badchrom = qcfail = 0
    n = len(start)
    pos = 0
    units = 0
    counted = (te_oracle.T_GENE, te_oracle.T_TE, te_oracle.T_SNRNA)
    reject = te_oracle.F_UNMAPPED | te_oracle.F_DUP | te_oracle.F_QCFAIL
    while True:
        units += 1
        if paired:
            if pos + 2 > n:
                break
            r1, r2 = pos, pos + 1
            pos += 2
            if flag[r1] & reject or flag[r2] & reject:
                qcfail += 1
                continue
            if mapq[r1] < qual:
                lowq += 1
                continue
            if flag[r1] & te_oracle.F_NAME_MISMATCH:
                raise te_oracle.ReferenceCrash("AttributeError", "sys.quit (te_count.py:94)")
            c, loc1, loc2 = chrom[r1], start[r1], start[r2]
        else:
            if pos + 1 > n:
                break
            r1 = pos
            pos += 1
            if flag[r1] & reject:
                qcfail += 1
                continue
            if mapq[r1] < qual:
                lowq += 1
                continue
            c, loc1, loc2 = chrom[r1], start[r1], end[r1]
        if c not in idx.buckets:
            badchrom += 1
            continue
        loc_ids = set()
        for buck in (((loc1 - 1) // bs) * bs, ((loc2 + 1) // bs) * bs):
            if buck in idx.buckets[c]:
                loc_ids.update(idx.buckets[c][buck])
        result = []
        for i in loc_ids:
            if candidate is not None and not candidate(i, r1):
                continue
            if loc1 >= idx.L[i] and loc1 + 1 <= idx.R[i]:
                result.append(i)
            if loc2 - 1 >= idx.L[i] and loc2 <= idx.R[i]:
                result.append(i)
        if result:
            te_oracle._bulk_tally(idx, result, counts)
            if any(idx.type_code[i] in counted for i in result):
                for i in set(result):
                    loci[i] += 1
            assigned += 1
    return counts, {"total_reads": units, "assigned": assigned, "lowq": lowq,
                    "badchrom": badchrom, "qcfail": qcfail}, loci


def bulk_count_loci_stranded(idx, paired, qual, start, end, chrom, mapq, flag):
    """bulk_count_loci under the bulk --strand rule (see the module header): the candidate of oracle/te_oracle_ext.bulk_count_stranded."""
    def candidate(i, r1):
        fs = idx.strand_code[i]
        us = 1 if (flag[r1] & F_REVERSE) else 0
        return not (fs in (0, 1) and fs != us)
    return bulk_count_loci(idx, paired, qual, start, end, chrom, mapq, flag, candidate=candidate)


def load():
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="tec_locus_oracle_"), "liblocusoracle.so")
        subprocess.run([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-pthread", "-shared", "-o", out,
                        os.path.join(HERE, "locus_oracle_c.c")], check=True)
        lib = ctypes.CDLL(out)
        vp = ctypes.c_void_p
        lib.teo_index_build.restype = vp
        lib.teo_index_build.argtypes = [ctypes.c_int64, vp, vp, vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int]
        lib.teo_index_free.argtypes = [vp]
        lib.lo_bulk_count_loci.restype = ctypes.c_int
        lib.lo_bulk_count_loci.argtypes = [vp, ctypes.c_int, ctypes.c_int, ctypes.c_int64] + [vp] * 9 + [ctypes.c_int]
        _lib = lib
    return _lib


class CIndex:
    """The bucket hash of oracle/te_oracle_c.c over arrays in linearData order (index.GlbIndex)."""

    def __init__(self, idx):
        self._keep = [np.ascontiguousarray(idx.chrom_id, np.int32), np.ascontiguousarray(idx.L, np.int32),
                      np.ascontiguousarray(idx.R, np.int32), np.ascontiguousarray(idx.ensg_id, np.int32),
                      np.ascontiguousarray(idx.type_code, np.uint8)]
        self.n_ensg, self.n_feat = int(idx.n_ensg), len(self._keep[1])
        self._lib = load()
        self._h = self._lib.teo_index_build(self.n_feat, *[a.ctypes.data for a in self._keep], int(idx.n_chrom),
                                            self.n_ensg, int(idx.bucket_size))

    def __del__(self):
        try:
            self._lib.teo_index_free(self._h)
        except Exception:
            pass


def c_bulk_count_loci(cidx, paired, qual, start, end, chrom, mapq, flag, strand_code=None, threads=0):
    """(counts int64[n_ensg], stats int64[7] in include/tecount.h order, loci int64[n_features] in linearData order)"""
    lib = load()
    cols = [np.ascontiguousarray(a, dtype=dt) for a, dt in zip((start, end, chrom, mapq, flag),
                                                                (np.int32, np.int32, np.uint16, np.uint8, np.uint8))]
    sc = None if strand_code is None else np.ascontiguousarray(strand_code, np.uint8)
    counts = np.zeros(cidx.n_ensg, np.int64)
    stats = np.zeros(7, np.int64)
    loci = np.zeros(cidx.n_feat, np.int64)
    lib.lo_bulk_count_loci(cidx._h, 1 if paired else 0, int(qual), len(cols[0]), *[c.ctypes.data for c in cols],
                           None if sc is None else sc.ctypes.data, counts.ctypes.data, stats.ctypes.data, loci.ctypes.data,
                           int(threads or os.cpu_count() or 1))
    return counts, stats, loci
