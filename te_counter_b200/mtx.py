"""
The single-cell matrix as a 10x-style Matrix Market directory, the layout Cell Ranger writes as
filtered_feature_bc_matrix/ and that scanpy.read_10x_mtx and Seurat's Read10X read:

    matrix.mtx.gz     "%%MatrixMarket matrix coordinate integer general", "<features> <cells> <nnz>", then one
                      "<feature> <cell> <count>" line per non-zero (1-based), ascending in (cell, feature)
    features.tsv.gz   "<name>\\t<name>\\tGene Expression" per feature, in the order of the matrix rows
    barcodes.tsv.gz   one barcode per matrix column

The matrix text is normally built on the device (include/tecount.h tec_sc_matrix_mtx); `mtx_text` formats the same
bytes from the triples on the host, for runs whose device does not hold the job's triples.

Every file is gzip in independent members of at most PIECE bytes of text, compressed on a thread pool (zlib releases
the GIL) with mtime 0 and written in order: the bytes depend on the text only, not on the thread count.
Multi-member gzip is standard (RFC 1952 section 2.2); Python's gzip, scipy.io.mmread, scanpy and R read it.
"""
import gzip
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np

BANNER = b"%%MatrixMarket matrix coordinate integer general\n"
PIECE = 16 << 20
LEVEL = 6                          # zlib's and the gzip tool's default level

_POW10 = np.array([10 ** k for k in range(1, 20)], dtype=np.uint64)


def default_threads():
    return max(1, min(32, len(os.sched_getaffinity(0))))


def _ndigits(v):
    """decimal digits of each element of the uint64 array v (1 for 0)"""
    d = np.ones(len(v), dtype=np.int64)
    for p in _POW10:
        d += v >= p
    return d


def _lines(fields):
    """One line "<f0> <f1> ... <fk>\\n" per element of the equal-length uint64 arrays `fields`, as bytes."""
    n = len(fields[0])
    if not n:
        return b""
    nd = [_ndigits(f) for f in fields]
    length = sum(nd) + len(fields)
    at = np.cumsum(length) - length
    out = np.empty(int(at[-1] + length[-1]), dtype=np.uint8)
    for i, (f, d) in enumerate(zip(fields, nd)):
        v = f.copy()
        for p in range(int(d.max())):                     # digit p from the right, where the number has one
            m = d > p
            out[(at + d - 1 - p)[m]] = (v[m] % np.uint64(10)).astype(np.uint8) + ord("0")
            v //= np.uint64(10)
        at = at + d
        out[at] = ord(" ") if i + 1 < len(fields) else ord("\n")
        at = at + 1
    return out.tobytes()


def mtx_text(n_ensg, ensg, cell, count, cells):
    """The text of tec_sc_matrix_mtx from (ensg, cell, count) triples: column k is whitelist id cells[k]; triples of
    cells not listed are left out."""
    cells = np.asarray(cells, dtype=np.int64)
    cell = np.asarray(cell, dtype=np.int64)
    order = np.argsort(cells, kind="stable")
    sc = cells[order]
    pos = np.minimum(np.searchsorted(sc, cell), max(len(sc) - 1, 0))
    keep = sc[pos] == cell if len(sc) else np.zeros(len(cell), bool)
    k = order[pos[keep]]
    e = np.asarray(ensg, dtype=np.int64)[keep]
    v = np.asarray(count, dtype=np.int64)[keep]
    o = np.lexsort((e, k))
    head = BANNER + b"%d %d %d\n" % (n_ensg, len(cells), len(o))
    return head + _lines([(e[o] + 1).astype(np.uint64), (k[o] + 1).astype(np.uint64), v[o].astype(np.uint64)])


def features_text(names):
    return "".join("%s\t%s\tGene Expression\n" % (n, n) for n in names).encode()


def barcodes_text(barcodes):
    return "".join(b + "\n" for b in barcodes).encode()


class GzipPieces:
    """Binary file object: what is written to it goes to `fh` as gzip members of PIECE bytes of input each (the last
    one shorter), compressed by `pool`.  At most `window` pieces are in flight.  close() writes the rest; it does not
    close `fh`."""

    def __init__(self, fh, pool, window):
        self._fh, self._pool, self._window = fh, pool, max(1, window)
        self._buf = bytearray()
        self._pending = []
        self._pieces = 0

    def write(self, data):
        self._buf += data
        while len(self._buf) >= PIECE:
            self._submit(bytes(self._buf[:PIECE]))
            del self._buf[:PIECE]
        return len(data)

    def _submit(self, piece):
        self._pieces += 1
        self._pending.append(self._pool.submit(gzip.compress, piece, LEVEL, mtime=0))
        while len(self._pending) > self._window:
            self._fh.write(self._pending.pop(0).result())

    def close(self):
        if self._buf or not self._pieces:
            self._submit(bytes(self._buf))                # an empty text is one empty member: still a gzip file
            self._buf = bytearray()
        while self._pending:
            self._fh.write(self._pending.pop(0).result())


def write_gzip(path, produce, threads):
    """path = gzip of what produce(fh) writes into the binary file object it is given."""
    with open(path, "wb") as fh, ThreadPoolExecutor(max_workers=threads) as pool:
        gz = GzipPieces(fh, pool, 2 * threads)
        produce(gz)
        gz.close()
