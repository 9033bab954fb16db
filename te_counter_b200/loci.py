"""
The counts per index row of a bulk run with loci (measureTE.save_result_loci) as a TSV:

    ensg\\tchrom\\tleft\\tright\\tstrand\\tcount\\tcpm
    one line per index row, in linearData order

chrom is the index's chromosome key, strand the row's strand string ('.' when the row has none), cpm the count over
total_reads / 1e6 printed as Python's float repr -- the CPM of save_result_bulk.  A genome index has about 6 M rows, so
the text is assembled with array operations, a block of rows at a time: "ensg\\tchrom\\t" is formatted once per distinct
(ensg, chromosome) and "\\tstrand\\tcount\\tcpm\\n" once per distinct (strand, count); every row is then the bytes of its
two table entries with its left and right in decimal between them, laid out at fixed width with NUL padding, and the
padding is dropped (the text holds no NUL).
"""
import numpy as np

from .index import STRAND_MISSING

HEADER = b"ensg\tchrom\tleft\tright\tstrand\tcount\tcpm\n"
BLOCK = 1 << 20                    # rows per block: bounds the fixed-width scratch to about 100 MB
INT_WIDTH = 11                     # '-' and ten digits: any int32


def _table(strings):
    """uint8[len, width]: each string's bytes, NUL-padded"""
    enc = [s.encode("utf-8") for s in strings]
    t = np.zeros((len(enc), max([len(b) for b in enc] + [1])), dtype=np.uint8)
    for i, b in enumerate(enc):
        t[i, :len(b)] = np.frombuffer(b, dtype=np.uint8)
    return t


def _decimal(v):
    """uint8[len, INT_WIDTH]: v right-aligned in decimal, NUL-padded on the left"""
    a = np.abs(v.astype(np.int64))
    out = np.zeros((len(v), INT_WIDTH), dtype=np.uint8)
    more = np.ones(len(v), dtype=bool)
    for col in range(INT_WIDTH - 1, 0, -1):
        out[:, col] = np.where(more, a % 10 + ord("0"), 0)
        a //= 10
        lead = more & (a == 0)                    # the digit just written was the leading one
        more &= a > 0
        out[lead & (v < 0), col - 1] = ord("-")
    return out


def tsv_text(genome, counts, total_reads):
    """The TSV bytes.  genome: index.GlbIndex; counts: int64[n_features] in linearData order."""
    counts = np.asarray(counts, dtype=np.int64)
    n = genome.n_features
    if len(counts) != n:
        raise ValueError("%d counts for an index of %d rows" % (len(counts), n))
    if not n:
        return HEADER
    per_million = total_reads / 1e6
    strands = list(genome.strand_strings) + ["."]
    strand_idx = np.where(genome.strand_code == STRAND_MISSING, len(genome.strand_strings), genome.strand_code).astype(np.int64)
    head_key, head_at = np.unique(genome.ensg_id.astype(np.int64) * genome.n_chrom + genome.chrom_id, return_inverse=True)
    head = _table(["%s\t%s\t" % (genome.names[k // genome.n_chrom], genome.chrom_keys[k % genome.n_chrom])
                   for k in head_key.tolist()])
    tail_key, tail_at = np.unique(counts * len(strands) + strand_idx, return_inverse=True)
    tail = _table(["\t%s\t%d\t%r\n" % (strands[k % len(strands)], k // len(strands), (k // len(strands)) / per_million)
                   for k in tail_key.tolist()])
    tab = np.full((min(n, BLOCK), 1), ord("\t"), dtype=np.uint8)
    parts = [HEADER]
    for a in range(0, n, BLOCK):
        b = min(n, a + BLOCK)
        m = np.concatenate([head[head_at[a:b]], _decimal(genome.L[a:b]), tab[:b - a], _decimal(genome.R[a:b]),
                            tail[tail_at[a:b]]], axis=1)
        parts.append(m[m != 0].tobytes())
    return b"".join(parts)
