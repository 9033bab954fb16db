"""Counts per index row (bulk locus mode, include/tecount.h tec_bulk_loci) without a GPU: the Python oracle pinned to
the reference's per-name counts, the known answers, the C oracle against the Python one, the TSV writer against a
plain loop, and the CLI refusal."""
import numpy as np
import pytest

import helpers as H
import locus_oracle as LO
from te_counter_b200 import synth
from te_counter_b200.index import GlbIndex
from te_counter_b200.te_count import measureTE

COLS = ("start", "end", "chrom", "mapq", "flag")


def py_loci(idx, paired, qual, r, strand=False):
    f = LO.bulk_count_loci_stranded if strand else LO.bulk_count_loci
    return f(H.oracle_index(idx), paired, qual, *[np.asarray(r[k]).tolist() for k in COLS])


def c_loci(idx, paired, qual, r, strand=False, threads=3):
    return LO.c_bulk_count_loci(LO.CIndex(idx), paired, qual, *[r[k] for k in COLS],
                                strand_code=idx.strand_code if strand else None, threads=threads)


@pytest.mark.parametrize("name", H.case_names("bulk"))
def test_oracle_counts_from_its_rows_equal_the_reference(name):
    """The per-name counts bulk_count_loci derives from its own `result` lists are the reference's, and the row sums
    bound them from above."""
    case = H.load_case(name)
    idx = H.load_index(case["glb"])
    r = H.pack_bulk(case, idx)
    counts, st, loci = py_loci(idx, case["paired"], case["qual"], r)
    assert dict(zip(idx.names, counts)) == case["expected"]["result"]
    s = H.bulk_expected_stats(case["expected"])
    assert (st["total_reads"], st["assigned"], st["lowq"], st["badchrom"], st["qcfail"]) == \
        (s["total_reads"], s["assigned"], s["lowq"], s["badchrom"], s["qcfail"])
    per_name = np.bincount(idx.ensg_id, weights=np.asarray(loci), minlength=idx.n_ensg)
    assert (per_name >= np.asarray(counts)).all()
    c2, st2, l2 = c_loci(idx, case["paired"], case["qual"], r)
    assert c2.tolist() == counts and l2.tolist() == loci


def test_appendix_a_known_answer():
    """SURVEY.md Appendix A, toy index, single end: row 4 (the pseudogene) is hit but not counted."""
    case = H.load_case("bulk_se_appendixA")
    idx = H.load_index(case["glb"])
    _, _, loci = py_loci(idx, False, case["qual"], H.pack_bulk(case, idx))
    assert loci == [3, 1, 1, 1, 0]


def two_row_gene_index():
    # gene G has two rows on chromosome 1; T is a TE row elsewhere
    return GlbIndex(["1"], np.zeros(3, np.int32), np.array([1000, 5000, 30000], np.int32),
                    np.array([2000, 6000, 31000], np.int32), np.array([0, 0, 1], np.int32),
                    np.array([1, 1, 2], np.uint8), np.array([0, 0, 1], np.uint8), ["G", "T"])


def test_mates_on_two_rows_of_one_gene():
    """read1 starts in row 0 of G, read2 in row 1: the name counts once, each row once."""
    idx = two_row_gene_index()
    r = {"start": np.array([1500, 5500], np.int32), "end": np.array([1600, 5600], np.int32),
         "chrom": np.zeros(2, np.uint16), "mapq": np.full(2, 60, np.uint8), "flag": np.zeros(2, np.uint8)}
    counts, _, loci = py_loci(idx, True, 20, r)
    assert counts == [1, 0] and loci == [1, 1, 0]
    c2, _, l2 = c_loci(idx, True, 20, r)
    assert c2.tolist() == [1, 0] and l2.tolist() == [1, 1, 0]


def test_sum_identity_without_double_hits():
    """No unit hits two rows of one name: the row sums per name equal the per-name counts."""
    idx = two_row_gene_index()
    r = {"start": np.array([1500, 5500, 30100, 100], np.int32), "end": np.array([1600, 5600, 30200, 200], np.int32),
         "chrom": np.zeros(4, np.uint16), "mapq": np.full(4, 60, np.uint8), "flag": np.zeros(4, np.uint8)}
    counts, _, loci = py_loci(idx, False, 20, r)
    assert np.bincount(idx.ensg_id, weights=loci, minlength=idx.n_ensg).tolist() == counts == [2, 1]


@pytest.mark.parametrize("strand", [False, True])
@pytest.mark.parametrize("paired", [False, True])
@pytest.mark.parametrize("bs", [10000, 777])
def test_c_oracle_loci_match_python(paired, strand, bs):
    base = synth.synth_index(43, n_te=20000, n_exon=6000, n_gene=400, chrom_len=1_500_000, n_chrom=3)
    idx = GlbIndex(base.chrom_keys, base.chrom_id, base.L, base.R, base.ensg_id, base.type_code, base.strand_code,
                   base.names, bucket_size=bs)
    idx.chrom_lengths = base.chrom_lengths
    r = synth.synth_bulk_reads(44, idx, 30000, paired=paired, edge_frac=0.05)
    s = r["start"].copy()
    s[::7] = (s[::7] // bs) * bs                      # bucket edges of this bucket size
    s[3::11] = -5
    r["start"] = s
    r["flag"] = r["flag"] | np.where(np.arange(len(s)) % 3 == 0, 8, 0).astype(np.uint8)    # both strands
    counts, st, loci = py_loci(idx, paired, 20, r, strand)
    c2, st2, l2 = c_loci(idx, paired, 20, r, strand, threads=4)
    assert c2.tolist() == counts and l2.tolist() == loci
    assert (int(st2[0]) + 1, int(st2[1])) == (st["total_reads"], st["assigned"])
    per_name = np.bincount(idx.ensg_id, weights=l2, minlength=idx.n_ensg)
    assert (per_name >= c2).all() and sum(loci) > 1000


def plain_tsv(genome, counts, total_reads):
    per_million = total_reads / 1e6
    lines = ["ensg\tchrom\tleft\tright\tstrand\tcount\tcpm\n"]
    for i in range(genome.n_features):
        sc = int(genome.strand_code[i])
        strand = "." if sc == 255 else genome.strand_strings[sc]
        c = int(counts[i])
        lines.append("{}\t{}\t{}\t{}\t{}\t{}\t{}\n".format(genome.names[genome.ensg_id[i]], genome.chrom_keys[genome.chrom_id[i]],
                                                           int(genome.L[i]), int(genome.R[i]), strand, c, c / per_million))
    return "".join(lines).encode()


@pytest.mark.parametrize("n_chrom", [1, 2])
@pytest.mark.parametrize("total_reads", [1, 7, 1234567, 98765432101])
def test_save_result_loci_equals_a_plain_loop(tmp_path, n_chrom, total_reads):
    rng = np.random.default_rng(n_chrom * 7 + total_reads % 1000)
    n = 500
    L = np.sort(rng.integers(0, 250_000_000, n)).astype(np.int32)
    R = (L + rng.integers(0, 100_000, n)).astype(np.int32)
    strand = rng.choice(np.array([0, 1, 2, 255], np.uint8), n)
    names = ["ENSG%011d" % i for i in range(40)] + ["LINE:L1:L1HS", "LTR:ERVK:HERVK-int", "x"]
    idx = GlbIndex(["chr1", "chrUn_KI270302v1"][:n_chrom], rng.integers(0, n_chrom, n).astype(np.int32), L, R,
                   rng.integers(0, len(names), n).astype(np.int32), rng.integers(0, 5, n).astype(np.uint8), strand, names,
                   strand_strings=("+", "-", "."))
    counts = (10 ** rng.integers(0, 7, n) * rng.random(n)).astype(np.int64)   # 1 to 7 digits
    counts[:5] = [0, 9, 10, 9999999, 1234567]
    mte = measureTE("test", 20)
    mte.genome, mte.locus_counts, mte.total_reads = idx, counts, total_reads
    out = tmp_path / "loci.tsv"
    mte.save_result_loci(str(out))
    assert out.read_bytes() == plain_tsv(idx, counts, total_reads)


def test_save_result_loci_needs_a_locus_run(tmp_path):
    with pytest.raises(ValueError):
        measureTE("test", 20).save_result_loci(str(tmp_path / "x.tsv"))


def test_sharded_cli_refuses_loci_in_single_cell_mode():
    from te_counter_b200 import sharded
    with pytest.raises(SystemExit):
        sharded.main(["--glb", "x.glb", "--bam", "x.bam", "--mode", "sc", "--loci", "l.tsv", "-o", "o.tsv"])
