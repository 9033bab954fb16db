/*
 * tecount.h -- C ABI of libtecount.so, the B200 (sm_100a) counting engine behind te_count.
 *
 * The reference (oaxiom/te_counter) is pure Python and has no FFI; the seam this library sits
 * behind is the `measureTE` method set (reference te_count/te_count.py:14-754) called from
 * bin/te_count:77-120.  Each entry point below names the reference lines whose work it takes
 * over.  Python binds it with ctypes (te_counter_b200/_lib.py); INTEGRATION.md shows the stub a
 * maintainer of the reference would add.
 *
 * Conventions
 *   - every call returns 0 (TEC_OK) or a negative tec_status; nothing throws across the ABI;
 *     tec_last_error(ctx) gives the text of the last failure on that context.
 *   - plain pointers and sizes only.  The caller owns every host buffer.  The library owns all
 *     device memory inside the context, except where a parameter is documented as a device
 *     pointer (`*_dev` entry points), which the caller (e.g. a torch tensor) owns.
 *   - one context per GPU; a context is not thread-safe.  Work is enqueued on the context's
 *     stream; calls that return results to host memory synchronise before returning.
 *   - there is no CPU fallback: tec_create fails when no CUDA device is usable.
 *
 * Record layout (structure of arrays, one element per alignment record, SURVEY.md 8d):
 *   int32  start   pysam reference_start (0-based)
 *   int32  end     pysam reference_end   (exclusive)
 *   uint16 chrom   index chromosome id (< n_chrom of tec_index_upload); any other value means
 *                  "not in the index"; 0xFFFE = name contains '_' or 'alt' (single-cell skip)
 *   uint8  mapq
 *   uint8  flag    bit0 unmapped(0x4) bit1 duplicate(0x400) bit2 qcfail(0x200) bit3 reverse(0x10)
 *                  bit4 paired-end query-name mismatch (te_count.py:92)
 *   uint32 cell    [single cell] id of the barcode in the sorted whitelist, 0xFFFFFFFF = not in it
 *   uint64 umi     [single cell] order-preserving code of the UMI string
 */
#ifndef TECOUNT_H
#define TECOUNT_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TEC_ABI_VERSION 1

typedef struct tec_ctx tec_ctx;

typedef enum tec_status {
    TEC_OK = 0,
    TEC_ERR_CUDA = -1,          /* a CUDA runtime call failed (text in tec_last_error) */
    TEC_ERR_ARG = -2,           /* bad argument */
    TEC_ERR_STATE = -3,         /* call out of order (no index, no begin, ...) */
    TEC_ERR_NOMEM = -4,         /* device or host allocation failed */
    TEC_ERR_LIMIT = -5,         /* input exceeds a documented limit (key width, record count) */
    TEC_ERR_UNIMPLEMENTED = -6,
    TEC_ERR_IO = -7,            /* tec_bam_open: the file cannot be opened or mapped */
    TEC_ERR_FORMAT = -8,        /* tec_bam_*: corrupt or truncated BAM / BGZF data */
    TEC_ERR_UNSUPPORTED = -9,   /* tec_bam_*: a file the device decoder refuses (not BGZF, or record boundaries it
                                   cannot establish block-parallel): decode it with libtecbam instead */
    /* tec_bam_count: a record on which the reference's read loop raises (same numbers as tecbam.h) */
    TEC_ERR_BAM_NO_BARCODE_TAG = -10, TEC_ERR_BAM_NO_UMI_TAG = -11, TEC_ERR_BAM_UMI = -12, TEC_ERR_BAM_END_NONE = -13,
    TEC_ERR_BAM_CHROM_NAME = -14, TEC_ERR_BAM_REF_NONE = -15
} tec_status;

/* feature type codes: which branch of te_count.py:134-146 / :662-682 a feature can trigger */
#define TEC_T_OTHER 0
#define TEC_T_GENE 1            /* protein_coding, lincRNA, lncRNA */
#define TEC_T_TE 2
#define TEC_T_SNRNA 3
#define TEC_T_ENHANCER 4
#define TEC_STRAND_MISSING 255  /* feature row has no 'strand' key */

#define TEC_F_UNMAPPED 1
#define TEC_F_DUP 2
#define TEC_F_QCFAIL 4
#define TEC_F_REVERSE 8
#define TEC_F_NAME_MISMATCH 16
#define TEC_CHROM_SC_SKIP 0xFFFE
#define TEC_CELL_INVALID 0xFFFFFFFFu

/* bulk statistics block, int64[TEC_BULK_NSTATS]  (te_count.py:158-163, :269-275) */
#define TEC_BULK_NSTATS 8
#define TEC_BS_UNITS 0          /* records (SE) or pairs (PE) consumed; total_reads = this + 1 */
#define TEC_BS_ASSIGNED 1       /* "Reads were assigned to a gene" */
#define TEC_BS_LOWQ 2           /* "Read quality is too low" */
#define TEC_BS_BADCHROM 3       /* "Reads mapped to an invalid chromosome" */
#define TEC_BS_QCFAIL 4         /* "Reads are QC fails" */
#define TEC_BS_CRASH_ENHANCER 5 /* units at which the reference raises NameError (te_count.py:147) */
#define TEC_BS_CRASH_NAME 6     /* units at which the reference dies in sys.quit (te_count.py:94) */
#define TEC_BS_NO_MATE 7        /* pairing by read name: records excluded from pairing plus records left without a
                                   mate (0 in the other modes) */

/* single-cell statistics block, int64[TEC_SC_NSTATS]  (te_count.py:696-705) */
#define TEC_SC_NSTATS 16
#define TEC_SS_UNITS 0          /* records consumed; total_reads = this + 1 */
#define TEC_SS_INVALID_BARCODE 1
#define TEC_SS_ALREADY_SEEN 2
#define TEC_SS_LOWQ 3
#define TEC_SS_QCFAIL 4
#define TEC_SS_VALID 5          /* lines kept by Part 2 ("total valid reads") */
#define TEC_SS_ASSIGNED 6       /* "Assigned N of total valid reads to features" */
#define TEC_SS_RAW_BARCODES 7   /* "Observed N raw barcodes" */
#define TEC_SS_BUNDLES 8        /* spill bundles the reference would have written */
#define TEC_SS_CRASH_STRAND 9   /* fragments at which the reference raises KeyError 'strand' (:661) */
#define TEC_SS_SURVIVORS 10     /* records that reached the UMI table */
#define TEC_SS_SEGMENTS 11      /* (cell, UMI, bundle) lines over all bundles */

/* ---- life cycle ------------------------------------------------------------------------- */
int tec_abi_version(void);
const char* tec_strerror(int status);
/* device: CUDA ordinal.  Replaces measureTE.__init__ state (te_count.py:15-29). */
int tec_create(int device, tec_ctx** out);
void tec_destroy(tec_ctx* ctx);
const char* tec_last_error(const tec_ctx* ctx);
int tec_sync(tec_ctx* ctx);
/* pinned host memory for the SoA batches (optional; any host memory is accepted) */
int tec_host_alloc(tec_ctx* ctx, uint64_t bytes, void** out);
int tec_host_free(tec_ctx* ctx, void* p);
/* the CUDA stream of the context as a cudaStream_t value (for event timing by the caller) */
void* tec_stream(tec_ctx* ctx);
/* elapsed GPU milliseconds of the kernels of the last bulk push / sc finalize on this context */
float tec_last_kernel_ms(tec_ctx* ctx);
/* number of kernel launches issued by this context since creation */
int64_t tec_launch_count(const tec_ctx* ctx);

/* release cached device scratch (the single-cell finalize keeps its temporaries for the next call) */
int tec_trim(tec_ctx* ctx);

/* tuning knobs: "bulk_algo" (-1 auto, 0 exact search kernel, 1 round-1 cell-table kernel -- set before
 * tec_index_upload --, 2 two-pass kernels), "stab_shift" (log2 of the cell size, 8..11, or 0 = default: 10 for
 * bulk, 11 for the single-cell pair table; used by the next tec_index_upload), "bulk_mode" (bit 0 table sectors
 * evict_last in L2, bit 1 sector prefetch, bit 2 tally through the per-warp hit queue, bit 3 deep pipeline, bit 4
 * queue filled behind a warp prefix sum, bit 5 768-thread CTAs, bit 6 queue drained once per tile; default 77),
 * "second_mode" (second bulk pass: the register set of a unit's distinct ensg, 0 stored by position, 1 shifted
 * in, 2 = 1 + the units that two sectors answer go through a straight-line kernel first), "second_parts" (warps
 * per segment of the deferred list), "ctas_per_sm",
 * "all_hot" (counters of every ensg in shared memory when they fit), "sc_algo" (-1 auto, 0 exact search in
 * Part 3, 1 cell table), "sc_pack_umi" (2-bit UMI sort keys when possible), "bulk_loci" (0 / 1: counts per index row,
 * see tec_bulk_loci).
 * tec_get_info: "has_stab", "stab_bytes", "has_sc_stab", "sc_stab_bytes", "n_sm", "n_features", "bulk_counter_words"
 * (length of the block at tec_bulk_counts_dev),
 * "stab_primary", "stab_overflow", "stab_entries", "last_slow_units", "last_deferred_units", "last_left_units"
 * (deferred units the two-sector kernel left for the second pass), "stab_refused",
 * "sc_last_sort" (how the last tec_sc_finalize grouped the survivors by (cell, UMI): 1 one packed 64-bit key per
 * survivor sorted by csrc/radix.cuh, 2 library sorts on 2-bit-per-character UMI keys, 3 library sorts on the 3-bit
 * UMI codes; 0 nothing was sorted), "sc_last_sort_passes" (radix passes of that packed sort, 0 on the other routes);
 * -1 for unknown keys. */
int tec_set_option(tec_ctx* ctx, const char* key, int64_t value);
int64_t tec_get_info(tec_ctx* ctx, const char* key);
/* why the last tec_index_upload could not build the bulk cell table ("" when it could): with such an index
 * (more than 65535 ensg, or an ensg that carries two feature types) bulk counting runs on the exact search kernel,
 * about ten times slower.  The caller should log it (te_counter_b200/te_count.py does). */
const char* tec_index_note(const tec_ctx* ctx);

/* ---- index ------------------------------------------------------------------------------
 * Replaces load_genome() + the structures of genelist._optimiseData that the read loops reach
 * into (te_count.py:31-35, :68-73, :586-590; miniglbase/genelist.py:332-396).
 * Features are grouped by chromosome id and sorted by (L, R) inside each chromosome:
 *   chrom_off[n_chrom + 1]  offsets into the feature arrays
 *   L, R                    loc['left'], loc['right']
 *   ensg_id                 index into sorted(set(ensg))  (== output row / column order)
 *   type_code               TEC_T_*;  strand_code 0 '+', 1 '-', 2..3 other strings, 255 missing
 *   bucket_size             miniglbase/config.py:36 (10000)
 */
int tec_index_upload(tec_ctx* ctx, int32_t n_chrom, const int64_t* chrom_off,
                     const int32_t* L, const int32_t* R, const int32_t* ensg_id,
                     const uint8_t* type_code, const uint8_t* strand_code,
                     int32_t n_ensg, int32_t bucket_size);

/* ---- bulk (parse_bamse te_count.py:167-277, parse_bampe te_count.py:42-165) ---------------
 * begin: zero the per-feature counters and statistics.  paired != 0 consumes records two at a
 * time (record 2i = read1, 2i+1 = read2); every push must then hold an even number of records.
 * push: filter + mate merge + point overlap + type rule + tally for one batch, host buffers.
 * push_dev: the same with DEVICE pointers, asynchronous on the context stream.
 * finish: counts[n_ensg] and stats[TEC_BULK_NSTATS] to host (either may be NULL).
 */
int tec_bulk_begin(tec_ctx* ctx, int paired, int qual);
/* Paired end by read name: tec_bulk_begin(ctx, 2, qual).  For files whose mates are not adjacent (coordinate-sorted
 * BAMs).  The rule:
 *   - a record takes part when it is primary and carries exactly one mate flag: 0x1 set, 0x100 and 0x800 clear, exactly
 *     one of 0x40 (read1) / 0x80 (read2).  Every other record is excluded: neither paired nor counted;
 *   - records are grouped by their exact QNAME bytes (through a 128-bit key of two independent 64-bit hashes,
 *     bgzf_dev.h name_key).  Within a name, the k-th read1 in input order pairs with the k-th read2 in input order;
 *   - each pair is counted as a pair of paired = 1 whose record 2i is that read1 and 2i+1 that read2 (filters on both
 *     mates, read1's MAPQ and chromosome, both starts).  Mates have identical names, so the name check never fires.
 * Records arrive through tec_bulk_push_named, tec_bam_count(b, 3, ...) or the byte ranges of mode 4 (below) only; the other
 * pushes, and tec_bam_count and tec_bam_count_range in modes 0-2, return TEC_ERR_STATE until the next begin.  tec_bulk_finish and tec_bulk_allreduce end
 * the input: records still waiting for a mate count as no-mate.  stats[TEC_BS_NO_MATE] = excluded + no-mate records.
 * tec_get_info: "bulk_name_excluded" (excluded records), "bulk_name_pending_peak" (largest number of records waiting for
 * their mate after a batch), "bulk_name_ms" (device milliseconds of the pairing stage: sorts and group pass).  A batch
 * needs fewer than 2^32 - 2^13 records together with the ones still waiting (TEC_ERR_LIMIT); a device allocation that
 * fails returns TEC_ERR_NOMEM.
 * tec_bulk_push_named: n records in the usual layout plus samflag[n] (the SAM flag) and the QNAME of record i as bytes
 * [name_off[i], name_off[i+1]) of `names` (name_off[0] = 0, at most 254 bytes each).  Synchronous. */
int tec_bulk_push_named(tec_ctx* ctx, int64_t n, const int32_t* start, const int32_t* end, const uint16_t* chrom,
                        const uint8_t* mapq, const uint8_t* flag, const uint16_t* samflag, const int64_t* name_off,
                        const char* names);
int tec_bulk_push(tec_ctx* ctx, int64_t n_rec, const int32_t* start, const int32_t* end,
                  const uint16_t* chrom, const uint8_t* mapq, const uint8_t* flag);
int tec_bulk_push_dev(tec_ctx* ctx, int64_t n_rec, const int32_t* start, const int32_t* end,
                      const uint16_t* chrom, const uint8_t* mapq, const uint8_t* flag);
int tec_bulk_finish(tec_ctx* ctx, int64_t* counts, int64_t* stats);
/* device address of the int64 counters [n_ensg] followed by stats [TEC_BULK_NSTATS] (and, in a run with loci, the
 * row counters [n_features]); lets the caller run the cross-GPU reduction (NCCL) on the library's buffer without a
 * host round trip.  The block is tec_get_info(ctx, "bulk_counter_words") words long; a begin with loci may move it.
 * The counters are in the library's internal order (the same on every rank for the same index);
 * tec_bulk_finish returns them in ensg-id order. */
void* tec_bulk_counts_dev(tec_ctx* ctx);
/* Counts per index row ("loci"; an extension outside the parity claim): tec_set_option(ctx, "bulk_loci", 1) before
 * tec_bulk_begin, read at the begin and held until the next one.  The rule, in every bulk mode (single end, paired end
 * by index or by name):
 *   - filters, mate merge, candidate rule, point tests, type rule and statistics are unchanged;
 *   - a unit is counted exactly when the per-name tally adds to it: its hit rows include a gene, TE or snRNA type.
 *     A counted unit adds 1 to every row it hits, once per row;
 *   - a unit that is not counted adds nothing (no hit, only uncounted types, the enhancer crash unit);
 *   - with "bulk_strand", rows the strand filter removes are not hits.
 * So for every name e, the sum over the rows of e is at least count[e], and equal when no unit hits two rows of e;
 * per-name counts and statistics are those of a run without loci.  The run uses the exact search kernel.  The counter
 * block grows by n_features words (all-reduce, bank copy and name exchange carry them).
 * tec_bulk_loci: counts[n_features] in the row order of tec_index_upload.  Same checks as tec_bulk_finish (and the same
 * flush of rows still waiting for a mate); TEC_ERR_STATE when the run did not begin with loci. */
int tec_bulk_loci(tec_ctx* ctx, int64_t* counts);
/* ---- single cell (sc_parse_bamse te_count.py:298-707, sc_save_result :709-754) ------------ */
int tec_sc_begin(tec_ctx* ctx, int qual, int strand, int64_t n_whitelist);
int tec_sc_push(tec_ctx* ctx, int64_t n_rec, const int32_t* start, const int32_t* end,
                const uint16_t* chrom, const uint8_t* mapq, const uint8_t* flag,
                const uint32_t* cell, const uint64_t* umi);
int tec_sc_push_dev(tec_ctx* ctx, int64_t n_rec, const int32_t* start, const int32_t* end,
                    const uint16_t* chrom, const uint8_t* mapq, const uint8_t* flag,
                    const uint32_t* cell, const uint64_t* umi);
/* Parts 1-3: bundle_keys is the 1e7 of te_count.py:377, pad the +1000 of :502.
 * Returns the sizes of the two result lists. */
int tec_sc_finalize(tec_ctx* ctx, int64_t bundle_keys, int64_t maxcells, int64_t pad,
                    int64_t* n_triples, int64_t* n_hit_cells);
/* triples sorted by (ensg, cell): final_results[ensg][barcode] = count (te_count.py:668-682);
 * hit cells ascending by cell id: self.barcodes after Part 3 (te_count.py:653-655);
 * stats[TEC_SC_NSTATS].  Any pointer may be NULL. */
int tec_sc_fetch(tec_ctx* ctx, int32_t* ensg, uint32_t* cell, int64_t* count,
                 uint32_t* hit_cell, int64_t* hit_count, int64_t* stats);
/* ---- single cell on several GPUs (one process per GPU; SURVEY.md 8e) -------------------------
 * The (cell, UMI) collapse is per cell, so after Part 1's filter the survivors are exchanged by cell
 * (all-to-all, done by the caller on the packed records of tec_sc_partition_dev), each carrying its
 * position in the job-wide survivor order.  tec_sc_finalize then runs the same pipeline per rank and calls the
 * collective at the few points that are global: the bundle boundaries of te_count.py:377 (a running
 * count over the whole file), the per-cell raw counts and first appearances behind the top-cell
 * choice (:502), the per-bundle cell presence behind the held-line rule (:528), the per-cell hit
 * counts (:653) and the statistics.  Triples stay on the rank that owns the cell.
 *   fn(user, dev_ptr, count, dtype, op): in-place all-reduce of a device buffer over the ranks;
 *   dtype 0 u32, 1 u64, 2 i64; op 0 sum, 1 min, 2 max; returns 0 on success. */
typedef int (*tec_allreduce_fn)(void* user, void* dev_ptr, int64_t count, int dtype, int op);
int tec_sc_set_collective(tec_ctx* ctx, tec_allreduce_fn fn, void* user, int rank, int world);
/* number of survivors held after the pushes */
int tec_sc_survivors(tec_ctx* ctx, int64_t* n);

/* the exchange: survivors packed as 32-byte records {u64 umi, u64 position,
 * u32 cell, u32 cs, i32 left, i32 right} grouped by owner rank cell % world (at most 8 ranks), file
 * order kept inside a group; counts[world] (host) are the group sizes, *records the device buffer.
 * After the all-to-all (received groups concatenated by source rank) hand the records back with
 * tec_sc_import_packed_dev. */
int tec_sc_partition_dev(tec_ctx* ctx, int world, int64_t gidx_base, int64_t* counts, void** records);
int tec_sc_import_packed_dev(tec_ctx* ctx, int64_t n, const void* records);

/* ---- collectives issued by the library (NCCL, bound at run time with dlopen; SURVEY.md 8b proposed
 * tec_reduce(ctx, ncclComm), 8e lists the exchange steps) ---------------------------------------
 * One communicator per context: rank 0 calls tec_comm_unique_id, the TEC_COMM_ID_BYTES bytes travel to
 * the other ranks by any means (te_counter_b200/dist.py: torch.distributed broadcast), every rank calls
 * tec_comm_init.  From then on the library runs its collectives itself, on its own stream and buffers:
 *   tec_bulk_allreduce        sum of the ranks' counter blocks, in place, behind the pushes; tec_bulk_finish
 *                             then returns the job's counts on every rank (te_count.py:128-149 summed)
 *   tec_sc_exchange           after the pushes: all-to-all of the survivors by owner rank cell % world
 *                             (tec_sc_partition_dev + grouped send / receive + tec_sc_import_packed_dev);
 *                             tec_sc_finalize then all-reduces through NCCL where tec_sc_set_collective
 *                             would have called back
 *   tec_sc_allgather_triples  after tec_sc_finalize: every rank holds the job's triples, ascending in
 *                             (ensg, cell); tec_sc_fetch returns them
 *   tec_bulk_name_exchange    after tec_bam_count_range(b, 4, ...): partition, all-gather of the group sizes, grouped
 *                             send / receive, import (see tec_bulk_name_partition_dev).  The ranks agree on success
 *                             before any record moves (the receive buffer and the pairing stage's rows are allocated
 *                             first): a rank that fails makes every rank return its status
 * Every rank must make the same sequence of these calls.  TEC_ERR_UNSUPPORTED: libnccl.so.2 not found. */
#define TEC_COMM_ID_BYTES 128
int tec_comm_unique_id(tec_ctx* ctx, void* id, int32_t capacity);
int tec_comm_init(tec_ctx* ctx, const void* id, int32_t rank, int32_t world);
int tec_comm_destroy(tec_ctx* ctx);
int tec_comm_info(tec_ctx* ctx, int32_t* rank, int32_t* world);
int tec_bulk_allreduce(tec_ctx* ctx);
int tec_sc_exchange(tec_ctx* ctx, int64_t* n_owned);
int tec_sc_allgather_triples(tec_ctx* ctx, int64_t* n_triples);
int tec_bulk_name_exchange(tec_ctx* ctx, int64_t* n_owned);

/* sc_save_result's choice of rows (te_count.py:724-733): hit cells by count descending, ties by
 * ascending id, at most maxcells.  cells_out must hold min(maxcells, n_hit_cells) entries. */
int tec_sc_select(tec_ctx* ctx, int64_t maxcells, uint32_t* cells_out, int64_t* n_out);

/*
 * Dense matrix rows of sc_save_result as text (te_count.py:744-754), built on the device: for each of
 * the n_rows cells, in the order given (normally tec_sc_select's), one line
 *     <barcode> '\t' <count of ensg 0> '\t' <count of ensg 1> ... '\n'
 * with every ensg of the index in id (= sorted name) order, zeros included, decimal integers.
 * cells[r] = whitelist id of row r (each at most once); barcodes = the rows' barcode strings
 * concatenated, row r is bytes [bc_off[r], bc_off[r+1]).  *n_bytes = length of the text, which stays
 * in device memory until the next tec_sc_matrix_text / tec_sc_begin; tec_sc_matrix_read copies the
 * byte range [offset, offset + n) of it into host memory (stream it to the file in chunks).
 * The header line (te_count.py:745) is the caller's: it is made of the feature names.
 */
int tec_sc_matrix_text(tec_ctx *ctx, int64_t n_rows, const uint32_t *cells, const char *barcodes,
                       const int64_t *bc_off, int64_t *n_bytes);
int tec_sc_matrix_read(tec_ctx *ctx, int64_t offset, int64_t n, char *out);

/*
 * The cell x feature matrix of sc_save_result as the text of a Matrix Market file, 10x orientation: one row per feature
 * (ensg id order = the dense TSV's columns), one column per given cell (cells[k] = whitelist id of column k, each at
 * most once; normally tec_sc_select's order).  Text = "%%MatrixMarket matrix coordinate integer general\n",
 * "<n_ensg> <n_cols> <nnz>\n", then one line "<ensg + 1> <k + 1> <count>\n" per non-zero, ascending in (k, ensg).
 * *nnz = entries written, *n_bytes = text length.  The text replaces the one tec_sc_matrix_text keeps and is read
 * with tec_sc_matrix_read.  n_cols == 0 gives the two header lines only.
 */
int tec_sc_matrix_mtx(tec_ctx *ctx, int64_t n_cols, const uint32_t *cells, int64_t *nnz, int64_t *n_bytes);

/* ---- BAM file -> counting path, decoded on the device (SURVEY.md 8f-1; te_count.py:65-98, :190-214, :351-438)
 *
 * The same job as libtecbam (include/tecbam.h: BGZF inflate, record split, fields -> SoA columns, same
 * field semantics and the same error conditions) done by CUDA kernels with one thread per BGZF block,
 * with the columns handed to tec_bulk_push_dev / tec_sc_push_dev without leaving the device.  The host
 * reads the compressed file into pinned memory and walks the per-block results once per window (an
 * exact check of the record chain).  Usage: tec_bam_open, read the reference names, tec_bam_set_chrom_map
 * (and tec_bam_set_whitelist) exactly as for tbam_*, tec_bulk_begin / tec_sc_begin, tec_bam_count (decodes
 * the whole file into the running count), tec_bulk_finish / tec_sc_finalize, tec_bam_close.
 * mode: 0 single end, 1 paired end, 2 single cell, 3 paired end by read name (tec_bulk_begin(ctx, 2, qual); whole files
 * only: tec_bam_count_range refuses it with TEC_ERR_ARG and takes mode 4 instead, below).  On TEC_ERR_UNSUPPORTED start over with libtecbam.
 * Options (tec_set_option): "bam_window_blocks" (BGZF blocks per pass, default 65536: 4.3 GB of inflated bytes
 * in HBM), "bam_lanes" (blocks decoded per warp, default 1).  Limits shared with libtecbam: reference_end comes
 * from the CIGAR field of the record (for alignments of more than 65535 operations that field is the placeholder
 * <l_seq>S<ref_len>N of SAMv1 4.2.2, whose N operation carries the reference length: no expansion of the CG tag is
 * needed); tag values are compared as bytes. */
typedef struct tec_bam tec_bam;
int tec_bam_open(tec_ctx *ctx, const char *path, tec_bam **out);
void tec_bam_close(tec_bam *b);
int tec_bam_n_references(const tec_bam *b);
const char *tec_bam_reference_name(const tec_bam *b, int i);
int tec_bam_set_chrom_map(tec_bam *b, const uint16_t *bulk_ids, const uint16_t *sc_ids, int32_t n, int32_t n_index);
int tec_bam_set_whitelist(tec_bam *b, const char *barcodes, const int64_t *offsets, int32_t n);
int tec_bam_count(tec_bam *b, int mode, int qual, int64_t *n_records);
/* One BYTE RANGE of the file, for several ranks that split one BAM.  Counts the records that START in the BGZF blocks
 * whose first byte lies in [byte_lo, byte_hi) into the running count.  out[TEC_BAM_RANGE_WORDS] = {records counted, start_block,
 * start_off, exit_block, exit_off, file size}: where this range's first record starts and where the chain stands
 * behind its last record, each as {file offset of the BGZF block, offset in its inflated data}.  start_block -1: the
 * range began at the BAM header (byte_lo == 0, exact); -2: no record starts in the range.  The first record of any other
 * range is the block-parallel guess, so the CALLER must check exit(rank) == start(next rank with records) for every
 * rank and exit(last) == {file size, 0}; if that fails, decode the file in one piece (te_count.py does both). */
#define TEC_BAM_RANGE_WORDS 6
int tec_bam_count_range(tec_bam *b, int mode, int qual, int64_t byte_lo, int64_t byte_hi, int64_t *out);
/* Paired end (mode 1) over byte ranges.  The reference pairs records by their GLOBAL index (record 2i is read1,
 * 2i+1 read2, a trailing odd record is dropped), which a range does not know until the ranges in front of it are
 * counted.  So tec_bam_count_range(b, 1, ...) counts every adjacent pair (j, j+1) of the range (j = range-local index)
 * into one of two counter banks, bank j & 1, both starting from the running count; out[0] is still the number of
 * records.  Once the caller knows the range's global offset o (the sum of the record counts of the ranges in front):
 *   tec_bulk_keep_bank(ctx, o & 1)   makes that bank the running count and drops the other.  Until it is called,
 *                                    tec_bulk_push*, tec_bulk_allreduce, tec_bulk_finish, tec_bam_count and
 *                                    tec_bam_count_range return TEC_ERR_STATE; tec_bulk_begin clears that state.
 *   if o is odd and the range has records, its first record is read2 of a pair whose read1 is the last record of the
 *   nearest range in front that has records: tec_bam_pair_columns parses the two, tec_bulk_push counts them.
 * tec_bam_range_record: raw bytes (block_size word included) of the first (which = 0) or last (which = 1) record of
 * the last paired-end tec_bam_count_range on b; *len = their number (0: no record, or another mode).  buf = NULL only
 * asks for the length; otherwise cap must be at least *len.
 * tec_bam_pair_columns: read1 = rec1[0, n1), read2 = rec2[0, n2), each one raw record of this file, parsed on the host
 * with b's chromosome map into rows 0 and 1 (the record layout above), with the same rules and the same status as the
 * device parse (TEC_ERR_FORMAT for a malformed record, TEC_ERR_ARG when a buffer is not one whole record). */
int tec_bulk_keep_bank(tec_ctx *ctx, int bank);
/* Paired end by read name over byte ranges.  A mate may lie in any range, so tec_bam_count_range(b, 4, ...) (after
 * tec_bulk_begin(ctx, 2, qual)) pairs and counts nothing: the rows of the range's records (one per record, with name key and
 * role) are appended in file order to a HELD set; out[] means what it means in single-end mode.  Then every rank:
 *   tec_bulk_name_partition_dev(ctx, world, counts, &records)   counts the held excluded records (bulk_name_excluded,
 *       stats[TEC_BS_NO_MATE]) and drops them, and packs the others as 32-byte records grouped by owner rank
 *       key_lo % world (1..8 ranks; key_lo is a splitmix64 output), file order kept inside a group; counts[world] (host)
 *       are the group sizes, *records the device buffer (valid until the next import, partition or begin on ctx);
 *   the caller moves group r of every rank to rank r (an all-to-all), received groups laid out by source rank;
 *   tec_bulk_name_import_dev(ctx, n, records)   takes the n received records (device pointer), which are then in file
 *       order, and pairs them in one pass of the pairing stage; records left without a mate stay pending, so
 *       tec_bulk_finish / tec_bulk_allreduce count them as no-mate.
 * Summed over the ranks the counters and statistics equal those of one tec_bam_count(b, 3, ...) of the whole file.
 * tec_bulk_name_exchange does the three steps over the communicator of tec_comm_init (below) and returns the number of
 * records this rank received.
 * State: while held rows wait for the partition, the pushes, tec_bam_count, tec_bulk_finish and tec_bulk_allreduce
 * return TEC_ERR_STATE; tec_bulk_begin drops the held rows.  Mode 4 in a run that has records pushed into the pairing
 * stage returns TEC_ERR_STATE.  The limit of 2^32 - 2^13 records per pairing pass applies to the records one rank holds
 * and to those one owner receives (TEC_ERR_LIMIT). */
int tec_bulk_name_partition_dev(tec_ctx *ctx, int world, int64_t *counts, void **records);
int tec_bulk_name_import_dev(tec_ctx *ctx, int64_t n, const void *records);
int tec_bam_range_record(const tec_bam *b, int which, void *buf, int64_t cap, int64_t *len);
int tec_bam_pair_columns(tec_bam *b, const void *rec1, int64_t n1, const void *rec2, int64_t n2, int qual,
                         int32_t *start, int32_t *end, uint16_t *chrom, uint8_t *mapq, uint8_t *flag);
/* what = 0 blocks inflated by zlib on the host, 1..4 microseconds in load / inflate / chain / parse */
int64_t tec_bam_info(const tec_bam *b, int what);

#ifdef __cplusplus
}
#endif
#endif /* TECOUNT_H */
