"""
Drop-in mirror of the reference's `measureTE` (te_count/te_count.py:14-754) whose read loops run
on the GPU through libtecount.so.

Same method names, arguments, return types, side effects (`self.total_reads`, `self.barcodes`),
log lines and exceptions as the reference; the differences are:
  * records are pulled from pysam in batches, repacked into pinned structure-of-arrays buffers
    (te_counter_b200/reads.py) and counted by CUDA kernels -- there is no Python per-read
    overlap/tally and no CPU fallback;
  * the single-cell spill bundles (tmp.*.bun, te_count.py:357-390, :506-575) are never written:
    their observable effects (bundle boundaries, the Part-2 held-line drop, first-bundle-wins) are
    reproduced on the device;
  * the hash-seed dependent `next(iter(set))` at te_count.py:452 is replaced by the canonical
    "first inserted fragment" (SURVEY.md 8a-9);
  * sc results come back as a lazy read-only mapping `ScResult` (same keys / inner dicts as the
    reference's dict of dicts) so that a 10k-cell matrix is not expanded into Python dicts unless
    the caller asks for it.
"""
import os
import random
from collections.abc import Mapping
from operator import itemgetter

import numpy as np

from . import _lib
from . import fastbam as _fastbam
from . import index as _index
from . import loci as _loci
from . import mtx as _mtx
from . import reads as _reads
from . import shard as _shard

BATCH_RECORDS = 1 << 20
SC_BUNDLE_KEYS = 10000000        # te_count.py:377  `len(umis) >= 1e7`
SC_CELL_PAD = 1000               # te_count.py:502  `maxcells+1000`


def _open_alignment(filename, tags_optional=False, by_name=False):
    """Host readers.  tags_optional (the --noumi extension): only the readers with pysam's interface, whose
    records are packed by reads.fill_sc, can leave the UMI tags unread.  by_name (parse_bampe(pairing='name')): only
    they hand out QNAMEs and SAM flags (reads.fill_bulk_named); libtecbam does not.
      TEC_BAM_DECODER = auto (default) | gpu | native | pysam | python.  `auto` / `gpu`:
    the callers first try the device decoder (tec_bam_*) and come here only for files it refuses;
    then block-compressed BAM goes through libtecbam (threads inflate and parse into the pinned
    batch, fastbam.py) when it is built; anything else through pysam as in the reference
    (te_count.py:11, :65), or through the pure-Python stand-in with pysam's interface (bam.py) where
    pysam is not installed."""
    mode = os.environ.get('TEC_BAM_DECODER', 'auto')
    if mode not in ('auto', 'gpu', 'native', 'pysam', 'python'):
        raise ValueError('TEC_BAM_DECODER must be auto, gpu, native, pysam or python')
    if mode == 'gpu':
        mode = 'auto'
    if not (tags_optional or by_name) and (mode == 'native' or (mode == 'auto' and _fastbam.available())):
        try:
            return _fastbam.NativeBam(filename)
        except (_fastbam.NotBgzf, OSError):             # SAM text, plain gzip, not a regular file: next reader
            if mode == 'native':
                raise
    if mode != 'python':
        try:
            import pysam
            return pysam.AlignmentFile(filename, 'r')
        except ImportError:
            if mode == 'pysam':
                raise
    from . import bam as _bam
    return _bam.AlignmentFile(filename, 'r')


def _device_decoder_wanted(eng):
    """`auto` and `gpu`: decode the BAM on the device (tec_bam_*: 2.7x the 16 host cores of the B200 box);
    files it refuses (SAM text, record layouts it cannot split block-parallel) go to the host readers."""
    return os.environ.get('TEC_BAM_DECODER', 'auto') in ('auto', 'gpu') and hasattr(eng, 'bam_open')


class ScResult(Mapping):
    """final_results of sc_parse_bamse (te_count.py:583, :668-682): {ensg: {barcode: count}} for
    every ensg (empty dict when nothing hit).  Backed by the (ensg, cell, count) triples the
    engine returns, sorted by (ensg, cell)."""

    def __init__(self, names, id_to_barcode, ensg, cell, count):
        self._names = names
        self._row = {n: i for i, n in enumerate(names)}
        self._id_to_barcode = id_to_barcode
        self.ensg, self.cell, self.count = ensg, cell, count
        self._ptr = np.searchsorted(ensg, np.arange(len(names) + 1))
        self._cache = {}

    def __len__(self):
        return len(self._names)

    def __iter__(self):
        return iter(self._names)

    def __contains__(self, k):
        return k in self._row

    def __getitem__(self, k):
        d = self._cache.get(k)
        if d is None:
            i = self._row[k]
            a, b = self._ptr[i], self._ptr[i + 1]
            bc = self._id_to_barcode
            d = {bc[c]: v for c, v in zip(self.cell[a:b].tolist(), self.count[a:b].tolist())}
            self._cache[k] = d
        return d


class measureTE:
    def __init__(self, base_path, quality_threshold, device=None, extensions=None):
        '''
        **Arguments**
            base_path (Required)
                the path we are being run in
            quality_threshold
                MAPQ threshold
            device (extension)
                CUDA ordinal; default LOCAL_RANK or 0
            extensions (extension; default: the environment variable TEC_EXTENSIONS == '1')
                Defined semantics for flag combinations on which the reference raises (SURVEY.md 8f-4).
                Off: every one of them raises exactly what the reference raises.  On:
                  -q N       a one-element list (bin/te_count:30 hands one over) means its element
                  --strand   in bulk mode: a feature on '+' / '-' is only a candidate for units whose first
                             record is on that strand (exact-search kernel; te_count.py:58-59 raises)
                  --noumi    every surviving record is its own molecule (te_count.py:429-442, :703 raise)
                Nothing here is part of the parity claim; oracle/te_oracle_ext.py restates the rules.
        '''
        self.extensions = (os.environ.get('TEC_EXTENSIONS') == '1') if extensions is None else bool(extensions)
        self.base_path = base_path
        self.total_reads = 0
        self.quality_threshold = quality_threshold
        self.random_number = f'{random.randint(1000, 100000):06d}'
        self.device = int(os.environ.get('LOCAL_RANK', 0)) if device is None else device
        self._engine_obj = None
        self._index_on_device = False
        self.genome = None
        self.locus_counts = None

    # ---------------------------------------------------------------- engine plumbing
    def _engine(self):
        if self._engine_obj is None:
            self._engine_obj = _lib.Engine(self.device)      # raises without a GPU / built library
        if not self._index_on_device:
            self._engine_obj.upload_index(self.genome)
            self._index_on_device = True
            note = self._engine_obj.index_note()
            if note:                                         # no silent slow path (exact search kernel, ~10x slower in bulk)
                import logging
                logging.getLogger('te_count').warning(
                    'bulk cell table not built (%s): bulk counting uses the exact search kernel, about ten times slower', note)
        return self._engine_obj

    def _qual(self):
        q = self.quality_threshold
        if self.extensions and isinstance(q, (list, tuple)) and len(q) == 1 and isinstance(q[0], (int, np.integer)):
            return int(q[0])                                 # extension: -q N
        if not isinstance(q, (int, np.integer)):
            # bin/te_count:30 hands over a list when -q is given; te_count.py:88 then raises
            raise TypeError("'<' not supported between instances of 'int' and '%s'" % type(q).__name__)
        return int(q)

    # ---------------------------------------------------------------- genome
    def load_genome(self):
        assert self.genelist_glb_filename, 'You need to bind the genome first'
        self.genome = _index.load_glb(self.genelist_glb_filename)
        self.all_feature_names = self.genome.names            # sorted(set(ensg)), te_count.py:35
        self._index_on_device = False

    def bind_genome(self, genelist_glb_filename):
        # For delayed loading
        assert os.path.isfile(genelist_glb_filename), f'{genelist_glb_filename} not found'
        self.genelist_glb_filename = genelist_glb_filename

    # ---------------------------------------------------------------- bulk
    def _parse_bulk(self, filename, strand, log, paired, pairing='index', loci=False):
        assert filename, 'You must specify a filename'
        if pairing not in ('index', 'name'):
            raise ValueError("pairing must be 'index' or 'name', not %r" % (pairing,))
        if strand and not self.extensions:
            raise NotImplementedError()                       # te_count.py:58-59 / :183-184
        qual = self._qual()
        self.locus_counts = None
        eng = self._engine()
        eng.set_option('bulk_strand', 1 if strand else 0)     # extension: strand-aware candidates (exact-search kernel)
        eng.set_option('bulk_loci', 1 if loci else 0)         # extension: counts per index row (exact-search kernel)
        try:
            return self._parse_bulk_run(eng, filename, log, paired, qual, pairing == 'name', loci)
        finally:
            eng.set_option('bulk_strand', 0)
            eng.set_option('bulk_loci', 0)

    def _parse_bulk_run(self, eng, filename, log, paired, qual, by_name=False, loci=False):
        cm = _reads.ChromMap(self.genome.chrom_keys)
        label = 'reads' if paired else 'SE reads'
        more, done, next_log = True, 0, 1000000
        # pairing by read name: pairs are only known once the pairing stage has seen their mates, so the progress lines
        # are written from the final pair count
        begin = (lambda: eng.bulk_begin(paired, qual, pairing='name')) if by_name else (lambda: eng.bulk_begin(paired, qual))
        # One file, several ranks (torch.distributed job, one process per GPU; shard.py): every rank decodes a byte range
        # on its GPU and the counters are summed; paired end keeps the counter bank of the rank's record parity and
        # counts the pair across its front border; paired end by read name sends the rows of its range to the ranks that
        # own their names, and each owner pairs what it receives.  Files whose ranges the decoders cannot tile are decoded
        # by rank 0 alone; the sum is the same.
        rank, world = _shard.world_info()
        in_library = _shard.join_collectives(eng) if world > 1 else False
        if world > 1:
            sharded = None
            if _device_decoder_wanted(eng):
                def open_and_bind():
                    dev = eng.bam_open(filename)
                    dev.bind(cm)
                    return dev
                begin()
                sharded = _shard.count_ranges(open_and_bind, 4 if by_name else 1 if paired else 0, qual)
            if sharded is not None:
                done, more = sharded[1], False
                if by_name:
                    import torch
                    from . import dist as _tdist
                    _tdist.bulk_name_exchange(eng, torch.device('cuda', self.device))
                    done = 0
                elif paired:
                    bank, border = sharded[2]
                    eng.bulk_keep_bank(bank)
                    if border is not None:
                        eng.bulk_push(2, border['start'], border['end'], border['chrom'], border['mapq'], border['flag'])
                    done //= 2
                log.info('{:,} of them decoded by this rank ({} of {})'.format(sharded[0], rank, world))
            elif rank != 0:
                begin()                                       # nothing to decode here: rank 0 reads the whole file
                more = False
        if more and _device_decoder_wanted(eng):
            try:                                              # BGZF inflate, record split and packing on the device
                dev = eng.bam_open(filename)
                try:
                    dev.bind(cm)
                    begin()
                    done = dev.count(3 if by_name else 1 if paired else 0, qual)
                    done = 0 if by_name else done // 2 if paired else done
                    more = False
                    self._bam_info = dev.info()
                finally:
                    dev.close()
            except (_lib.BamUnsupported, OSError):
                more = True                                   # start over with a host reader
            except _lib.TecError as e:
                if e.status != _lib.ERR_NOMEM:                # no room for the decode window next to the other
                    raise                                     # buffers of this GPU: decode on the host instead
                eng.trim()                                    # the decoder's buffers went back to the block cache
                more = True
            while done >= next_log:
                log.info('Processed {:,} {}'.format(next_log, label))
                next_log += 1000000
        sam = batch = None
        if more:
            done, next_log = 0, 1000000
            sam = _open_alignment(filename, by_name=by_name)
            native = isinstance(sam, _fastbam.NativeBam)
            if native:
                sam.bind(cm)
            batch = _reads.Batch(BATCH_RECORDS, alloc=eng.pinned, named=by_name)
            begin()
        while more and by_name:
            more = _reads.fill_bulk_named(batch, sam, cm)
            eng.bulk_push_named(batch.n, batch.start, batch.end, batch.chrom, batch.mapq, batch.flag, batch.samflag,
                                batch.name_off, batch.names)
        while more:
            more = sam.fill_bulk(batch, paired, qual) if native else _reads.fill_bulk(batch, sam, cm, paired, qual)
            eng.bulk_push(batch.n, batch.start, batch.end, batch.chrom, batch.mapq, batch.flag)
            done += batch.n // 2 if paired else batch.n
            while done >= next_log:
                log.info('Processed {:,} {}'.format(next_log, label))
                next_log += 1000000
        if sam is not None:
            sam.close()
        if world > 1 and in_library:
            eng.bulk_allreduce()                              # NCCL, issued by the library on its stream (row counters too)
        counts, st = eng.bulk_finish()
        rows = eng.bulk_loci() if loci else np.zeros(0, np.int64)
        if world > 1 and not in_library:
            from . import dist as _tdist
            both, st = _tdist.allreduce_counts_host(np.concatenate([counts, rows]), st)
            counts, rows = both[:len(counts)], both[len(counts):]
        if by_name:
            while int(st[_lib.BS_UNITS]) >= next_log:
                log.info('Processed {:,} {}'.format(next_log, label))
                next_log += 1000000
        if st[_lib.BS_CRASH_NAME]:
            log.error('Unmatched pair!')
            raise AttributeError("module 'sys' has no attribute 'quit'")      # te_count.py:94
        if st[_lib.BS_CRASH_ENHANCER]:
            raise NameError("name 'barcode' is not defined")                  # te_count.py:147 / :260
        idx = int(st[_lib.BS_UNITS]) + 1                     # idx += 1 precedes next(), :77 / :202
        if not paired:
            log.info('Processed {:,} SE reads'.format(idx))
        log.info('Processed {:,} reads'.format(idx))
        log.info('{:,} Reads were assigned to a gene'.format(int(st[_lib.BS_ASSIGNED])))
        log.info('{:,} Read quality is too low (<{})'.format(int(st[_lib.BS_LOWQ]), self.quality_threshold))
        log.info('{:,} Reads mapped to an invalid chromosome'.format(int(st[_lib.BS_BADCHROM])))
        log.info('{:,} Reads are QC fails'.format(int(st[_lib.BS_QCFAIL])))
        if by_name:
            excluded = eng.get_info('bulk_name_excluded')
            if world > 1:                                     # every rank counted the excluded records it decoded
                import torch.distributed as dist
                parts = [None] * world
                dist.all_gather_object(parts, excluded)
                excluded = sum(parts)
            log.info('{:,} records were not paired by name: {:,} not primary or without exactly one mate flag, {:,} without '
                     'a mate'.format(int(st[_lib.BS_NO_MATE]), excluded, int(st[_lib.BS_NO_MATE]) - excluded))
        self.total_reads = idx
        if loci:                                              # device rows -> linearData order
            self.locus_counts = np.empty(len(rows), np.int64)
            self.locus_counts[self.genome.sorted_layout()['order']] = rows
        return dict(zip(self.all_feature_names, counts.tolist()))

    def parse_bampe(self, filename, strand=False, log=None, pairing='index', loci=False):
        '''Load in a BAMPE file (reference te_count.py:42-165).

        pairing (extension): 'index' (default) pairs records as the reference does, record 2i with record 2i+1, which is
        only right for a name-collated file.  'name' pairs the k-th read1 of a read name with its k-th read2 wherever
        they lie (coordinate-sorted BAMs: STAR SortedByCoordinate, samtools sort); only primary records with exactly one
        of the flags 0x40 / 0x80 (and 0x1) take part.  The result equals the reference's on the name-collated pairs.
        loci (extension): also count per index row, see parse_bamse.'''
        return self._parse_bulk(filename, strand, log, True, pairing, loci)

    def parse_bamse(self, filename, strand=False, log=None, loci=False):
        '''Load in a BAMSE file (reference te_count.py:167-277)

        loci (extension): in the same run, count per index row (one TE copy, one gene row): every unit the per-name
        tally counts adds 1 to each row it hits.  The returned dict is unchanged; self.locus_counts then holds
        int64[n_features] in linearData order (None without loci) and save_result_loci writes it.'''
        return self._parse_bulk(filename, strand, log, False, loci=loci)

    def save_result_bulk(self, result, out_filename, log=None):
        '''Save the data to a TSV file (reference te_count.py:279-296): name, count, CPM where
        CPM = count / (total_reads / 1e6) printed with float repr.'''
        assert out_filename, 'You must specify a filename'
        per_million = self.total_reads / 1e6
        with open(out_filename, 'w') as oh:
            oh.write(''.join('{0}\t{1}\t{2}\n'.format(k, result[k], result[k] / per_million)
                             for k in sorted(result.keys())))
        log.info('Saved {0}'.format(out_filename))

    def save_result_loci(self, out_filename, log=None):
        '''Extension: the counts per index row of the last parse_bamse / parse_bampe(..., loci=True) as a TSV
        (te_counter_b200/loci.py): a header, then one line per index row in linearData order -- so the files of several
        samples on one index line up row for row -- with ensg, chromosome key, left, right, strand ('.' when the row
        has none), count and the CPM of save_result_bulk.'''
        assert out_filename, 'You must specify a filename'
        if self.locus_counts is None:
            raise ValueError('no counts per index row: call parse_bamse / parse_bampe with loci=True first')
        text = _loci.tsv_text(self.genome, self.locus_counts, self.total_reads)
        with open(out_filename, 'wb') as oh:
            oh.write(text)
        if log is not None:
            log.info('Saved {0}'.format(out_filename))

    # ---------------------------------------------------------------- single cell
    def sc_parse_bamse(self,
        filename:str,
        UMIS:bool = True,
        whitelistfilename:str = None,
        strand:bool = False,
        log=None,
        label:str = None,
        maxcells:int = None,
        _bundle_keys:int = SC_BUNDLE_KEYS,
        _pad:int = SC_CELL_PAD):
        '''Single-cell counting (reference te_count.py:298-707).  `_bundle_keys` / `_pad` expose the
        two literals of te_count.py:377 and :502 for tests; leave them alone for parity.'''
        assert filename, 'You must specify a filename'
        assert whitelistfilename, 'You must specify a whitelist of barcodes'
        assert label, 'You must specify a label'
        whitelist = _reads.Whitelist(whitelistfilename)
        if not UMIS and not self.extensions:
            # te_count.py:429-442 records nothing without UMIs and the run ends at :703
            raise ZeroDivisionError('division by zero')
        qual = self._qual()
        self.barcodes = {}
        self.load_genome()                                    # te_count.py:581 (done up front here)
        eng = self._engine()
        cm = _reads.ChromMap(self.genome.chrom_keys)
        log.info('Part 1: Collapsing UMI/CB combinations')
        more, done, next_log = True, 0, 10000000
        # One file, several ranks (shard.py): byte ranges decoded per GPU, survivors exchanged by cell, the job-wide steps
        # of Parts 1-3 all-reduced; rank r's records precede rank r + 1's, so the job-wide record order is the file's.
        rank, world = _shard.world_info()
        in_library = _shard.join_collectives(eng) if world > 1 else False
        if world > 1:
            sharded = None
            if UMIS and _device_decoder_wanted(eng):
                def open_and_bind():
                    dev = eng.bam_open(filename)
                    dev.bind(cm, whitelist)
                    return dev
                eng.sc_begin(qual, strand, len(whitelist))
                sharded = _shard.count_ranges(open_and_bind, 2, qual)
            if sharded is not None:
                done, more = sharded[1], False
            elif rank != 0:
                eng.sc_begin(qual, strand, len(whitelist))    # rank 0 reads the whole file; this rank only receives its cells
                more = False
        if more and UMIS and _device_decoder_wanted(eng):
            try:
                dev = eng.bam_open(filename)
                try:
                    dev.bind(cm, whitelist)
                    eng.sc_begin(qual, strand, len(whitelist))
                    done = dev.count(2, qual)
                    more = False
                    self._bam_info = dev.info()
                finally:
                    dev.close()
            except (_lib.BamUnsupported, OSError):
                more = True
            except _lib.TecError as e:
                if e.status != _lib.ERR_NOMEM:
                    raise
                eng.trim()
                more = True
            while done >= next_log:
                log.info('  Processed {:,} SE valid reads'.format(next_log))
                next_log += 10000000
        sam = batch = None
        if more:
            done, next_log = 0, 10000000
            sam = _open_alignment(filename, tags_optional=not UMIS)
            native = isinstance(sam, _fastbam.NativeBam)
            if native:
                sam.bind(cm, whitelist)
            batch = _reads.Batch(BATCH_RECORDS, sc=True, alloc=eng.pinned)
            eng.sc_begin(qual, strand, len(whitelist))
        while more:
            more = sam.fill_sc(batch, qual) if native else _reads.fill_sc(batch, sam, cm, whitelist, qual, umis=UMIS, umi_base=done)
            eng.sc_push(batch.n, batch.start, batch.end, batch.chrom, batch.mapq, batch.flag,
                        batch.cell, batch.umi)
            done += batch.n
            while done >= next_log:
                log.info('  Processed {:,} SE valid reads'.format(next_log))
                next_log += 10000000
        if sam is not None:
            sam.close()
        log.info(f'Part 2: Get the best {maxcells} barcodes and remove dupes')
        self._sc_device_matrix = True
        if world > 1:
            import torch
            from . import dist as _tdist
            _tdist.sc_exchange_by_cell(eng, torch.device('cuda', self.device))
        n_triples, n_hit = eng.sc_finalize(_bundle_keys, maxcells, _pad)
        if world > 1 and in_library:
            n_triples = eng.sc_allgather_triples()            # every rank holds the job's triples (on the device too)
        ensg, cell, count, hcell, hcount, st = eng.sc_fetch(n_triples, n_hit)
        if world > 1 and not in_library:
            ensg, cell, count = _tdist.sc_gather_triples(ensg, cell, count)
            self._sc_device_matrix = False                    # the device holds this rank's cells only: rows are written by the host
        idx = int(st[_lib.SS_UNITS]) + 1
        valid = int(st[_lib.SS_VALID])
        log.info(f'  Observed {int(st[_lib.SS_RAW_BARCODES]):,} raw barcodes')
        log.info(f'  Preserved {valid:,}/{idx:,} ({valid/idx*100:.1f}%) of the reads')
        log.info('Part 3: Mapping the remaining UMIs to features')
        if st[_lib.SS_CRASH_STRAND]:
            raise KeyError('strand')                          # te_count.py:661 on an index without strands
        assigned = int(st[_lib.SS_ASSIGNED])
        id_to_barcode = whitelist.id_to_barcode
        self.barcodes = {id_to_barcode[c]: h for c, h in zip(hcell.tolist(), hcount.tolist())}
        log.info('  In the total pipeling, processed {:,} SE reads'.format(idx))
        log.info('  {:,} invalid barcode reads'.format(int(st[_lib.SS_INVALID_BARCODE])))
        log.info('  {:,} UMI-CB combinations were seen multiple times and removed'.format(int(st[_lib.SS_ALREADY_SEEN])))
        log.info('  {:,} Read quality is too low (<{})'.format(int(st[_lib.SS_LOWQ]), self.quality_threshold))
        log.info('  {:,} Reads QC failed'.format(int(st[_lib.SS_QCFAIL])))
        log.info('  {:,} total valid reads'.format(valid))
        log.info('  Assigned {:,} ({:.1f}%) of total valid reads to features'.format(assigned, ((assigned / valid) * 100.0)))
        self.total_reads = idx
        self._sc_hit = (hcell, hcount)
        return ScResult(self.all_feature_names, id_to_barcode, ensg, cell, count)

    def sc_save_result(self, result, out_filename, maxcells=None, log=None):
        '''Save the cell x feature matrix and the barcode frequency file (te_count.py:709-754).'''
        assert out_filename, 'You must specify a filename'
        assert maxcells, 'You must specify maxcells'

        log.info('Densifying and saving "{0}"'.format(out_filename))
        log.info('Found {0:,} barcodes'.format(len(self.barcodes)))

        sel = None
        if isinstance(result, ScResult) and self._engine_obj is not None and getattr(self, '_sc_hit', None) is not None:
            # top-maxcells on the device: count descending, ties by ascending whitelist id
            sel = self._engine_obj.sc_select(maxcells, len(self._sc_hit[0]))
            barcodes_to_do = [result._id_to_barcode[c] for c in sel.tolist()]
        else:
            barcodes_to_do = [i[0] for i in sorted(self.barcodes.items(), key=itemgetter(1), reverse=True)][0:maxcells]
        if len(self.barcodes) > maxcells:
            log.info(f'Keeping the best {maxcells:,} barcodes')
        elif maxcells > len(self.barcodes):
            log.warning('Asked for {0:,} maxcells, but only {1:,} barcodes found'.format(maxcells, len(self.barcodes)))

        if '.tsv' not in out_filename:
            out_filename = f"{out_filename}.tsv"
        barcode_freq_filename = out_filename.replace('.tsv', '.barcode_freq.tsv')

        with open(barcode_freq_filename, 'w') as oh:
            for b in barcodes_to_do:
                oh.write('{0}\t{1}\n'.format(b, self.barcodes[b]))
        log.info('Saving barcode read frequency file to {0}'.format(barcode_freq_filename))

        with open(out_filename, 'w') as oh:
            oh.write('{}\t{}\n'.format('name', '\t'.join(result.keys())))
            if sel is not None and hasattr(self._engine_obj, 'sc_matrix_text') and getattr(self, '_sc_device_matrix', True):
                # the rows are formatted on the device (libtecount tec_sc_matrix_text) and streamed out
                oh.flush()
                n_bytes = self._engine_obj.sc_matrix_text(sel, barcodes_to_do)
                with open(out_filename, 'ab') as ob:
                    self._engine_obj.sc_matrix_write(ob, n_bytes)
            elif isinstance(result, ScResult):
                _write_dense_rows(oh, result, barcodes_to_do)
            else:
                for barcode in barcodes_to_do:
                    counts = [str(result[f].get(barcode, 0)) for f in result]
                    oh.write('{}\n'.format('\t'.join([barcode] + counts)))

    def sc_save_mtx(self, result, out_dir, maxcells, log=None, threads=None):
        '''Extension (not in the reference): the matrix of sc_save_result -- the same cells, in the same order -- as a
        10x-style Matrix Market directory (matrix.mtx.gz, features.tsv.gz, barcodes.tsv.gz; te_counter_b200/mtx.py)
        that scanpy.read_10x_mtx and Seurat's Read10X read.  `threads`: gzip threads (default: the usable cores).'''
        if not isinstance(result, ScResult):
            raise TypeError('sc_save_mtx takes the ScResult of sc_parse_bamse, not %s' % type(result).__name__)
        assert out_dir, 'You must specify a directory'
        assert maxcells, 'You must specify maxcells'
        threads = threads or _mtx.default_threads()

        log.info('Saving the sparse matrix to "{0}"'.format(out_dir))
        log.info('Found {0:,} barcodes'.format(len(self.barcodes)))
        eng = self._engine_obj
        sel = eng.sc_select(maxcells, len(self._sc_hit[0]))   # sc_save_result's rows: count descending, ties by ascending id
        barcodes_to_do = [result._id_to_barcode[c] for c in sel.tolist()]
        if len(self.barcodes) > maxcells:
            log.info(f'Keeping the best {maxcells:,} barcodes')
        elif maxcells > len(self.barcodes):
            log.warning('Asked for {0:,} maxcells, but only {1:,} barcodes found'.format(maxcells, len(self.barcodes)))

        os.makedirs(out_dir, exist_ok=True)
        path = os.path.join(out_dir, 'matrix.mtx.gz')
        if hasattr(eng, 'sc_matrix_mtx') and getattr(self, '_sc_device_matrix', True):
            # the text is formatted on the device (libtecount tec_sc_matrix_mtx) and streamed into the compressors
            _, n_bytes = eng.sc_matrix_mtx(sel)
            _mtx.write_gzip(path, lambda fh: eng.sc_matrix_write(fh, n_bytes, chunk=_mtx.PIECE), threads)
        else:
            text = _mtx.mtx_text(len(result), result.ensg, result.cell, result.count, sel)
            _mtx.write_gzip(path, lambda fh: fh.write(text), threads)
        _mtx.write_gzip(os.path.join(out_dir, 'features.tsv.gz'), lambda fh: fh.write(_mtx.features_text(result.keys())), threads)
        _mtx.write_gzip(os.path.join(out_dir, 'barcodes.tsv.gz'), lambda fh: fh.write(_mtx.barcodes_text(barcodes_to_do)), threads)
        log.info('Saved {0}'.format(path))


def _write_dense_rows(oh, result, barcodes_to_do):
    """Dense integer rows from the sparse triples: zeros are emitted as slices of one long
    '\\t0\\t0...' string, so the cost is O(non-zeros) per row, not O(features)."""
    n_ensg = len(result)
    bc_to_id = {b: i for i, b in enumerate(result._id_to_barcode)}
    want = np.array([bc_to_id[b] for b in barcodes_to_do], dtype=np.int64)
    rank = np.full(len(result._id_to_barcode), -1, dtype=np.int64)
    rank[want] = np.arange(len(want))
    r = rank[result.cell]
    keep = r >= 0
    r, e, v = r[keep], result.ensg[keep].astype(np.int64), result.count[keep]
    order = np.lexsort((e, r))
    r, e, v = r[order], e[order], v[order]
    ptr = np.searchsorted(r, np.arange(len(want) + 1))
    zeros = '\t0' * n_ensg
    for i, barcode in enumerate(barcodes_to_do):
        a, b = ptr[i], ptr[i + 1]
        parts = [barcode]
        prev = -1
        for col, val in zip(e[a:b].tolist(), v[a:b].tolist()):
            parts.append(zeros[:2 * (col - prev - 1)])
            parts.append('\t%d' % val)
            prev = col
        parts.append(zeros[:2 * (n_ensg - prev - 1)])
        parts.append('\n')
        oh.write(''.join(parts))
