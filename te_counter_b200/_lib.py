"""
ctypes binding of libtecount.so (include/tecount.h).  There is no CPU fallback: importing the
engine without the built CUDA library, or creating it without a usable GPU, raises.
"""
import ctypes
import os
import weakref

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TEC_LIB") or os.path.join(_HERE, "libtecount.so")

BULK_NSTATS = 8
BS_UNITS, BS_ASSIGNED, BS_LOWQ, BS_BADCHROM, BS_QCFAIL, BS_CRASH_ENHANCER, BS_CRASH_NAME, BS_NO_MATE = range(8)
SC_NSTATS = 16
(SS_UNITS, SS_INVALID_BARCODE, SS_ALREADY_SEEN, SS_LOWQ, SS_QCFAIL, SS_VALID, SS_ASSIGNED,
 SS_RAW_BARCODES, SS_BUNDLES, SS_CRASH_STRAND, SS_SURVIVORS, SS_SEGMENTS) = range(12)

_c_i32p = ctypes.POINTER(ctypes.c_int32)
_c_i64p = ctypes.POINTER(ctypes.c_int64)
_c_u8p = ctypes.POINTER(ctypes.c_uint8)
_c_u16p = ctypes.POINTER(ctypes.c_uint16)
_c_u32p = ctypes.POINTER(ctypes.c_uint32)
_c_u64p = ctypes.POINTER(ctypes.c_uint64)
_vp = ctypes.c_void_p

# name -> (restype, argtypes); tests check that every symbol of include/tecount.h is listed and exported
SIGNATURES = {
    "tec_abi_version": (ctypes.c_int, []),
    "tec_strerror": (ctypes.c_char_p, [ctypes.c_int]),
    "tec_create": (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(_vp)]),
    "tec_destroy": (None, [_vp]),
    "tec_last_error": (ctypes.c_char_p, [_vp]),
    "tec_sync": (ctypes.c_int, [_vp]),
    "tec_host_alloc": (ctypes.c_int, [_vp, ctypes.c_uint64, ctypes.POINTER(_vp)]),
    "tec_host_free": (ctypes.c_int, [_vp, _vp]),
    "tec_stream": (_vp, [_vp]),
    "tec_last_kernel_ms": (ctypes.c_float, [_vp]),
    "tec_launch_count": (ctypes.c_int64, [_vp]),
    "tec_trim": (ctypes.c_int, [_vp]),
    "tec_set_option": (ctypes.c_int, [_vp, ctypes.c_char_p, ctypes.c_int64]),
    "tec_get_info": (ctypes.c_int64, [_vp, ctypes.c_char_p]),
    "tec_index_note": (ctypes.c_char_p, [_vp]),
    "tec_index_upload": (ctypes.c_int, [_vp, ctypes.c_int32, _c_i64p, _c_i32p, _c_i32p, _c_i32p, _c_u8p,
                                        _c_u8p, ctypes.c_int32, ctypes.c_int32]),
    "tec_bulk_begin": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int]),
    "tec_bulk_push": (ctypes.c_int, [_vp, ctypes.c_int64, _vp, _vp, _vp, _vp, _vp]),
    "tec_bulk_push_dev": (ctypes.c_int, [_vp, ctypes.c_int64, _vp, _vp, _vp, _vp, _vp]),
    "tec_bulk_push_named": (ctypes.c_int, [_vp, ctypes.c_int64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, ctypes.c_char_p]),
    "tec_bulk_finish": (ctypes.c_int, [_vp, _c_i64p, _c_i64p]),
    "tec_bulk_counts_dev": (_vp, [_vp]),
    "tec_bulk_loci": (ctypes.c_int, [_vp, _c_i64p]),
    "tec_sc_begin": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int64]),
    "tec_sc_push": (ctypes.c_int, [_vp, ctypes.c_int64, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "tec_sc_push_dev": (ctypes.c_int, [_vp, ctypes.c_int64, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "tec_sc_finalize": (ctypes.c_int, [_vp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, _c_i64p, _c_i64p]),
    "tec_sc_fetch": (ctypes.c_int, [_vp, _c_i32p, _c_u32p, _c_i64p, _c_u32p, _c_i64p, _c_i64p]),
    "tec_sc_select": (ctypes.c_int, [_vp, ctypes.c_int64, _c_u32p, _c_i64p]),
    "tec_bam_open": (ctypes.c_int, [_vp, ctypes.c_char_p, ctypes.POINTER(_vp)]),
    "tec_bam_close": (None, [_vp]),
    "tec_bam_n_references": (ctypes.c_int, [_vp]),
    "tec_bam_reference_name": (ctypes.c_char_p, [_vp, ctypes.c_int]),
    "tec_bam_set_chrom_map": (ctypes.c_int, [_vp, _vp, _vp, ctypes.c_int32, ctypes.c_int32]),
    "tec_bam_set_whitelist": (ctypes.c_int, [_vp, ctypes.c_char_p, _vp, ctypes.c_int32]),
    "tec_bam_count": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, _c_i64p]),
    "tec_bam_count_range": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int64, ctypes.c_int64, _c_i64p]),
    "tec_bam_range_record": (ctypes.c_int, [_vp, ctypes.c_int, _vp, ctypes.c_int64, _c_i64p]),
    "tec_bam_pair_columns": (ctypes.c_int, [_vp, _vp, ctypes.c_int64, _vp, ctypes.c_int64, ctypes.c_int, _vp, _vp, _vp, _vp, _vp]),
    "tec_bulk_keep_bank": (ctypes.c_int, [_vp, ctypes.c_int]),
    "tec_bulk_name_partition_dev": (ctypes.c_int, [_vp, ctypes.c_int, _c_i64p, ctypes.POINTER(_vp)]),
    "tec_bulk_name_import_dev": (ctypes.c_int, [_vp, ctypes.c_int64, _vp]),
    "tec_bulk_name_exchange": (ctypes.c_int, [_vp, _c_i64p]),
    "tec_bam_info": (ctypes.c_int64, [_vp, ctypes.c_int]),
    "tec_sc_matrix_text": (ctypes.c_int, [_vp, ctypes.c_int64, _c_u32p, ctypes.c_char_p, _c_i64p, _c_i64p]),
    "tec_sc_matrix_read": (ctypes.c_int, [_vp, ctypes.c_int64, ctypes.c_int64, _vp]),
    "tec_sc_matrix_mtx": (ctypes.c_int, [_vp, ctypes.c_int64, _c_u32p, _c_i64p, _c_i64p]),
    "tec_sc_set_collective": (ctypes.c_int, [_vp, _vp, _vp, ctypes.c_int, ctypes.c_int]),
    "tec_sc_survivors": (ctypes.c_int, [_vp, _c_i64p]),
    "tec_sc_partition_dev": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int64, _c_i64p, ctypes.POINTER(_vp)]),
    "tec_sc_import_packed_dev": (ctypes.c_int, [_vp, ctypes.c_int64, _vp]),
    "tec_comm_unique_id": (ctypes.c_int, [_vp, _vp, ctypes.c_int32]),
    "tec_comm_init": (ctypes.c_int, [_vp, _vp, ctypes.c_int32, ctypes.c_int32]),
    "tec_comm_destroy": (ctypes.c_int, [_vp]),
    "tec_comm_info": (ctypes.c_int, [_vp, ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int32)]),
    "tec_bulk_allreduce": (ctypes.c_int, [_vp]),
    "tec_sc_exchange": (ctypes.c_int, [_vp, _c_i64p]),
    "tec_sc_allgather_triples": (ctypes.c_int, [_vp, _c_i64p]),
}

COMM_ID_BYTES = 128

ALLREDUCE_FN = ctypes.CFUNCTYPE(ctypes.c_int, _vp, _vp, ctypes.c_int64, ctypes.c_int, ctypes.c_int)

_lib = None


def _point_at_bundled_nccl():
    """TEC_NCCL_LIB = the libnccl.so.2 PyTorch ships (nvidia/nccl/lib), unless the caller set one: the library binds
    NCCL at run time, and a process that imports torch afterwards must find the copy torch was linked against."""
    if os.environ.get("TEC_NCCL_LIB"):
        return
    try:
        import importlib.util
        spec = importlib.util.find_spec("nvidia")
        for base in (spec.submodule_search_locations if spec else ()):
            cand = os.path.join(base, "nccl", "lib", "libnccl.so.2")
            if os.path.exists(cand):
                os.environ["TEC_NCCL_LIB"] = cand
                return
    except (ImportError, ValueError):
        pass


def load_library():
    """dlopen libtecount.so and attach the prototypes.  Raises ImportError when it is not built."""
    global _lib
    if _lib is None:
        _point_at_bundled_nccl()
        if not os.path.exists(LIB_PATH):
            raise ImportError("libtecount.so is not built (%s); run `python -m te_counter_b200.build` "
                              "-- there is no CPU fallback" % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


class TecError(RuntimeError):
    def __init__(self, status, text):
        RuntimeError.__init__(self, "libtecount: %s (status %d)" % (text, status))
        self.status = status


ERR_NOMEM = -4
ERR_IO, ERR_FORMAT, ERR_UNSUPPORTED = -7, -8, -9
ERR_BAM_NO_BARCODE_TAG, ERR_BAM_NO_UMI_TAG, ERR_BAM_UMI, ERR_BAM_END_NONE, ERR_BAM_CHROM_NAME, ERR_BAM_REF_NONE = -10, -11, -12, -13, -14, -15


class BamUnsupported(Exception):
    """The device decoder refuses this file (not BGZF, or a record layout it cannot split
    block-parallel): decode it on the host (fastbam.NativeBam) instead."""


class DeviceBam:
    """BAM file decoded on the device straight into the running count (include/tecount.h tec_bam_*).
    Same hand-over of the chromosome map / whitelist and same exceptions as fastbam.NativeBam."""

    def __init__(self, engine, filename):
        self._eng = engine
        self._lib = engine._lib
        self._h = _vp()
        self.filename = filename
        rc = self._lib.tec_bam_open(engine._h, os.fsencode(filename), ctypes.byref(self._h))
        if rc == ERR_UNSUPPORTED:
            raise BamUnsupported(filename)
        if rc == ERR_IO:
            raise OSError("cannot open %s" % filename)
        engine._check(rc)
        engine._bams.append(weakref.ref(self))
        self.references = [self._lib.tec_bam_reference_name(self._h, i).decode("ascii")
                           for i in range(self._lib.tec_bam_n_references(self._h))]

    def bind(self, chrom_map, whitelist=None):
        bulk = np.array([chrom_map.bulk_id(n) for n in self.references], dtype=np.uint16)
        sc = np.empty(len(self.references), dtype=np.uint16)
        for i, n in enumerate(self.references):
            try:
                sc[i] = chrom_map.sc_id(n)
            except ValueError:
                sc[i] = 0xFFFD                          # raised when a counted record gets there
        self._eng._check(self._lib.tec_bam_set_chrom_map(self._h, bulk.ctypes.data, sc.ctypes.data, len(self.references),
                                                         chrom_map.n_index))
        if whitelist is not None:
            enc = [b.encode("utf-8") for b in whitelist.id_to_barcode]
            off = np.zeros(len(enc) + 1, dtype=np.int64)
            if enc:
                np.cumsum([len(b) for b in enc], out=off[1:])
            self._eng._check(self._lib.tec_bam_set_whitelist(self._h, b"".join(enc), off.ctypes.data, len(enc)))

    def count(self, mode, qual):
        """mode 0 single end, 1 paired end, 2 single cell, 3 paired end by read name (after bulk_begin(..., pairing='name'));
        returns the number of records decoded."""
        n = ctypes.c_int64(0)
        rc = self._lib.tec_bam_count(self._h, int(mode), int(qual), ctypes.byref(n))
        if rc == 0:
            return n.value
        self._raise(rc, mode)

    def count_range(self, mode, qual, byte_lo, byte_hi):
        """The records that start in the BGZF blocks of [byte_lo, byte_hi) (include/tecount.h: tec_bam_count_range).
        Returns {n, start, exit, size}: start / exit are (block file offset, offset in the inflated block).  Paired end
        (mode 1) adds first / last: the raw bytes of the range's first and last record (b"" without records); the
        engine then waits for Engine.bulk_keep_bank.  Paired end by read name (mode 4, after bulk_begin(..., pairing='name'))
        holds the range's rows unpaired; the engine then waits for Engine.bulk_name_partition_dev (or bulk_name_exchange)."""
        out = (ctypes.c_int64 * 6)()
        rc = self._lib.tec_bam_count_range(self._h, int(mode), int(qual), int(byte_lo), int(byte_hi), out)
        if rc != 0:
            self._raise(rc, mode)
        info = {"n": out[0], "start": (out[1], out[2]), "exit": (out[3], out[4]), "size": out[5]}
        if int(mode) == 1:
            info["first"], info["last"] = self._range_record(0), self._range_record(1)
        return info

    def _range_record(self, which):
        n = ctypes.c_int64(0)
        self._eng._check(self._lib.tec_bam_range_record(self._h, which, None, 0, ctypes.byref(n)))
        buf = ctypes.create_string_buffer(max(1, n.value))
        self._eng._check(self._lib.tec_bam_range_record(self._h, which, buf, n.value, ctypes.byref(n)))
        return buf.raw[:n.value]

    def pair_columns(self, rec1, rec2, qual):
        """read1 = rec1, read2 = rec2 (raw records of this file, e.g. count_range's last / first) parsed on the host with
        this file's chromosome map: {start, end, chrom, mapq, flag}, two rows each, the layout bulk_push takes."""
        cols = {"start": np.zeros(2, np.int32), "end": np.zeros(2, np.int32), "chrom": np.zeros(2, np.uint16),
                "mapq": np.zeros(2, np.uint8), "flag": np.zeros(2, np.uint8)}
        rc = self._lib.tec_bam_pair_columns(self._h, rec1, len(rec1), rec2, len(rec2), int(qual),
                                            *[cols[k].ctypes.data for k in ("start", "end", "chrom", "mapq", "flag")])
        if rc != 0:
            self._raise(rc, 1)
        return cols

    def _raise(self, rc, mode):
        msg = (self._lib.tec_last_error(self._eng._h) or b"").decode()
        if rc == ERR_UNSUPPORTED:
            raise BamUnsupported("%s: %s" % (self.filename, msg))
        if rc == ERR_BAM_NO_BARCODE_TAG:
            raise AssertionError('CB or CR tag not found!')                     # te_count.py:409
        if rc == ERR_BAM_NO_UMI_TAG:
            raise AssertionError('UB or UR tag not found!')                     # te_count.py:426
        if rc == ERR_BAM_END_NONE:
            raise TypeError("unsupported operand type(s) for +: 'NoneType' and 'int'" if mode != 2
                            else "reference_end is None for a counted read (%s)" % msg)
        if rc == ERR_BAM_REF_NONE:
            raise AttributeError("'NoneType' object has no attribute 'replace'")    # te_count.py:431
        if rc in (ERR_BAM_UMI, ERR_BAM_CHROM_NAME):
            raise ValueError("%s: %s (%s)" % (self.filename, "UMI the code cannot hold" if rc == ERR_BAM_UMI
                                              else "chromosome name contains ':' (unsupported in --sc)", msg))
        if rc == ERR_FORMAT:
            if "truncated" in msg:
                raise EOFError("%s: %s" % (self.filename, msg))
            raise ValueError("%s: %s" % (self.filename, msg))
        self._eng._check(rc)

    def info(self):
        names = ("host_inflated_blocks", "us_load", "us_inflate", "us_chain", "us_parse")
        return {k: int(self._lib.tec_bam_info(self._h, i)) for i, k in enumerate(names)}

    def close(self):
        if self._h:
            self._lib.tec_bam_close(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _ptr(a, dtype):
    if a is None:
        return None
    if not isinstance(a, np.ndarray) or a.dtype != dtype or not a.flags.c_contiguous:
        raise TypeError("expected a C-contiguous numpy array of %s" % np.dtype(dtype).name)
    return a.ctypes.data


class Engine:
    """One CUDA context of libtecount on one GPU."""

    def __init__(self, device=0):
        self._lib = load_library()
        h = _vp()
        rc = self._lib.tec_create(int(device), ctypes.byref(h))
        if rc != 0:
            raise TecError(rc, "tec_create(device=%d) failed: %s -- a CUDA GPU is required, there is no "
                               "CPU fallback" % (device, self._lib.tec_strerror(rc).decode()))
        self._h = h
        self.device = device
        self.n_ensg = 0
        self.n_features = 0
        self._pinned = []
        self._bams = []

    def close(self):
        if getattr(self, "_h", None):
            for ref in getattr(self, "_bams", []):          # device decoders hold buffers of this context
                b = ref()
                if b is not None:
                    b.close()
            self._bams = []
            for p in self._pinned:
                self._lib.tec_host_free(self._h, p)
            self._pinned = []
            self._lib.tec_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise TecError(rc, (self._lib.tec_last_error(self._h) or b"").decode() or
                           self._lib.tec_strerror(rc).decode())

    # -- memory / timing
    def pinned(self, n, dtype):
        """numpy array of n elements backed by cudaHostAlloc memory (lives as long as the engine)."""
        dt = np.dtype(dtype)
        p = _vp()
        self._check(self._lib.tec_host_alloc(self._h, max(1, n) * dt.itemsize, ctypes.byref(p)))
        self._pinned.append(p)
        buf = (ctypes.c_char * (max(1, n) * dt.itemsize)).from_address(p.value)
        return np.frombuffer(buf, dtype=dt, count=n)

    def sync(self):
        self._check(self._lib.tec_sync(self._h))

    @property
    def stream(self):
        return self._lib.tec_stream(self._h)

    def last_kernel_ms(self):
        return float(self._lib.tec_last_kernel_ms(self._h))

    def launch_count(self):
        return int(self._lib.tec_launch_count(self._h))

    def trim(self):
        """free the device scratch cached by the single-cell finalize"""
        self._check(self._lib.tec_trim(self._h))

    def set_option(self, key, value):
        self._check(self._lib.tec_set_option(self._h, key.encode(), int(value)))

    def get_info(self, key):
        return int(self._lib.tec_get_info(self._h, key.encode()))

    def index_note(self):
        """Why the uploaded index has no bulk cell table ('' when it has one): see tec_index_note."""
        return (self._lib.tec_index_note(self._h) or b"").decode()

    # -- index
    def upload_index(self, idx):
        """idx: te_counter_b200.index.GlbIndex"""
        s = idx.sorted_layout()
        self.upload_index_arrays(idx.n_chrom, s["chrom_off"], s["L"], s["R"], s["ensg_id"], s["type_code"],
                                 s["strand_code"], idx.n_ensg, idx.bucket_size)

    def upload_index_arrays(self, n_chrom, chrom_off, L, R, ensg_id, type_code, strand_code, n_ensg, bucket_size):
        f = self._lib.tec_index_upload
        self._check(f(self._h, int(n_chrom),
                      ctypes.cast(_ptr(chrom_off, np.int64), _c_i64p), ctypes.cast(_ptr(L, np.int32), _c_i32p),
                      ctypes.cast(_ptr(R, np.int32), _c_i32p), ctypes.cast(_ptr(ensg_id, np.int32), _c_i32p),
                      ctypes.cast(_ptr(type_code, np.uint8), _c_u8p), ctypes.cast(_ptr(strand_code, np.uint8), _c_u8p),
                      int(n_ensg), int(bucket_size)))
        self.n_ensg = int(n_ensg)
        self.n_features = int(chrom_off[int(n_chrom)])

    # -- bulk
    def bulk_begin(self, paired, qual, pairing="index"):
        """pairing='name' (paired end only): mates are paired by read name (include/tecount.h, tec_bulk_begin(ctx, 2, qual));
        records then go in through bulk_push_named or DeviceBam.count(3, qual)."""
        if pairing not in ("index", "name"):
            raise ValueError("pairing must be 'index' or 'name'")
        mode = (2 if pairing == "name" else 1) if paired else 0
        self._check(self._lib.tec_bulk_begin(self._h, mode, int(qual)))

    def bulk_push_named(self, n, start, end, chrom, mapq, flag, samflag, name_off, names):
        """Host records for pairing by read name: the usual columns plus samflag (uint16 SAM flags), name_off (int64[n + 1])
        and names (the QNAME bytes, concatenated)."""
        if len(name_off) < int(n) + 1:
            raise ValueError("name_off needs n + 1 entries")
        self._check(self._lib.tec_bulk_push_named(self._h, int(n), _ptr(start, np.int32), _ptr(end, np.int32),
                                                  _ptr(chrom, np.uint16), _ptr(mapq, np.uint8), _ptr(flag, np.uint8),
                                                  _ptr(samflag, np.uint16), _ptr(name_off, np.int64), bytes(names)))

    def bulk_push(self, n, start, end, chrom, mapq, flag):
        self._check(self._lib.tec_bulk_push(self._h, int(n), _ptr(start, np.int32), _ptr(end, np.int32),
                                            _ptr(chrom, np.uint16), _ptr(mapq, np.uint8), _ptr(flag, np.uint8)))

    def bulk_push_dev(self, n, start, end, chrom, mapq, flag):
        """device pointers (ints), asynchronous"""
        self._check(self._lib.tec_bulk_push_dev(self._h, int(n), start, end, chrom, mapq, flag))

    def bulk_finish(self):
        counts = np.zeros(self.n_ensg, dtype=np.int64)
        stats = np.zeros(BULK_NSTATS, dtype=np.int64)
        self._check(self._lib.tec_bulk_finish(self._h, ctypes.cast(counts.ctypes.data, _c_i64p),
                                              ctypes.cast(stats.ctypes.data, _c_i64p)))
        return counts, stats

    def bulk_loci(self):
        """Counts per index row of a run begun with set_option('bulk_loci', 1) (include/tecount.h tec_bulk_loci):
        int64[n_features] in the row order of the upload (GlbIndex.sorted_layout())."""
        loci = np.zeros(self.n_features, dtype=np.int64)
        self._check(self._lib.tec_bulk_loci(self._h, ctypes.cast(loci.ctypes.data, _c_i64p)))
        return loci

    def bulk_keep_bank(self, bank):
        """after a paired-end count_range: keep counter bank `bank` (the parity of the range's global record offset)"""
        self._check(self._lib.tec_bulk_keep_bank(self._h, int(bank)))

    def bulk_name_partition_dev(self, world):
        """after count_range(4, ...): (counts per owner rank, device pointer of the packed 32-byte records)"""
        counts = (ctypes.c_int64 * world)()
        p = _vp()
        self._check(self._lib.tec_bulk_name_partition_dev(self._h, int(world), counts, ctypes.byref(p)))
        return list(counts), (p.value or 0)

    def bulk_name_import_dev(self, n, records):
        """the n records this rank owns (device pointer, laid out by source rank), paired in one pass"""
        self._check(self._lib.tec_bulk_name_import_dev(self._h, int(n), records))

    def bulk_counts_dev(self):
        return self._lib.tec_bulk_counts_dev(self._h)

    # -- single cell
    def sc_begin(self, qual, strand, n_whitelist):
        self._check(self._lib.tec_sc_begin(self._h, int(qual), 1 if strand else 0, int(n_whitelist)))

    def sc_push(self, n, start, end, chrom, mapq, flag, cell, umi):
        self._check(self._lib.tec_sc_push(self._h, int(n), _ptr(start, np.int32), _ptr(end, np.int32),
                                          _ptr(chrom, np.uint16), _ptr(mapq, np.uint8), _ptr(flag, np.uint8),
                                          _ptr(cell, np.uint32), _ptr(umi, np.uint64)))

    def sc_push_dev(self, n, start, end, chrom, mapq, flag, cell, umi):
        self._check(self._lib.tec_sc_push_dev(self._h, int(n), start, end, chrom, mapq, flag, cell, umi))

    def sc_finalize(self, bundle_keys, maxcells, pad):
        nt, nh = ctypes.c_int64(0), ctypes.c_int64(0)
        self._check(self._lib.tec_sc_finalize(self._h, int(bundle_keys), int(maxcells), int(pad),
                                              ctypes.byref(nt), ctypes.byref(nh)))
        return nt.value, nh.value

    def _result_buf(self, name, n, dtype):
        """grow-only pinned result buffer (view valid until the next fetch that uses it)"""
        buf = self._res.get(name)
        if buf is None or len(buf) < n or buf.dtype != np.dtype(dtype):
            buf = self.pinned(max(n + n // 4, 1024), dtype)
            self._res[name] = buf
        return buf[:n]

    def sc_fetch(self, n_triples, n_hit_cells, pinned=False):
        """(ensg, cell, count, hit_cell, hit_count, stats).  pinned=True: the arrays are views of reusable
        page-locked buffers (fast device-to-host copies) that the next pinned fetch overwrites."""
        if pinned:
            if not hasattr(self, "_res"):
                self._res = {}
            ensg = self._result_buf("ensg", n_triples, np.int32)
            cell = self._result_buf("cell", n_triples, np.uint32)
            count = self._result_buf("count", n_triples, np.int64)
            hcell = self._result_buf("hcell", n_hit_cells, np.uint32)
            hcount = self._result_buf("hcount", n_hit_cells, np.int64)
        else:
            ensg = np.zeros(n_triples, dtype=np.int32)
            cell = np.zeros(n_triples, dtype=np.uint32)
            count = np.zeros(n_triples, dtype=np.int64)
            hcell = np.zeros(n_hit_cells, dtype=np.uint32)
            hcount = np.zeros(n_hit_cells, dtype=np.int64)
        stats = np.zeros(SC_NSTATS, dtype=np.int64)
        self._check(self._lib.tec_sc_fetch(self._h, ctypes.cast(ensg.ctypes.data, _c_i32p),
                                           ctypes.cast(cell.ctypes.data, _c_u32p),
                                           ctypes.cast(count.ctypes.data, _c_i64p),
                                           ctypes.cast(hcell.ctypes.data, _c_u32p),
                                           ctypes.cast(hcount.ctypes.data, _c_i64p),
                                           ctypes.cast(stats.ctypes.data, _c_i64p)))
        return ensg, cell, count, hcell, hcount, stats

    def sc_set_collective(self, fn, rank, world):
        """fn(dev_ptr, count, dtype, op) -> None: in-place all-reduce over the ranks (dist.py)."""
        if fn is None:
            self._coll = None
            self._check(self._lib.tec_sc_set_collective(self._h, None, None, 0, 1))
            return

        def _cb(_user, ptr, count, dtype, op):
            try:
                fn(ptr, count, dtype, op)
                return 0
            except Exception:          # never let an exception cross the C boundary
                import traceback
                traceback.print_exc()
                return -1

        self._coll = ALLREDUCE_FN(_cb)                    # keep the trampoline alive
        self._check(self._lib.tec_sc_set_collective(self._h, ctypes.cast(self._coll, _vp), None, int(rank), int(world)))

    def sc_survivors(self):
        """number of survivors held after the pushes"""
        n = ctypes.c_int64(0)
        self._check(self._lib.tec_sc_survivors(self._h, ctypes.byref(n)))
        return n.value

    def sc_partition_dev(self, world, gidx_base):
        """(counts per owner rank, device pointer of the packed 32-byte records)"""
        counts = (ctypes.c_int64 * world)()
        p = _vp()
        self._check(self._lib.tec_sc_partition_dev(self._h, int(world), int(gidx_base), counts, ctypes.byref(p)))
        return list(counts), (p.value or 0)

    def sc_import_packed_dev(self, n, records):
        self._check(self._lib.tec_sc_import_packed_dev(self._h, int(n), records))

    # ---- collectives issued by the library (NCCL; include/tecount.h)
    def comm_unique_id(self):
        """bytes of a fresh communicator id (rank 0; carry them to the other ranks, then comm_init everywhere)"""
        buf = ctypes.create_string_buffer(COMM_ID_BYTES)
        self._check(self._lib.tec_comm_unique_id(self._h, buf, COMM_ID_BYTES))
        return buf.raw

    def comm_init(self, comm_id, rank, world):
        if len(comm_id) != COMM_ID_BYTES:
            raise ValueError("communicator id must be %d bytes" % COMM_ID_BYTES)
        self._check(self._lib.tec_comm_init(self._h, ctypes.c_char_p(bytes(comm_id)), int(rank), int(world)))

    def comm_destroy(self):
        self._check(self._lib.tec_comm_destroy(self._h))

    def comm_world(self):
        r, w = ctypes.c_int32(0), ctypes.c_int32(1)
        self._check(self._lib.tec_comm_info(self._h, ctypes.byref(r), ctypes.byref(w)))
        return r.value, w.value

    def bulk_allreduce(self):
        """sum of the ranks' counter blocks in place (behind the pushes, on the library's stream)"""
        self._check(self._lib.tec_bulk_allreduce(self._h))

    def bulk_name_exchange(self):
        """after count_range(4, ...) on every rank: the rows exchanged by name owner and paired; returns the number of
        records this rank received"""
        n = ctypes.c_int64(0)
        self._check(self._lib.tec_bulk_name_exchange(self._h, ctypes.byref(n)))
        return n.value

    def sc_exchange(self):
        """all-to-all of the survivors by owner rank; returns the number of records this rank now owns"""
        n = ctypes.c_int64(0)
        self._check(self._lib.tec_sc_exchange(self._h, ctypes.byref(n)))
        return n.value

    def sc_allgather_triples(self):
        """after sc_finalize: the job's triples on every rank; returns their number (pass it to sc_fetch)"""
        n = ctypes.c_int64(0)
        self._check(self._lib.tec_sc_allgather_triples(self._h, ctypes.byref(n)))
        return n.value

    def sc_select(self, maxcells, n_hit_cells):
        out = np.zeros(max(1, min(int(maxcells), int(n_hit_cells))), dtype=np.uint32)
        n = ctypes.c_int64(0)
        self._check(self._lib.tec_sc_select(self._h, int(maxcells), ctypes.cast(out.ctypes.data, _c_u32p),
                                            ctypes.byref(n)))
        return out[:n.value]

    def bam_open(self, filename):
        return DeviceBam(self, filename)

    def sc_matrix_text(self, cells, barcodes):
        """Builds sc_save_result's dense rows (te_count.py:744-754) as text on the device for the
        given whitelist ids / barcode strings; returns the number of bytes."""
        cells = np.ascontiguousarray(cells, dtype=np.uint32)
        enc = [b.encode("utf-8") for b in barcodes]
        assert len(enc) == len(cells)
        off = np.zeros(len(enc) + 1, dtype=np.int64)
        if enc:
            np.cumsum([len(b) for b in enc], out=off[1:])
        n = ctypes.c_int64(0)
        self._check(self._lib.tec_sc_matrix_text(self._h, len(cells), ctypes.cast(cells.ctypes.data, _c_u32p), b"".join(enc),
                                                 ctypes.cast(off.ctypes.data, _c_i64p), ctypes.byref(n)))
        return n.value

    def sc_matrix_mtx(self, cells):
        """Builds the matrix as Matrix Market text on the device (include/tecount.h tec_sc_matrix_mtx): one row per
        feature, one column per given whitelist id, in that order.  Returns (non-zeros, bytes); stream it with
        sc_matrix_write."""
        cells = np.ascontiguousarray(cells, dtype=np.uint32)
        nnz, n = ctypes.c_int64(0), ctypes.c_int64(0)
        self._check(self._lib.tec_sc_matrix_mtx(self._h, len(cells), ctypes.cast(cells.ctypes.data, _c_u32p),
                                                ctypes.byref(nnz), ctypes.byref(n)))
        return nnz.value, n.value

    def sc_matrix_write(self, fh, n_bytes, chunk=1 << 26):
        """Streams the text built by sc_matrix_text or sc_matrix_mtx into the binary file object `fh`."""
        if getattr(self, "_text_buf", None) is None or len(self._text_buf) < min(chunk, max(1, n_bytes)):
            self._text_buf = self.pinned(min(chunk, max(1, n_bytes)), np.uint8)
        buf = self._text_buf
        done = 0
        while done < n_bytes:
            k = min(len(buf), n_bytes - done)
            self._check(self._lib.tec_sc_matrix_read(self._h, done, k, buf.ctypes.data))
            fh.write(memoryview(buf)[:k])
            done += k
