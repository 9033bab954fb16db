"""
Host-side repacking of aligned reads into the structure-of-arrays batches the CUDA library takes
(SURVEY.md 8d record layout: i32 start, i32 end, u16 chrom, u8 mapq, u8 flag bits; single cell adds
u32 cell id and u64 order-preserving UMI code).

Everything that is string handling in the reference's read loop lives here, so the kernels see
integers only:
  * chromosome key     reference_name.replace('chr', '')              (te_count.py:96, :212, :431)
  * 'in the index?'    key in genome.buckets                           (te_count.py:100, :216, :614)
  * sc silent skip     '_' in key or 'alt' in key                      (te_count.py:432)
  * whitelist ids      position in sorted(set(lines))                  (te_count.py:330-339)
  * barcode / UMI tag  CB else CR, UB else UR, AssertionError if none  (te_count.py:403-427)
  * PE name check      '_'.join(name.split('/')[0:-1]) of both mates   (te_count.py:92)
"""
import numpy as np

F_UNMAPPED, F_DUP, F_QCFAIL, F_REVERSE, F_NAME_MISMATCH = 1, 2, 4, 8, 16
CHROM_SC_SKIP = 0xFFFE
CHROM_INVALID = 0xFFFF
CELL_INVALID = 0xFFFFFFFF
MAX_CHROM_IDS = 0xFFF0

_UMI_CODE = {"A": 1, "C": 2, "G": 3, "N": 4, "T": 5}      # ASCII order, 0 = end of string
UMI_MAX_LEN = 21


def encode_umi(umi):
    """Order-preserving 63-bit code: 3 bits per character, left aligned, 0-padded, so that integer
    order == Python str order (shorter prefix first) -- the bundle files are sorted by UMI string
    (te_count.py:358) and the Part-2 scan drops the smallest one, so order is observable."""
    n = len(umi)
    if n > UMI_MAX_LEN:
        raise ValueError("UMI %r longer than %d characters" % (umi, UMI_MAX_LEN))
    code = 0
    try:
        for ch in umi:
            code = (code << 3) | _UMI_CODE[ch]
    except KeyError:
        raise ValueError("UMI %r has a character outside A,C,G,N,T" % (umi,))
    return code << (3 * (UMI_MAX_LEN - n))


class ChromMap:
    """reference_name -> u16 id.  ids < n_index are index chromosomes (same ids as GlbIndex);
    other names get fresh ids >= n_index (needed by the sc chrom:strand comparison,
    te_count.py:446-452, which also sees chromosomes that are not in the index)."""

    def __init__(self, index_chrom_keys):
        self.n_index = len(index_chrom_keys)
        self._key_id = {k: i for i, k in enumerate(index_chrom_keys)}
        self._name_bulk = {}
        self._name_sc = {}

    def _key(self, reference_name):
        key = reference_name.replace("chr", "")
        cid = self._key_id.get(key)
        if cid is None:
            cid = len(self._key_id)
            if cid >= MAX_CHROM_IDS:
                raise ValueError("more than %d distinct chromosome names" % MAX_CHROM_IDS)
            self._key_id[key] = cid
        return key, cid

    def bulk_id(self, reference_name):
        """Bulk mode only asks `chrom in buckets` (te_count.py:100 / :216): a name that is not an index
        chromosome needs no id of its own (a header may list far more sequences than there are u16 ids)."""
        cid = self._name_bulk.get(reference_name)
        if cid is None:
            if reference_name is None:
                cid = CHROM_INVALID
            else:
                cid = self._key_id.get(reference_name.replace("chr", ""), CHROM_INVALID)
                if cid >= self.n_index:
                    cid = CHROM_INVALID
            self._name_bulk[reference_name] = cid
        return cid

    def sc_id(self, reference_name):
        cid = self._name_sc.get(reference_name)
        if cid is None:
            key, cid = self._key(reference_name)
            if "_" in key or "alt" in key:
                cid = CHROM_SC_SKIP
            elif ":" in key:
                # the reference re-splits 'chrom:strand:left:rite' on ':' (te_count.py:605) and
                # then raises ValueError or silently mis-keys; not reproduced
                raise ValueError("chromosome name %r contains ':' (unsupported in --sc)" % reference_name)
            self._name_sc[reference_name] = cid
        return cid


class Whitelist:
    """te_count.py:328-339."""

    def __init__(self, filename):
        import os
        if not os.path.exists(filename):
            raise AssertionError(f'{filename} -w whitelist file not found')
        wl = []
        with open(filename, "r") as oh:
            for line in oh:
                wl.append(line.strip())
        self.id_to_barcode = sorted(set(wl))
        self.barcode_to_id = {bc: i for i, bc in enumerate(self.id_to_barcode)}

    def __len__(self):
        return len(self.id_to_barcode)


def _flagbits(read):
    f = 0
    if read.is_unmapped:
        f |= F_UNMAPPED
    if read.is_duplicate:
        f |= F_DUP
    if read.is_qcfail:
        f |= F_QCFAIL
    if read.is_reverse:
        f |= F_REVERSE
    return f


class Batch:
    """Preallocated SoA buffers (pinned when the library hands out the memory).  named: pairing by read name also
    carries each record's SAM flag and QNAME (fill_bulk_named)."""

    def __init__(self, capacity, sc=False, alloc=None, named=False):
        alloc = alloc or (lambda n, dt: np.empty(n, dtype=dt))
        self.capacity = capacity
        self.start = alloc(capacity, np.int32)
        self.end = alloc(capacity, np.int32)
        self.chrom = alloc(capacity, np.uint16)
        self.mapq = alloc(capacity, np.uint8)
        self.flag = alloc(capacity, np.uint8)
        self.cell = alloc(capacity, np.uint32) if sc else None
        self.umi = alloc(capacity, np.uint64) if sc else None
        self.samflag = alloc(capacity, np.uint16) if named else None
        self.name_off = np.zeros(capacity + 1, dtype=np.int64) if named else None
        self.names = b""
        self.n = 0


def fill_bulk(batch, sam, chrom_map, paired, qual):
    """Pull up to batch.capacity records (an even number when paired) from the pysam iterator.
    Returns False when the iterator is exhausted.  A trailing unpaired record is dropped, as
    the second next() of te_count.py:79 raises StopIteration."""
    start, end, chrom, mapq, flag = batch.start, batch.end, batch.chrom, batch.mapq, batch.flag
    n = 0
    cap = batch.capacity - (batch.capacity & 1 if paired else 0)
    more = True
    bulk_id = chrom_map.bulk_id
    while n < cap:
        try:
            r1 = next(sam)
        except StopIteration:
            more = False
            break
        f1 = _flagbits(r1)
        if paired:
            try:
                r2 = next(sam)
            except StopIteration:
                more = False
                break
            f2 = _flagbits(r2)
            rejected = (f1 | f2) & (F_UNMAPPED | F_DUP | F_QCFAIL) or int(r1.mapping_quality) < qual
            if not rejected:
                a = r1.query_name.split('/')
                b = r2.query_name.split('/')
                if '_'.join(a[0:-1]) != '_'.join(b[0:-1]):
                    f1 |= F_NAME_MISMATCH
            start[n] = r1.reference_start if r1.reference_start is not None else -1
            end[n] = r1.reference_end if r1.reference_end is not None else -1
            chrom[n] = bulk_id(r1.reference_name)
            mapq[n] = int(r1.mapping_quality)
            flag[n] = f1
            n += 1
            s2 = r2.reference_start
            if s2 is None:
                if not rejected:
                    raise TypeError("unsupported operand type(s) for +: 'NoneType' and 'int'")
                s2 = -1
            start[n] = s2
            end[n] = r2.reference_end if r2.reference_end is not None else -1
            chrom[n] = bulk_id(r2.reference_name)
            mapq[n] = int(r2.mapping_quality)
            flag[n] = f2
            n += 1
        else:
            e1 = r1.reference_end
            if e1 is None:
                if not (f1 & (F_UNMAPPED | F_DUP | F_QCFAIL)) and int(r1.mapping_quality) >= qual \
                        and bulk_id(r1.reference_name) < chrom_map.n_index:
                    # te_count.py:223  (loc2+1) with loc2 = None
                    raise TypeError("unsupported operand type(s) for +: 'NoneType' and 'int'")
                e1 = -1
            start[n] = r1.reference_start if r1.reference_start is not None else -1
            end[n] = e1
            chrom[n] = bulk_id(r1.reference_name)
            mapq[n] = int(r1.mapping_quality)
            flag[n] = f1
            n += 1
    batch.n = n
    return more


def fill_bulk_named(batch, sam, chrom_map):
    """Pairing by read name (libtecount tec_bulk_push_named): one row per record in file order, as for single end,
    plus its SAM flag and its QNAME bytes (batch.names, record i at [name_off[i], name_off[i + 1])).  Which records
    pair is decided on the device.  Returns False when the iterator is exhausted."""
    start, end, chrom, mapq, flag, samflag = batch.start, batch.end, batch.chrom, batch.mapq, batch.flag, batch.samflag
    names = []
    n = 0
    more = True
    bulk_id = chrom_map.bulk_id
    while n < batch.capacity:
        try:
            r = next(sam)
        except StopIteration:
            more = False
            break
        s, e = r.reference_start, r.reference_end
        start[n] = s if s is not None else -1
        end[n] = e if e is not None else -1
        chrom[n] = bulk_id(r.reference_name)
        mapq[n] = int(r.mapping_quality)
        flag[n] = _flagbits(r)
        samflag[n] = int(r.flag)
        names.append(r.query_name.encode())
        n += 1
    batch.name_off[0] = 0
    if n:
        np.cumsum([len(x) for x in names], out=batch.name_off[1:n + 1])
    batch.names = b"".join(names)
    batch.n = n
    return more


def fill_sc(batch, sam, chrom_map, whitelist, qual, umis=True, umi_base=0):
    """Single-cell variant (te_count.py:393-438).  Tags are only looked at for records that pass the
    flag and MAPQ tests, exactly where the reference would raise AssertionError for a missing tag.
    umis=False is the opt-in --noumi extension (measureTE(extensions=True)): UB / UR are not looked at and
    the UMI code of a record is its ordinal in the file, umi_base + position in the batch."""
    start, end, chrom, mapq, flag = batch.start, batch.end, batch.chrom, batch.mapq, batch.flag
    cell, umi = batch.cell, batch.umi
    n = 0
    cap = batch.capacity
    more = True
    sc_id = chrom_map.sc_id
    bc_to_id = whitelist.barcode_to_id
    umi_cache = {}
    while n < cap:
        try:
            r = next(sam)
        except StopIteration:
            more = False
            break
        f = _flagbits(r)
        q = int(r.mapping_quality)
        mapq[n] = q
        flag[n] = f
        if (f & (F_UNMAPPED | F_DUP | F_QCFAIL)) or q < qual:
            start[n] = -1
            end[n] = -1
            chrom[n] = CHROM_INVALID
            cell[n] = CELL_INVALID
            umi[n] = 0
            n += 1
            continue
        tags = dict(r.get_tags())
        if 'CB' in tags:
            barcode = tags['CB']
        elif 'CR' in tags:
            barcode = tags['CR']
        else:
            raise AssertionError('CB or CR tag not found!')
        cid = bc_to_id.get(barcode)
        if cid is None:
            start[n] = -1
            end[n] = -1
            chrom[n] = CHROM_INVALID
            cell[n] = CELL_INVALID
            umi[n] = 0
            n += 1
            continue
        if not umis:
            code = umi_base + n
        else:
            if 'UB' in tags:
                u = tags['UB']
            elif 'UR' in tags:
                u = tags['UR']
            else:
                raise AssertionError('UB or UR tag not found!')
            code = umi_cache.get(u)
            if code is None:
                code = encode_umi(u)
                if len(umi_cache) < (1 << 20):
                    umi_cache[u] = code
        c = sc_id(r.reference_name)
        start[n] = r.reference_start
        e = r.reference_end
        if e is None:
            if c != CHROM_SC_SKIP:
                raise TypeError("reference_end is None for a counted read")
            e = -1
        end[n] = e
        chrom[n] = c
        cell[n] = cid
        umi[n] = code
        n += 1
    batch.n = n
    return more
