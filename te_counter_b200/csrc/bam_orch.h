// Window loop of the block-parallel BAM decoder (bgzf_dev.h has the per-block routines): file
// mapping, BGZF header walk, BAM header, carry of the cut record between windows, the exact chain
// check over the per-block guesses, pair alignment of windows, end of file.  Templated on a
// backend that owns the buffers and runs the three passes (inflate, find+hop, parse) -- CUDA
// kernels in bamgpu.cuh, plain loops in tools/bgzf_dev_host.cpp -- so that the orchestration that
// runs on the GPU box is the code the CPU tests exercise.
#pragma once
#include "bgzf_dev.h"

#include <zlib.h>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

namespace bamorch {

enum {
    OK = 0,
    E_IO = -1,
    E_FORMAT = -2,
    E_NOT_BGZF = -3,
    E_ARG = -4,
    E_UNSUPPORTED = -5,         // a layout this decoder refuses (use the host decoder for this file)
    E_BACKEND = -6,
    E_RECORD = -100             // minus bgzfdev::E_*: conditions on which the reference's loop raises
};

struct BlockDesc {
    uint64_t in_off;            // in the window's compressed staging buffer
    uint64_t out_off;           // in the window's uncompressed buffer
    uint32_t in_len, out_len, crc, pad;
};

struct BlockChain {
    int64_t start, exit, last;  // bgzfdev::find_start / Hop
    uint32_t count, bad;
};

struct MappedFile {
    int fd = -1;
    const uint8_t* map = nullptr;
    size_t size = 0;
    ~MappedFile() {
        if (map && size) munmap((void*)map, size);
        if (fd >= 0) close(fd);
    }
    int open_path(const char* path) {
        fd = open(path, O_RDONLY);
        struct stat st;
        if (fd < 0 || fstat(fd, &st) != 0) return E_IO;
        size = (size_t)st.st_size;
        if (size < 28) return E_NOT_BGZF;
        void* m = mmap(nullptr, size, PROT_READ, MAP_PRIVATE, fd, 0);
        if (m == MAP_FAILED) {
            size = 0;
            return E_IO;
        }
        map = (const uint8_t*)m;
        madvise(m, size, MADV_SEQUENTIAL);
        return map[0] == 0x1f && map[1] == 0x8b ? OK : E_NOT_BGZF;
    }
};

// One BGZF block header at file offset p: payload position and sizes.  Returns the block length, or a negative status.
inline int64_t bgzf_block_at(const MappedFile& f, size_t p, const uint8_t** cdata, uint32_t* clen, uint32_t* isize, uint32_t* crc) {
    if (f.size - p < 18) return E_FORMAT;
    const uint8_t* h = f.map + p;
    if (h[0] != 0x1f || h[1] != 0x8b || h[2] != 8) return E_FORMAT;
    if (!(h[3] & 4)) return E_NOT_BGZF;
    const uint32_t xlen = h[10] | (h[11] << 8);
    if (f.size - p < 12 + (size_t)xlen) return E_FORMAT;
    int64_t bsize = -1;
    for (uint32_t o = 0; o + 4 <= xlen;) {
        const uint32_t slen = h[12 + o + 2] | (h[12 + o + 3] << 8);
        if (h[12 + o] == 'B' && h[12 + o + 1] == 'C' && slen == 2 && o + 6 <= xlen) bsize = (int64_t)(h[12 + o + 4] | (h[12 + o + 5] << 8)) + 1;
        o += 4 + slen;
    }
    if (bsize < 0) return E_NOT_BGZF;
    if (bsize < (int64_t)(12 + xlen + 8) || (size_t)bsize > f.size - p) return E_FORMAT;
    *cdata = h + 12 + xlen;
    *clen = (uint32_t)(bsize - 12 - xlen - 8);
    *crc = bgzfdev::ld32(h + bsize - 8);
    *isize = bgzfdev::ld32(h + bsize - 4);
    if (*isize > 65536) return E_FORMAT;
    return bsize;
}

inline bool zlib_block(const uint8_t* in, uint32_t in_n, uint8_t* out, uint32_t out_n, uint32_t crc) {
    z_stream zs;
    memset(&zs, 0, sizeof(zs));
    if (inflateInit2(&zs, -15) != Z_OK) return false;
    zs.next_in = const_cast<Bytef*>(in);
    zs.avail_in = in_n;
    zs.next_out = out;
    zs.avail_out = out_n;
    const int rc = inflate(&zs, Z_FINISH);
    const bool ok = rc == Z_STREAM_END && zs.avail_out == 0;
    inflateEnd(&zs);
    return ok && (uint32_t)crc32(crc32(0L, Z_NULL, 0), out, out_n) == crc;
}

// CRC32 lookup table and the "append 2^k zero bytes" operators of bgzfdev::crc32_shift (zlib's crc32_combine
// construction: the operator for one zero BIT, squared 3 times -> one byte, then squared once per k).
inline void crc32_tables(uint32_t table[256], uint32_t mats[bgzfdev::CRC_SHIFT_MATS * 32]) {
    for (uint32_t i = 0; i < 256; i++) {
        uint32_t c = i;
        for (int k = 0; k < 8; k++) c = (c & 1) ? 0xEDB88320u ^ (c >> 1) : c >> 1;
        table[i] = c;
    }
    uint32_t a[32], b[32];
    a[0] = 0xEDB88320u;                         // one zero bit: reflected CRC shifts right
    for (int n = 1; n < 32; n++) a[n] = 1u << (n - 1);
    auto times = [](const uint32_t* m, uint32_t v) {
        uint32_t r = 0;
        for (int i = 0; v; v >>= 1, i++)
            if (v & 1) r ^= m[i];
        return r;
    };
    auto square = [&](uint32_t* dst, const uint32_t* src) {
        for (int n = 0; n < 32; n++) dst[n] = times(src, src[n]);
    };
    square(b, a);                               // 2 bits
    square(a, b);                               // 4 bits
    square(b, a);                               // 8 bits = one byte
    for (int k = 0; k < bgzfdev::CRC_SHIFT_MATS; k++) {
        memcpy(mats + 32 * k, b, sizeof(b));
        square(a, b);
        memcpy(b, a, sizeof(b));
    }
}

struct Reader {
    MappedFile file;
    size_t pos = 0;                         // next BGZF block
    std::vector<std::string> refs;
    std::vector<uint8_t> after_header;      // inflated bytes behind the BAM header (start of the first window)
    std::vector<uint16_t> bulk_ids, sc_ids;
    int32_t n_index = 0;
    bool have_map = false;
    // whitelist (host copy; the backend mirrors it where it parses)
    std::string wl_bytes;
    std::vector<int64_t> wl_off;
    std::vector<uint32_t> wl_slot;
    std::string err;

    int fail(int status, const std::string& msg) {
        err = msg;
        return status;
    }

    int open_path(const char* path) {
        int rc = file.open_path(path);
        if (rc) return fail(rc, rc == E_NOT_BGZF ? "not a BGZF file" : "cannot open or map the file");
        // BAM header: inflate blocks on the host until it is complete
        std::vector<uint8_t> buf;
        size_t need_bytes = 12, stage = 0, cur = 0;
        int32_t n_ref = 0, l_text = 0;
        for (;;) {
            while (buf.size() < cur + need_bytes) {
                if (pos >= file.size) return fail(E_FORMAT, "truncated BAM header");
                const uint8_t* cdata;
                uint32_t clen, isize, crc;
                const int64_t bs = bgzf_block_at(file, pos, &cdata, &clen, &isize, &crc);
                if (bs < 0) return fail((int)bs, "bad BGZF block in the header");
                const size_t old = buf.size();
                buf.resize(old + isize);
                if (isize && !zlib_block(cdata, clen, buf.data() + old, isize, crc)) return fail(E_FORMAT, "corrupt BGZF block in the header");
                pos += (size_t)bs;
            }
            if (stage == 0) {
                if (memcmp(buf.data(), "BAM\1", 4) != 0) return fail(E_FORMAT, "not a BAM file (magic)");
                l_text = (int32_t)bgzfdev::ld32(buf.data() + 4);
                if (l_text < 0) return fail(E_FORMAT, "negative header text length");
                cur = 8 + (size_t)l_text;
                need_bytes = 4;
                stage = 1;
            } else if (stage == 1) {
                n_ref = (int32_t)bgzfdev::ld32(buf.data() + cur);
                if (n_ref < 0) return fail(E_FORMAT, "negative reference count");
                cur += 4;
                need_bytes = 4;
                stage = 2;
                if (n_ref == 0) break;
            } else if (stage == 2) {
                const int32_t l_name = (int32_t)bgzfdev::ld32(buf.data() + cur);
                if (l_name < 0) return fail(E_FORMAT, "negative reference name length");
                need_bytes = 8 + (size_t)l_name;
                stage = 3;
            } else {
                const int32_t l_name = (int32_t)bgzfdev::ld32(buf.data() + cur);
                const char* nm = (const char*)buf.data() + cur + 4;
                refs.emplace_back(nm, strnlen(nm, (size_t)l_name));
                cur += 8 + (size_t)l_name;
                need_bytes = 4;
                stage = 2;
                if ((int32_t)refs.size() == n_ref) break;
            }
        }
        after_header.assign(buf.begin() + (ptrdiff_t)cur, buf.end());
        return OK;
    }

    int set_chrom_map(const uint16_t* b, const uint16_t* s, int32_t n, int32_t n_idx) {
        if (n != (int32_t)refs.size() || n_idx < 0 || (n && (!b || !s))) return fail(E_ARG, "chrom map must have one entry per reference sequence");
        bulk_ids.assign(b, b + n);
        sc_ids.assign(s, s + n);
        n_index = n_idx;
        have_map = true;
        return OK;
    }

    int set_whitelist(const char* bytes, const int64_t* off, int32_t n) {
        if (n < 0 || !off || off[0] != 0) return fail(E_ARG, "bad whitelist arguments");
        for (int32_t i = 0; i < n; i++)
            if (off[i + 1] < off[i]) return fail(E_ARG, "whitelist offsets must ascend");
        wl_off.assign(off, off + n + 1);
        wl_bytes.assign(bytes ? bytes : "", (size_t)off[n]);
        size_t cap = 16;
        while (cap < 2 * (size_t)n + 2) cap <<= 1;
        wl_slot.assign(cap, 0);
        for (int32_t i = 0; i < n; i++) {
            uint64_t h = bgzfdev::wl_hash((const uint8_t*)wl_bytes.data() + off[i], (uint32_t)(off[i + 1] - off[i])) & (cap - 1);
            while (wl_slot[h]) h = (h + 1) & (cap - 1);
            wl_slot[h] = (uint32_t)(i + 1);
        }
        return OK;
    }

    // the parse context over the host copies of the maps
    bgzfdev::ParseCtx host_parse_ctx(int qual) const {
        bgzfdev::ParseCtx pc;
        pc.bulk_ids = bulk_ids.data(); pc.sc_ids = sc_ids.data(); pc.n_ref = (int32_t)refs.size(); pc.n_index = n_index; pc.qual = qual;
        pc.wl.slot = wl_slot.data(); pc.wl.off = wl_off.data(); pc.wl.bytes = (const uint8_t*)wl_bytes.data();
        pc.wl.mask = wl_slot.empty() ? 0 : wl_slot.size() - 1;
        return pc;
    }
};

// One paired-end pair parsed on the host from two raw records (block_size word included), with the file's chromosome
// map: the pair across the border of two byte ranges (decode_range).  Same routine as the device pass, rows 0 and 1.
inline int parse_pair(Reader& r, const uint8_t* rec1, int64_t n1, const uint8_t* rec2, int64_t n2, int qual,
                      int32_t* start, int32_t* end, uint16_t* chrom, uint8_t* mapq, uint8_t* flag) {
    if (!r.have_map) return r.fail(E_ARG, "the chromosome map has not been set");
    auto whole = [](const uint8_t* p, int64_t n) {
        return n >= 36 && n <= 4 + (int64_t)bgzfdev::MAX_BLOCK_SIZE && (int64_t)bgzfdev::ld32(p) + 4 == n;
    };
    if (!whole(rec1, n1) || !whole(rec2, n2)) return r.fail(E_ARG, "a mate is not one complete alignment record");
    std::vector<uint8_t> w((size_t)(n1 + n2));
    memcpy(w.data(), rec1, (size_t)n1);
    memcpy(w.data() + n1, rec2, (size_t)n2);
    const int64_t off[2] = {0, n1};
    const bgzfdev::ParseCtx pc = r.host_parse_ctx(qual);
    const bgzfdev::Columns set{start, end, chrom, mapq, flag, nullptr, nullptr};
    const int e = bgzfdev::parse_adjacent_pair(w.data(), off, 0, 0, pc, &set);
    if (e) return r.fail(E_RECORD - e, "the pair across the range border");
    return OK;
}

/*
 * Backend concept:
 *   int  reserve(size_t comp_bytes, size_t ubuf_bytes, int n_blocks)   grow the window buffers (ubuf content is kept)
 *   int  load(const MappedFile&, size_t lo, size_t n)                  file bytes [lo, lo + n) = the window's compressed blocks
 *   int  put(int64_t at, const uint8_t* data, size_t n)                host bytes into the uncompressed window
 *   int  carry(int64_t from, int64_t n)                                ubuf[0, n) = ubuf[from, from + n)
 *   int  inflate(const BlockDesc*, int n_blocks, int32_t* status)      bgzfdev::inflate_block + crc32_block per block (in_off relative to lo)
 *   int  chain(const BlockDesc*, int n_blocks, int64_t w_end, int32_t n_ref, BlockChain* out) find_start (block 0 starts at 0) + hop per block
 *   int  parse(const BlockDesc*, int n_blocks, const BlockChain* used, const int64_t* base, int64_t n_records, int64_t w_end,
 *              int mode, int qual, const Reader&, int* err, int64_t* err_rec)                 parse_record per record into the columns
 *   int  deliver(int64_t n_records, int mode)                          hand the columns on (tec_*_push_dev / copy out; MODE_PE_NAME:
 *                                                                      the rows, keys and roles to the pairing stage, pair_name.cuh;
 *                                                                      MODE_PE_NAME_RANGE: the same rows appended to its held set)
 * and for paired-end byte ranges (decode_range with MODE_PE):
 *   int  parse_pairs(const BlockChain*, const int64_t* base, int nb, int64_t n_records, int64_t g0, int qual, const Reader&,
 *                    int* err, int64_t* err_rec)                       parse_adjacent_pair per adjacent pair into the two column sets
 *   int  deliver_pairs(int64_t pairs0, int64_t pairs1)                 hand column set b on to counter bank b
 *   int  fetch(int64_t at, uint8_t* dst, size_t n)                     window bytes to the host
 */
template <class Backend>
int decode_all(Reader& r, Backend& be, int mode, int qual, int window_blocks, int64_t* n_records_out) {
    if (!r.have_map) return r.fail(E_ARG, "the chromosome map has not been set");
    if (window_blocks < 1) window_blocks = 1;
    const bool paired = mode == bgzfdev::MODE_PE;
    int64_t carry_n = (int64_t)r.after_header.size(), total_records = 0;
    bool carry_is_lone_mate = false;
    std::vector<BlockDesc> blocks;
    std::vector<const uint8_t*> src;
    std::vector<int32_t> status;
    std::vector<BlockChain> chain;
    std::vector<int64_t> base;
    std::vector<uint8_t> tmp;
    int rc = be.reserve(1, (size_t)carry_n + 1, 1);
    if (rc) return r.fail(E_BACKEND, "backend: cannot allocate the window");
    if (carry_n && be.put(0, r.after_header.data(), (size_t)carry_n)) return r.fail(E_BACKEND, "backend: copy failed");
    bool first = true;
    for (;;) {
        blocks.clear();
        src.clear();
        size_t total = 0;
        const size_t file_lo = r.pos;
        while (r.pos < r.file.size && (int)blocks.size() < window_blocks) {
            const uint8_t* cdata;
            uint32_t clen, isize, crc;
            const int64_t bs = bgzf_block_at(r.file, r.pos, &cdata, &clen, &isize, &crc);
            if (bs < 0) return r.fail((int)bs, bs == E_NOT_BGZF ? "gzip member without a BC field: not BGZF" : "bad or truncated BGZF block");
            r.pos += (size_t)bs;
            if (!isize) continue;
            BlockDesc d;
            d.in_off = (uint64_t)(cdata - r.file.map) - file_lo; d.in_len = clen; d.out_off = (uint64_t)carry_n + total; d.out_len = isize;
            d.crc = crc; d.pad = 0;
            blocks.push_back(d);
            src.push_back(cdata);
            total += isize;
        }
        const int nb = (int)blocks.size();
        const int64_t w_end = carry_n + (int64_t)total;
        // Behind a processed window the carry holds no complete record (only the cut one, or the
        // unpaired one), so a round without new blocks is only worth it for the bytes that came
        // with the header.
        if (!nb && (!first || !carry_n)) break;
        first = false;
        if (nb) {
            const size_t comp = r.pos - file_lo;
            rc = be.reserve(comp + 16, (size_t)w_end + 64, nb);
            if (rc) return r.fail(E_BACKEND, "backend: cannot allocate the window");
            if (be.load(r.file, file_lo, comp)) return r.fail(E_BACKEND, "backend: reading the compressed blocks failed");
            status.assign((size_t)nb, 0);
            if (be.inflate(blocks.data(), nb, status.data())) return r.fail(E_BACKEND, "backend: inflate pass failed");
            for (int i = 0; i < nb; i++) {
                if (status[(size_t)i] == bgzfdev::ST_OK) continue;
                const BlockDesc& d = blocks[(size_t)i];               // the block-parallel inflate declined: zlib decides
                tmp.resize(d.out_len);
                if (!zlib_block(src[(size_t)i], d.in_len, tmp.data(), d.out_len, d.crc))
                    return r.fail(E_FORMAT, "corrupt BGZF block (inflate or CRC32 failed)");
                if (be.put((int64_t)d.out_off, tmp.data(), d.out_len)) return r.fail(E_BACKEND, "backend: copy failed");
            }
        }
        // ---- record boundaries: per-block guesses, then the exact chain check
        BlockDesc whole;
        whole.in_off = 0; whole.in_len = 0; whole.out_off = 0; whole.out_len = (uint32_t)0; whole.crc = 0; whole.pad = 0;
        if (!nb) {                              // only the bytes behind the header: one pseudo block over them
            blocks.push_back(whole);
            blocks[0].out_len = (uint32_t)w_end;
        }
        const int nc = (int)blocks.size();
        chain.assign((size_t)nc, BlockChain());
        if (be.chain(blocks.data(), nc, w_end, (int32_t)r.refs.size(), chain.data())) return r.fail(E_BACKEND, "backend: chain pass failed");
        int64_t expect = 0, n_rec = 0;
        bool stopped = false;
        int last_used = -1;
        for (int b = 0; b < nc; b++) {
            const int64_t hi = (int64_t)blocks[(size_t)b].out_off + blocks[(size_t)b].out_len;
            BlockChain& c = chain[(size_t)b];
            if (stopped || expect >= hi) {      // no record starts in this block
                c.count = 0;
                c.start = bgzfdev::NO_START;
                continue;
            }
            if (expect + 36 > w_end) {          // fewer bytes left than any record has: the cut record, carried on
                stopped = true;
                c.count = 0;
                c.start = bgzfdev::NO_START;
                continue;
            }
            if (c.start != expect) {
                char buf[160];
                snprintf(buf, sizeof buf, "record boundaries could not be established block-parallel (block %d of the window: guess %lld, chain %lld)",
                         b, (long long)c.start, (long long)expect);
                return r.fail(E_UNSUPPORTED, buf);
            }
            if (c.bad) return r.fail(E_FORMAT, "alignment record with impossible block_size");
            n_rec += c.count;
            if (c.count) last_used = b;
            expect = c.exit;
            if (c.exit < hi) stopped = true;    // the chain stands in front of a record that ends outside the window
        }
        carry_is_lone_mate = false;
        if (paired && (n_rec & 1)) {            // windows hold whole pairs: the odd record waits for its mate
            BlockChain& c = chain[(size_t)last_used];
            carry_is_lone_mate = expect == w_end;
            expect = c.last;
            c.count--;
            n_rec--;
        }
        base.assign((size_t)nc, 0);
        int64_t acc = 0;
        for (int b = 0; b < nc; b++) {
            base[(size_t)b] = acc;
            acc += chain[(size_t)b].count;
        }
        if (n_rec) {
            int err = 0;
            int64_t err_rec = -1;
            if (be.parse(blocks.data(), nc, chain.data(), base.data(), n_rec, w_end, mode, qual, r, &err, &err_rec))
                return r.fail(E_BACKEND, "backend: parse pass failed");
            if (err) {
                char buf[96];
                snprintf(buf, sizeof buf, "record %lld", (long long)(total_records + err_rec));
                return r.fail(E_RECORD - err, buf);
            }
            if (be.deliver(n_rec, mode)) return r.fail(E_BACKEND, "backend: delivering the batch failed");
            total_records += n_rec;
        }
        const int64_t left = w_end - expect;
        if (left && expect && be.carry(expect, left)) return r.fail(E_BACKEND, "backend: carry failed");
        carry_n = left;
    }
    if (carry_n && !(paired && carry_is_lone_mate)) return r.fail(E_FORMAT, "truncated BAM file (partial record at the end)");
    if (n_records_out) *n_records_out = total_records;
    return OK;
}


// ---- one BYTE RANGE of the file (several ranks split one BAM; SURVEY.md 8e "reads shard ... across the GPUs") ----
// Rank r decodes the records that START in the BGZF blocks whose first byte lies in [lo, hi).  Its first block is the
// first block start at or after lo (found by scanning for a header that is followed by two more); its first record
// is the block-parallel GUESS of that block (find_start) -- unless the range begins at the BAM header, where the start
// is known.  The last record may end beyond hi: RANGE_TAIL_BLOCKS / RANGE_TAIL_BYTES further blocks are inflated so that it is
// complete, and the position where the chain then stands (`exit`) is where the next rank's first record must start.
// The caller compares every rank's exit with the next rank's start (both as {file offset of the block, offset inside
// its inflated data}): by induction from rank 0, whose start is exact, equality everywhere means every rank decoded
// exactly its share of the true record chain; any difference means a wrong guess and the caller must decode the file
// in one piece instead.
// Paired end: pairs are formed by the GLOBAL record parity, which a range does not know until the ranks in front of it
// have counted their records.  So every adjacent pair (j, j + 1) of the range (range-local indices) is parsed, into
// column set j & 1 (parse_pairs / deliver_pairs: two counter banks); the caller keeps the set of the range's global
// offset once it is known, and parses the pair across the border from the raw first / last records kept here.  The last
// complete record of a window is carried into the next one, so the pair across two windows is formed exactly once.
// Paired end by read name (MODE_PE_NAME_RANGE): a mate may lie in any range, so the range pairs nothing; its rows are
// delivered one per record, as in single end, and the caller exchanges them by name owner before they are paired.
constexpr int RANGE_TAIL_BLOCKS = 16;               // blocks behind the range that are inflated for its last record:
constexpr size_t RANGE_TAIL_BYTES = size_t(1) << 20;   // at least 16 of them and at least 1 MiB of inflated data
struct RangeResult {
    int64_t n_records = 0;
    int64_t start_block = -1, start_off = 0;      // -1: the range starts at the BAM header (exact); -2: no record starts in the range
    int64_t exit_block = -2, exit_off = 0;        // where the next record starts; block == file size: end of file
    std::vector<uint8_t> first_rec, last_rec;     // paired end: raw bytes (block_size word included) of the first / last record
};

// raw bytes of the record at window offset p (block_size word included)
template <class Backend>
int fetch_record(Backend& be, int64_t p, std::vector<uint8_t>& out) {
    uint8_t w[4];
    if (be.fetch(p, w, 4)) return 1;
    out.resize(4 + (size_t)bgzfdev::ld32(w));
    return be.fetch(p, out.data(), out.size());
}

inline bool bgzf_chain_ok(const MappedFile& f, size_t p, int n) {
    for (int i = 0; i < n && p < f.size; i++) {
        const uint8_t* cdata; uint32_t clen, isize, crc;
        const int64_t bs = bgzf_block_at(f, p, &cdata, &clen, &isize, &crc);
        if (bs < 0) return false;
        p += (size_t)bs;
    }
    return true;
}

template <class Backend>
int decode_range(Reader& r, Backend& be, int mode, int qual, int window_blocks, uint64_t lo, uint64_t hi, RangeResult* res) {
    if (!r.have_map) return r.fail(E_ARG, "the chromosome map has not been set");
    if (!res || lo > hi) return r.fail(E_ARG, "bad byte range");
    if (mode == bgzfdev::MODE_PE_NAME) return r.fail(E_ARG, "pairing by read name needs the whole file: no byte ranges");
    // MODE_PE_NAME_RANGE: one MODE_PE_NAME row per record, delivered under the range mode (the rows are held, not paired)
    const int parse_mode = mode == bgzfdev::MODE_PE_NAME_RANGE ? bgzfdev::MODE_PE_NAME : mode;
    if (window_blocks < 1) window_blocks = 1;
    *res = RangeResult();
    const bool paired = mode == bgzfdev::MODE_PE;
    int64_t carried = 0;                        // paired: the window begins with a record an earlier window counted (0 or 1)
    const size_t fsize = r.file.size;
    const size_t hi_eff = (size_t)std::min<uint64_t>(hi, fsize);
    const bool from_header = lo == 0;           // rank 0: the chain starts behind the BAM header, exactly
    size_t pos = r.pos;
    int64_t carry_n = 0;
    bool adopted = from_header;                 // the chain has a first record
    if (from_header) {
        carry_n = (int64_t)r.after_header.size();
        res->start_block = -1;
    } else {
        pos = std::max((size_t)lo, r.pos);      // the header's own blocks belong to rank 0
        while (pos + 18 <= fsize && !(r.file.map[pos] == 0x1f && r.file.map[pos + 1] == 0x8b && r.file.map[pos + 2] == 8 &&
                                      (r.file.map[pos + 3] & 4) && bgzf_chain_ok(r.file, pos, 3)))
            pos++;
        if (pos + 18 > fsize) pos = fsize;
        res->start_block = -2;
    }
    if (pos >= hi_eff && !from_header) {                        // no block starts in the range
        res->exit_block = -2;
        return OK;
    }
    std::vector<BlockDesc> blocks;
    std::vector<const uint8_t*> src;
    std::vector<size_t> foff;                   // file offset of every block of the window
    std::vector<int32_t> status;
    std::vector<BlockChain> chain;
    std::vector<int64_t> base;
    std::vector<uint8_t> tmp;
    int rc = be.reserve(1, (size_t)carry_n + 1, 1);
    if (rc) return r.fail(E_BACKEND, "backend: cannot allocate the window");
    if (carry_n && be.put(0, r.after_header.data(), (size_t)carry_n)) return r.fail(E_BACKEND, "backend: copy failed");
    int64_t total_records = 0;
    bool final_window = false;
    while (!final_window) {
        blocks.clear(); src.clear(); foff.clear();
        size_t total = 0;
        const size_t file_lo = pos;
        auto take = [&]() -> int {
            const uint8_t* cdata; uint32_t clen, isize, crc;
            const int64_t bs = bgzf_block_at(r.file, pos, &cdata, &clen, &isize, &crc);
            if (bs < 0) return (int)bs;
            const size_t at = pos;
            pos += (size_t)bs;
            if (!isize) return OK;
            BlockDesc d;
            d.in_off = (uint64_t)(cdata - r.file.map) - file_lo; d.in_len = clen; d.out_off = (uint64_t)carry_n + total; d.out_len = isize;
            d.crc = crc; d.pad = 0;
            blocks.push_back(d); src.push_back(cdata); foff.push_back(at);
            total += isize;
            return OK;
        };
        while (pos < hi_eff && (int)blocks.size() < window_blocks) {
            const int t = take();
            if (t) return r.fail(t, t == E_NOT_BGZF ? "gzip member without a BC field: not BGZF" : "bad or truncated BGZF block");
        }
        final_window = pos >= hi_eff;
        const int n_main = (int)blocks.size();
        const int64_t boundary = carry_n + (int64_t)total;       // window position of the first block that is not ours
        if (final_window) {
            const int want = n_main + RANGE_TAIL_BLOCKS;
            const size_t main_bytes = total;
            while (pos < fsize && ((int)blocks.size() < want || total - main_bytes < RANGE_TAIL_BYTES)) {
                const int t = take();
                if (t) return r.fail(t, "bad or truncated BGZF block");
            }
        }
        const size_t next_file_pos = pos;                        // block behind the window (end of file: fsize)
        const int nb = (int)blocks.size();
        const int64_t w_end = carry_n + (int64_t)total;
        if (!nb && !carry_n && !from_header) {                   // nothing left (only empty blocks were skipped)
            if (adopted) { res->exit_block = (int64_t)next_file_pos; res->exit_off = 0; }
            break;
        }
        if (nb) {
            const size_t comp = pos - file_lo;
            rc = be.reserve(comp + 16, (size_t)w_end + 64, nb + 1);
            if (rc) return r.fail(E_BACKEND, "backend: cannot allocate the window");
            if (be.load(r.file, file_lo, comp)) return r.fail(E_BACKEND, "backend: reading the compressed blocks failed");
            status.assign((size_t)nb, 0);
            if (be.inflate(blocks.data(), nb, status.data())) return r.fail(E_BACKEND, "backend: inflate pass failed");
            for (int i = 0; i < nb; i++) {
                if (status[(size_t)i] == bgzfdev::ST_OK) continue;
                const BlockDesc& d = blocks[(size_t)i];
                tmp.resize(d.out_len);
                if (!zlib_block(src[(size_t)i], d.in_len, tmp.data(), d.out_len, d.crc))
                    return r.fail(E_FORMAT, "corrupt BGZF block (inflate or CRC32 failed)");
                if (be.put((int64_t)d.out_off, tmp.data(), d.out_len)) return r.fail(E_BACKEND, "backend: copy failed");
            }
        }
        // Block 0 of the chain pass "starts at 0" (the carry).  An empty pseudo block in front keeps that true while the
        // chain has no first record yet and lets every real block make its own guess.
        BlockDesc pseudo;
        pseudo.in_off = 0; pseudo.in_len = 0; pseudo.out_off = 0; pseudo.out_len = 0; pseudo.crc = 0; pseudo.pad = 0;
        int shift = 0;
        if (!adopted || !n_main) {
            if (!n_main) pseudo.out_len = (uint32_t)carry_n;      // no block of ours in this window: only the carried bytes
            blocks.insert(blocks.begin(), pseudo);
            foff.insert(foff.begin(), 0);
            shift = 1;
        }
        const int nc = (int)blocks.size();
        chain.assign((size_t)nc, BlockChain());
        if (be.chain(blocks.data(), nc, w_end, (int32_t)r.refs.size(), chain.data())) return r.fail(E_BACKEND, "backend: chain pass failed");
        int64_t expect = 0, n_rec = 0;
        bool stopped = false;
        int first_used = -1, last_used = -1;
        for (int b = 0; b < nc; b++) {
            const int64_t lo_b = (int64_t)blocks[(size_t)b].out_off, hi_b = lo_b + blocks[(size_t)b].out_len;
            BlockChain& c = chain[(size_t)b];
            const bool ours = b - shift < n_main || (shift && b == 0);
            if (!adopted) {                                      // the first block that shows a record start gives the chain its start
                if (b == 0 || !ours || c.start == bgzfdev::NO_START) { c.count = 0; c.start = bgzfdev::NO_START; continue; }
                adopted = true;
                expect = c.start;
                res->start_block = (int64_t)foff[(size_t)b];
                res->start_off = c.start - lo_b;
            }
            if (stopped || expect >= hi_b || !ours) { c.count = 0; c.start = bgzfdev::NO_START; continue; }
            if (expect + 36 > w_end) { stopped = true; c.count = 0; c.start = bgzfdev::NO_START; continue; }
            if (c.start != expect) {
                char buf[160];
                snprintf(buf, sizeof buf, "record boundaries could not be established block-parallel (block %d of the window: guess %lld, chain %lld)",
                         b, (long long)c.start, (long long)expect);
                return r.fail(E_UNSUPPORTED, buf);
            }
            if (c.bad) return r.fail(E_FORMAT, "alignment record with impossible block_size");
            n_rec += c.count;
            if (c.count) { if (first_used < 0) first_used = b; last_used = b; }
            expect = c.exit;
            if (c.exit < hi_b) stopped = true;
        }
        if (!adopted) { carry_n = 0; continue; }                 // nothing starts in this window: its bytes belong to the rank before
        base.assign((size_t)nc, 0);
        int64_t acc = 0;
        for (int b = 0; b < nc; b++) { base[(size_t)b] = acc; acc += chain[(size_t)b].count; }
        if (paired && n_rec) {
            // n_rec complete records, the carried one included: n_rec - 1 adjacent pairs, the first record at range index g0
            const int64_t g0 = total_records - carried;
            if (res->first_rec.empty() && fetch_record(be, chain[(size_t)first_used].start, res->first_rec))
                return r.fail(E_BACKEND, "backend: copy failed");
            if (fetch_record(be, chain[(size_t)last_used].last, res->last_rec)) return r.fail(E_BACKEND, "backend: copy failed");
            if (n_rec > 1) {
                int err = 0;
                int64_t err_rec = -1;
                if (be.parse_pairs(chain.data(), base.data(), nc, n_rec, g0, qual, r, &err, &err_rec))
                    return r.fail(E_BACKEND, "backend: parse pass failed");
                if (err) {
                    char buf[96];
                    snprintf(buf, sizeof buf, "record %lld of the range", (long long)(g0 + err_rec));
                    return r.fail(E_RECORD - err, buf);
                }
                if (be.deliver_pairs(bgzfdev::pairs_in_set(n_rec, g0, 0), bgzfdev::pairs_in_set(n_rec, g0, 1)))
                    return r.fail(E_BACKEND, "backend: delivering the batch failed");
            }
            total_records += n_rec - carried;
            if (!final_window) {                                 // the last record pairs with the first one of the next window
                expect = chain[(size_t)last_used].last;
                carried = 1;
            }
        } else if (n_rec) {
            int err = 0;
            int64_t err_rec = -1;
            if (be.parse(blocks.data(), nc, chain.data(), base.data(), n_rec, w_end, parse_mode, qual, r, &err, &err_rec))
                return r.fail(E_BACKEND, "backend: parse pass failed");
            if (err) {
                char buf[96];
                snprintf(buf, sizeof buf, "record %lld of the range", (long long)(total_records + err_rec));
                return r.fail(E_RECORD - err, buf);
            }
            if (be.deliver(n_rec, mode)) return r.fail(E_BACKEND, "backend: delivering the batch failed");
            total_records += n_rec;
        }
        if (final_window) {
            if (expect < boundary) {
                if (next_file_pos >= fsize && nb - n_main == 0) return r.fail(E_FORMAT, "truncated BAM file (partial record at the end)");
                char buf[200];
                snprintf(buf, sizeof buf, "the last record of the range does not end within the tail window (chain at %lld, range ends at %lld, window %lld, %d + %d blocks)",
                         (long long)expect, (long long)boundary, (long long)w_end, n_main, nb - n_main);
                return r.fail(E_UNSUPPORTED, buf);
            }
            // the chain stands at `expect`: in one of the tail blocks, or right behind the window
            res->exit_block = (int64_t)next_file_pos;
            res->exit_off = 0;
            if (expect > w_end) return r.fail(E_FORMAT, "record chain runs past the window");
            for (int b = shift + n_main; b < nc; b++) {
                const int64_t lo_b = (int64_t)blocks[(size_t)b].out_off, hi_b = lo_b + blocks[(size_t)b].out_len;
                if (expect >= lo_b && expect < hi_b) { res->exit_block = (int64_t)foff[(size_t)b]; res->exit_off = expect - lo_b; break; }
            }
            break;
        }
        const int64_t left = w_end - expect;
        if (left && expect && be.carry(expect, left)) return r.fail(E_BACKEND, "backend: carry failed");
        carry_n = left;
    }
    if (!adopted) { res->start_block = -2; res->exit_block = -2; }
    res->n_records = total_records;
    return OK;
}

}  // namespace bamorch
