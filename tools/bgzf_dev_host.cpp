// TEST INFRASTRUCTURE: the block-parallel BAM decoder (te_counter_b200/csrc/bgzf_dev.h per-block
// routines + bam_orch.h window loop) with a backend of plain host loops in place of the CUDA
// kernels of bamgpu.cuh.  Same routines, same orchestration, one "thread" after the other, so the
// CPU-only build box can hold the whole logic against libtecbam (tests/test_bgzf_dev_cpu.py).
// Build: g++ -O2 -std=c++17 -shared -fPIC tools/bgzf_dev_host.cpp -lz -o tools/libbgzfdevhost.so
#include "../te_counter_b200/csrc/bam_orch.h"

#include <algorithm>

namespace {

struct HostBackend {
    std::vector<uint8_t> comp, ubuf, scratch;
    std::vector<int32_t> c_start, c_end;
    std::vector<uint16_t> c_chrom;
    std::vector<uint8_t> c_mapq, c_flag;
    std::vector<uint32_t> c_cell;
    std::vector<uint64_t> c_umi, c_key_hi, c_key_lo;
    std::vector<uint8_t> c_role;
    // everything delivered so far
    std::vector<int32_t> o_start, o_end;
    std::vector<uint16_t> o_chrom;
    std::vector<uint8_t> o_mapq, o_flag;
    std::vector<uint32_t> o_cell;
    std::vector<uint64_t> o_umi, o_key_hi, o_key_lo;      // MODE_PE_NAME: name keys and roles
    std::vector<uint8_t> o_role;
    // paired-end ranges: the two column sets of the window, and everything delivered into each
    struct Set {
        std::vector<int32_t> start, end;
        std::vector<uint16_t> chrom;
        std::vector<uint8_t> mapq, flag;
    } p_win[2], p_out[2];
    uint32_t crc_table[256], crc_mats[bgzfdev::CRC_SHIFT_MATS * 32];
    int n_inflate_declined = 0;
    int force_decline_every = 0;                // test hook: pretend the block-parallel inflate declined every k-th block

    HostBackend() {
        bamorch::crc32_tables(crc_table, crc_mats);
        scratch.resize(bgzfdev::SCRATCH_STRIDE);
    }
    int reserve(size_t comp_bytes, size_t ubuf_bytes, int) {
        if (comp.size() < comp_bytes) comp.resize(comp_bytes);
        if (ubuf.size() < ubuf_bytes) ubuf.resize(ubuf_bytes);
        return 0;
    }
    int load(const bamorch::MappedFile& f, size_t lo, size_t n) {
        memcpy(comp.data(), f.map + lo, n);
        return 0;
    }
    int put(int64_t at, const uint8_t* data, size_t n) {
        memcpy(ubuf.data() + at, data, n);
        return 0;
    }
    int carry(int64_t from, int64_t n) {
        memmove(ubuf.data(), ubuf.data() + from, (size_t)n);
        return 0;
    }
    int inflate(const bamorch::BlockDesc* bl, int nb, int32_t* status) {
        for (int b = 0; b < nb; b++) {          // one CUDA thread per b
            const bamorch::BlockDesc& d = bl[b];
            int st = bgzfdev::inflate_block(comp.data() + d.in_off, d.in_len, ubuf.data() + d.out_off, d.out_len, scratch.data());
            if (st == bgzfdev::ST_OK) {         // the device computes it with the 32 lanes of the warp: same shares here, one after the other
                uint32_t c = 0;
                for (int lane = 0; lane < 32; lane++) c ^= bgzfdev::crc32_lane_share(ubuf.data() + d.out_off, d.out_len, lane, crc_table, crc_mats);
                if ((c ^ 0xFFFFFFFFu) != d.crc || bgzfdev::crc32_block(ubuf.data() + d.out_off, d.out_len, crc_table) != d.crc) st = bgzfdev::ST_CRC;
            }
            if (force_decline_every && b % force_decline_every == 0) {
                memset(ubuf.data() + d.out_off, 0xAB, d.out_len);
                st = bgzfdev::ST_DECLINED;
            }
            n_inflate_declined += st != bgzfdev::ST_OK;
            status[b] = st;
        }
        return 0;
    }
    int chain(const bamorch::BlockDesc* bl, int nb, int64_t w_end, int32_t n_ref, bamorch::BlockChain* out) {
        for (int b = 0; b < nb; b++) {
            const int64_t lo = (int64_t)bl[b].out_off, hi = lo + bl[b].out_len;
            const int64_t s = b == 0 ? 0 : bgzfdev::find_start(ubuf.data(), lo, hi, w_end, n_ref);
            bamorch::BlockChain c;
            c.start = s; c.exit = s; c.last = bgzfdev::NO_START; c.count = 0; c.bad = 0;
            if (s != bgzfdev::NO_START) {
                const bgzfdev::Hop h = bgzfdev::hop(ubuf.data(), s, hi, w_end);
                c.exit = h.exit; c.last = h.last; c.count = h.count; c.bad = h.bad;
            }
            out[b] = c;
        }
        return 0;
    }
    int parse(const bamorch::BlockDesc* bl, int nb, const bamorch::BlockChain* ch, const int64_t* base, int64_t n, int64_t, int mode, int qual,
              const bamorch::Reader& r, int* err, int64_t* err_rec) {
        c_start.resize((size_t)n); c_end.resize((size_t)n); c_chrom.resize((size_t)n); c_mapq.resize((size_t)n); c_flag.resize((size_t)n);
        c_cell.resize((size_t)n); c_umi.resize((size_t)n); c_key_hi.resize((size_t)n); c_key_lo.resize((size_t)n); c_role.resize((size_t)n);
        bgzfdev::Columns o{c_start.data(), c_end.data(), c_chrom.data(), c_mapq.data(), c_flag.data(), c_cell.data(), c_umi.data(),
                           c_key_hi.data(), c_key_lo.data(), c_role.data()};
        bgzfdev::ParseCtx pc;
        pc.bulk_ids = r.bulk_ids.data(); pc.sc_ids = r.sc_ids.data(); pc.n_ref = (int32_t)r.refs.size(); pc.n_index = r.n_index; pc.qual = qual;
        pc.wl.slot = r.wl_slot.data(); pc.wl.off = r.wl_off.data(); pc.wl.bytes = (const uint8_t*)r.wl_bytes.data();
        pc.wl.mask = r.wl_slot.empty() ? 0 : r.wl_slot.size() - 1;
        uint64_t first_err = ~uint64_t(0);
        (void)bl;
        for (int b = 0; b < nb; b++) {          // one CUDA thread per b
            int64_t p = ch[b].start;
            for (uint32_t i = 0; i < ch[b].count; i++) {
                const int64_t k = base[b] + i, nxt = p + 4 + (int64_t)bgzfdev::ld32(ubuf.data() + p);
                if (mode != bgzfdev::MODE_PE || !(k & 1)) {
                    const int e = bgzfdev::parse_record(ubuf.data(), p, nxt, mode, pc, o, k);
                    if (e) first_err = std::min(first_err, ((uint64_t)k << 8) | (uint64_t)e);
                }
                p = nxt;
            }
        }
        *err = 0;
        if (first_err != ~uint64_t(0)) {
            *err = (int)(first_err & 0xFF);
            *err_rec = (int64_t)(first_err >> 8);
        }
        return 0;
    }
    int parse_pairs(const bamorch::BlockChain* ch, const int64_t* base, int nb, int64_t n, int64_t g0, int qual, const bamorch::Reader& r,
                    int* err, int64_t* err_rec) {
        std::vector<int64_t> rec_off((size_t)n);
        for (int b = 0; b < nb; b++) {          // bam_list_kernel: one CUDA thread per b
            int64_t p = ch[b].start;
            for (uint32_t i = 0; i < ch[b].count; i++) {
                rec_off[(size_t)(base[b] + i)] = p;
                p += 4 + (int64_t)bgzfdev::ld32(ubuf.data() + p);
            }
        }
        bgzfdev::Columns sets[2];
        for (int s = 0; s < 2; s++) {
            Set& w = p_win[s];
            w.start.resize((size_t)n); w.end.resize((size_t)n); w.chrom.resize((size_t)n); w.mapq.resize((size_t)n); w.flag.resize((size_t)n);
            sets[s] = bgzfdev::Columns{w.start.data(), w.end.data(), w.chrom.data(), w.mapq.data(), w.flag.data(), nullptr, nullptr};
        }
        const bgzfdev::ParseCtx pc = r.host_parse_ctx(qual);
        uint64_t first_err = ~uint64_t(0);
        for (int64_t i = 0; i + 1 < n; i++) {   // bam_parse_pairs_kernel: one CUDA thread per adjacent pair
            const int e = bgzfdev::parse_adjacent_pair(ubuf.data(), rec_off.data(), i, g0, pc, sets);
            if (e) first_err = std::min(first_err, ((uint64_t)i << 8) | (uint64_t)e);
        }
        *err = 0;
        if (first_err != ~uint64_t(0)) {
            *err = (int)(first_err & 0xFF);
            *err_rec = (int64_t)(first_err >> 8);
        }
        return 0;
    }
    int deliver_pairs(int64_t pairs0, int64_t pairs1) {
        for (int s = 0; s < 2; s++) {
            const size_t n = 2 * (size_t)(s ? pairs1 : pairs0);
            Set &w = p_win[s], &o = p_out[s];
            o.start.insert(o.start.end(), w.start.begin(), w.start.begin() + n);
            o.end.insert(o.end.end(), w.end.begin(), w.end.begin() + n);
            o.chrom.insert(o.chrom.end(), w.chrom.begin(), w.chrom.begin() + n);
            o.mapq.insert(o.mapq.end(), w.mapq.begin(), w.mapq.begin() + n);
            o.flag.insert(o.flag.end(), w.flag.begin(), w.flag.begin() + n);
        }
        return 0;
    }
    int fetch(int64_t at, uint8_t* dst, size_t n) {
        memcpy(dst, ubuf.data() + at, n);
        return 0;
    }
    int deliver(int64_t n, int mode) {
        o_start.insert(o_start.end(), c_start.begin(), c_start.begin() + n);
        o_end.insert(o_end.end(), c_end.begin(), c_end.begin() + n);
        o_chrom.insert(o_chrom.end(), c_chrom.begin(), c_chrom.begin() + n);
        o_mapq.insert(o_mapq.end(), c_mapq.begin(), c_mapq.begin() + n);
        o_flag.insert(o_flag.end(), c_flag.begin(), c_flag.begin() + n);
        if (mode == bgzfdev::MODE_SC) {
            o_cell.insert(o_cell.end(), c_cell.begin(), c_cell.begin() + n);
            o_umi.insert(o_umi.end(), c_umi.begin(), c_umi.begin() + n);
        }
        if (mode == bgzfdev::MODE_PE_NAME || mode == bgzfdev::MODE_PE_NAME_RANGE) {     // the device hands these to the pairing
                                                                                        // stage, or holds them (pair_name.cuh)
            o_key_hi.insert(o_key_hi.end(), c_key_hi.begin(), c_key_hi.begin() + n);
            o_key_lo.insert(o_key_lo.end(), c_key_lo.begin(), c_key_lo.begin() + n);
            o_role.insert(o_role.end(), c_role.begin(), c_role.begin() + n);
        }
        return 0;
    }
};

struct Session {
    bamorch::Reader reader;
    HostBackend be;
    std::vector<uint8_t> edge[2];               // first / last record of the last paired-end range
};

}  // namespace

extern "C" {

int bgzfdev_open(const char* path, void** out) {
    Session* s = new Session();
    int rc = s->reader.open_path(path);
    if (rc) {
        delete s;
        return rc;
    }
    *out = s;
    return 0;
}
void bgzfdev_close(void* h) { delete (Session*)h; }
const char* bgzfdev_error(void* h) { return ((Session*)h)->reader.err.c_str(); }
int bgzfdev_n_references(void* h) { return (int)((Session*)h)->reader.refs.size(); }
const char* bgzfdev_reference_name(void* h, int i) { return ((Session*)h)->reader.refs[(size_t)i].c_str(); }
int bgzfdev_set_chrom_map(void* h, const uint16_t* b, const uint16_t* s, int32_t n, int32_t n_index) {
    return ((Session*)h)->reader.set_chrom_map(b, s, n, n_index);
}
int bgzfdev_set_whitelist(void* h, const char* bytes, const int64_t* off, int32_t n) { return ((Session*)h)->reader.set_whitelist(bytes, off, n); }
void bgzfdev_force_decline(void* h, int every) { ((Session*)h)->be.force_decline_every = every; }
int bgzfdev_declined(void* h) { return ((Session*)h)->be.n_inflate_declined; }

int bgzfdev_decode(void* h, int mode, int qual, int window_blocks, int64_t* n_records) {
    Session* s = (Session*)h;
    return bamorch::decode_all(s->reader, s->be, mode, qual, window_blocks, n_records);
}

// one byte range of the file (bam_orch.h decode_range); out[6] = {n_records, start_block, start_off, exit_block, exit_off, file size}.
// Mode 4 (MODE_PE_NAME_RANGE): the rows, keys and roles of the range, as bgzfdev_fetch / bgzfdev_fetch_named give them
int bgzfdev_decode_range(void* h, int mode, int qual, int window_blocks, int64_t lo, int64_t hi, int64_t* out) {
    Session* s = (Session*)h;
    bamorch::RangeResult r;
    const int rc = bamorch::decode_range(s->reader, s->be, mode, qual, window_blocks, (uint64_t)lo, (uint64_t)hi, &r);
    out[0] = r.n_records; out[1] = r.start_block; out[2] = r.start_off; out[3] = r.exit_block; out[4] = r.exit_off;
    out[5] = (int64_t)s->reader.file.size;
    s->edge[0].swap(r.first_rec);
    s->edge[1].swap(r.last_rec);
    return rc;
}

// paired-end range: rows of column set `bank` delivered so far, and a copy of them
int64_t bgzfdev_set_rows(void* h, int bank) { return (int64_t)((Session*)h)->be.p_out[bank].start.size(); }
void bgzfdev_fetch_set(void* h, int bank, int32_t* start, int32_t* end, uint16_t* chrom, uint8_t* mapq, uint8_t* flag) {
    const HostBackend::Set& o = ((Session*)h)->be.p_out[bank];
    const size_t n = o.start.size();
    if (!n) return;
    memcpy(start, o.start.data(), n * 4);
    memcpy(end, o.end.data(), n * 4);
    memcpy(chrom, o.chrom.data(), n * 2);
    memcpy(mapq, o.mapq.data(), n);
    memcpy(flag, o.flag.data(), n);
}

// tec_bam_range_record of the host decoder: first (0) / last (1) record of the last paired-end range
int bgzfdev_range_record(void* h, int which, void* buf, int64_t cap, int64_t* len) {
    const std::vector<uint8_t>& e = ((Session*)h)->edge[which];
    *len = (int64_t)e.size();
    if (!buf) return 0;
    if (cap < *len) return bamorch::E_ARG;
    if (!e.empty()) memcpy(buf, e.data(), e.size());
    return 0;
}

// tec_bam_pair_columns of the host decoder
int bgzfdev_pair_columns(void* h, const void* rec1, int64_t n1, const void* rec2, int64_t n2, int qual, int32_t* start, int32_t* end,
                         uint16_t* chrom, uint8_t* mapq, uint8_t* flag) {
    return bamorch::parse_pair(((Session*)h)->reader, (const uint8_t*)rec1, n1, (const uint8_t*)rec2, n2, qual, start, end, chrom, mapq, flag);
}

// copies the delivered columns out (cell / umi only for single cell)
void bgzfdev_fetch(void* h, int32_t* start, int32_t* end, uint16_t* chrom, uint8_t* mapq, uint8_t* flag, uint32_t* cell, uint64_t* umi) {
    HostBackend& b = ((Session*)h)->be;
    const size_t n = b.o_start.size();
    if (!n) return;
    memcpy(start, b.o_start.data(), n * 4);
    memcpy(end, b.o_end.data(), n * 4);
    memcpy(chrom, b.o_chrom.data(), n * 2);
    memcpy(mapq, b.o_mapq.data(), n);
    memcpy(flag, b.o_flag.data(), n);
    if (cell && !b.o_cell.empty()) memcpy(cell, b.o_cell.data(), n * 4);
    if (umi && !b.o_umi.empty()) memcpy(umi, b.o_umi.data(), n * 8);
}

// CRC32 the way the warp computes it (32 lane shares), for holding it against zlib.crc32
uint32_t bgzfdev_crc32_lanes(const void* p, int64_t n) {
    static uint32_t table[256], mats[bgzfdev::CRC_SHIFT_MATS * 32];
    static bool init = false;
    if (!init) {
        bamorch::crc32_tables(table, mats);
        init = true;
    }
    uint8_t dummy = 0;
    uint32_t c = 0;
    for (int lane = 0; lane < 32; lane++) c ^= bgzfdev::crc32_lane_share(p ? (const uint8_t*)p : &dummy, (uint32_t)n, lane, table, mats);
    return c ^ 0xFFFFFFFFu;
}

// the whitelist hash of the decoder (bgzf_dev.h), for holding its numpy restatement against it
uint64_t bgzfdev_wl_hash(const void* p, uint32_t n) { return bgzfdev::wl_hash((const uint8_t*)p, n); }

// the read-name key and the pairing role of bgzf_dev.h, likewise; key[0] = high word, key[1] = low word
void bgzfdev_name_key(const void* p, uint32_t n, uint64_t* key) { bgzfdev::name_key((const uint8_t*)p, n, key[0], key[1]); }
int bgzfdev_name_role(uint32_t flag) { return bgzfdev::name_role(flag); }

// the name keys and roles delivered so far in MODE_PE_NAME (as many as bgzfdev_fetch's rows)
void bgzfdev_fetch_named(void* h, uint64_t* key_hi, uint64_t* key_lo, uint8_t* role) {
    HostBackend& b = ((Session*)h)->be;
    const size_t n = b.o_key_hi.size();
    if (!n) return;
    memcpy(key_hi, b.o_key_hi.data(), n * 8);
    memcpy(key_lo, b.o_key_lo.data(), n * 8);
    memcpy(role, b.o_role.data(), n);
}

// the block inflate alone, for holding it against zlib
int bgzfdev_inflate_raw(const void* in, int64_t n_in, void* out, int64_t n_out) {
    std::vector<uint8_t> scratch(bgzfdev::SCRATCH_STRIDE);
    uint8_t dummy = 0;
    return bgzfdev::inflate_block(in ? (const uint8_t*)in : &dummy, (uint32_t)n_in, out ? (uint8_t*)out : &dummy, (uint32_t)n_out, scratch.data());
}

}  // extern "C"
