// BAM decoding as data-parallel work over BGZF blocks: the per-block routines, written as plain
// C++ that compiles both for the device (included from bamgpu.cuh, one thread per BGZF block) and
// for the host (tools/bgzf_dev_host.cpp runs the very same routines in loops, so that the logic is
// checked against libtecbam on the CPU-only build box, tests/test_bgzf_dev_cpu.py).
//
//   inflate_block     raw DEFLATE of one block into its slot of the window (tables of 16-bit entries
//                     in a per-thread scratch area: they have to fit tens of thousands of times)
//   crc32_block       CRC32 of the inflated bytes (the BGZF trailer is checked on the device)
//   find_start + hop  record boundaries.  Records form a chain (each starts where the previous one
//                     ends) and may straddle blocks, so a block does not know where its first record
//                     starts.  Each block GUESSES it (first offset where two records in a row look
//                     plausible) and hops to the end of the block from there; the host then walks the
//                     per-block (guess, exit) pairs once: a block is used only if its guess equals the
//                     exit of the chain so far.  The result is exactly the true chain or a refusal,
//                     never a wrong split; the guess only makes it parallel.
//   parse_*           one record into the structure-of-arrays columns (same field semantics as
//                     bamdecode.cpp / reads.py; reference te_count.py:76-102, :203-218, :393-438)
#pragma once
#include <stdint.h>
#include <string.h>

#ifdef __CUDACC__
#define BGZF_HD __host__ __device__ __forceinline__
#else
#define BGZF_HD inline
#endif

namespace bgzfdev {

// ------------------------------------------------------------------------------------- inflate
// Decode tables of 16-bit entries, one lookup for codes up to LB / DB bits.  Longer codes (rare
// symbols by construction) are decoded bit by bit from the canonical code description
// (count per length + symbols sorted by code), which needs no second-level tables: the whole
// scratch area is 2.9 KB per block in flight (tens of thousands of blocks stay L2-resident).
constexpr int LB = 9, DB = 8, PB = 7;
constexpr int LIT_SYMS = 288, DIST_SYMS = 32, PRE_SYMS = 20;
constexpr int SCRATCH_U16 = (1 << LB) + LIT_SYMS + 16 + (1 << DB) + DIST_SYMS + 16 + (1 << PB) + PRE_SYMS + 16;
constexpr int SCRATCH_BYTES = SCRATCH_U16 * 2 + 320;                     // tables + code lengths
constexpr int SCRATCH_STRIDE = 2944;
static_assert(SCRATCH_BYTES <= SCRATCH_STRIDE, "scratch stride too small");

// table entry: [3:0] code length (0 = no such code), [5:4] kind, [15:6] value
constexpr uint32_t K_LIT = 0, K_SYM = 1, K_EOB = 2, K_LONG = 3;
constexpr uint32_t NO_VALUE = 0xFFFF;

enum { ST_OK = 0, ST_FORMAT = 1, ST_DECLINED = 2, ST_CRC = 3 };

struct Bits {
    const uint8_t* in;
    uint32_t n, p;
    uint64_t buf;
    int cnt;
};

// At least k <= 32 bits in the buffer?  Refills four bytes at a time while the input allows it (the
// device pays per instruction: one gather of four bytes instead of four turns of a byte loop).
BGZF_HD bool need(Bits& b, int k) {
    if (b.cnt >= k) return true;
    if (b.cnt <= 32 && b.n - b.p >= 4) {
        const uint8_t* q = b.in + b.p;
        const uint32_t w = (uint32_t)q[0] | ((uint32_t)q[1] << 8) | ((uint32_t)q[2] << 16) | ((uint32_t)q[3] << 24);
        b.buf |= (uint64_t)w << b.cnt;
        b.cnt += 32;
        b.p += 4;
        return true;                            // k <= 32 <= cnt
    }
    while (b.cnt < k) {
        if (b.p >= b.n) return false;
        b.buf |= (uint64_t)b.in[b.p++] << b.cnt;
        b.cnt += 8;
    }
    return true;
}
// k <= 32 bits off the buffer
BGZF_HD uint32_t take(Bits& b, int k) {
    const uint32_t lo = (uint32_t)b.buf;
    const uint32_t v = k >= 32 ? lo : lo & ((1u << k) - 1u);
    b.buf >>= k;
    b.cnt -= k;
    return v;
}

BGZF_HD uint32_t reverse_bits(uint32_t code, int len) {
    uint32_t r = 0;
    for (int i = 0; i < len; i++) r |= ((code >> i) & 1u) << (len - 1 - i);
    return r;
}

// alphabet: 0 literal/length, 1 distance, 2 code-length
BGZF_HD uint32_t entry_value(int alphabet, int s) {
    if (alphabet == 0) {
        if (s < 256) return (K_LIT << 4) | ((uint32_t)s << 6);
        if (s == 256) return K_EOB << 4;
        if (s < 286) return (K_SYM << 4) | ((uint32_t)(s - 257) << 6);
        return NO_VALUE;
    }
    if (alphabet == 1) return s < 30 ? ((K_SYM << 4) | ((uint32_t)s << 6)) : NO_VALUE;
    return (K_SYM << 4) | ((uint32_t)s << 6);
}

struct Code {
    uint16_t* table;            // 1 << bits entries
    uint16_t* symbol;           // symbols sorted by (length, value)
    uint16_t* count;            // [16] codes per length
    int bits, alphabet;
};

// ST_OK, or ST_FORMAT for an over-subscribed / not allowed incomplete code
BGZF_HD int build_code(const uint8_t* lens, int n_syms, Code& c, bool allow_incomplete) {
    for (int i = 0; i < 16; i++) c.count[i] = 0;
    for (int s = 0; s < n_syms; s++) c.count[lens[s]]++;
    c.count[0] = 0;
    uint32_t next_code[16], offs[16], code = 0;
    int kraft = 0;
    next_code[0] = 0;
    offs[0] = 0;
    offs[1] = 0;
    for (int l = 1; l <= 15; l++) {
        code = (code + (uint32_t)c.count[l - 1]) << 1;
        next_code[l] = code;
        kraft += (int)c.count[l] << (15 - l);
        if (l < 15) offs[l + 1] = offs[l] + c.count[l];
    }
    if (kraft > (1 << 15)) return ST_FORMAT;
    if (kraft < (1 << 15) && !allow_incomplete) return ST_FORMAT;
    const int primary = 1 << c.bits;
    for (int i = 0; i < primary; i++) c.table[i] = 0;
    for (int s = 0; s < n_syms; s++) {
        const int l = lens[s];
        if (!l) continue;
        c.symbol[offs[l]++] = (uint16_t)s;
        const uint32_t rev = reverse_bits(next_code[l]++, l);
        const uint32_t v = entry_value(c.alphabet, s);
        if (l <= c.bits) {
            if (v == NO_VALUE) continue;
            const uint16_t e = (uint16_t)(v | (uint32_t)l);
            for (uint32_t i = rev; i < (uint32_t)primary; i += 1u << l) c.table[i] = e;
        } else {
            c.table[rev & (uint32_t)(primary - 1)] = (uint16_t)(K_LONG << 4);       // length field 0: not a table hit
        }
    }
    return ST_OK;
}

// One symbol: its table entry (0 = error) after consuming its bits.
BGZF_HD uint32_t decode_sym(Bits& b, const Code& c) {
    need(b, 15);
    const uint32_t e = c.table[(uint32_t)b.buf & ((1u << c.bits) - 1)];
    const int l = (int)(e & 15);
    if (l) {                                    // table hit (the common case): one more test, then the bits go
        if (l > b.cnt) return 0;
        b.buf >>= l;
        b.cnt -= l;
        return e;
    }
    if (e != (K_LONG << 4)) return 0;           // no such code
    // canonical decode, one bit at a time (codes longer than the table index)
    uint32_t code = 0, first = 0, index = 0;
    for (int len = 1; len <= 15; len++) {
        if (b.cnt < 1) return 0;
        code |= take(b, 1);
        const uint32_t cnt = c.count[len];
        if (code < first + cnt) {
            const uint32_t v = entry_value(c.alphabet, c.symbol[index + (code - first)]);
            return v == NO_VALUE ? 0 : (v | 15u);
        }
        index += cnt;
        first = (first + cnt) << 1;
        code <<= 1;
    }
    return 0;
}

// One BGZF block: raw deflate stream in[0, in_n) -> out[0, out_n).  scratch: SCRATCH_BYTES, 2-byte aligned.
BGZF_HD int inflate_block(const uint8_t* in, uint32_t in_n, uint8_t* out, uint32_t out_n, uint8_t* scratch) {
    uint16_t* u = (uint16_t*)scratch;
    Code lit, dist, pre;
    lit.table = u; u += 1 << LB; lit.symbol = u; u += LIT_SYMS; lit.count = u; u += 16; lit.bits = LB; lit.alphabet = 0;
    dist.table = u; u += 1 << DB; dist.symbol = u; u += DIST_SYMS; dist.count = u; u += 16; dist.bits = DB; dist.alphabet = 1;
    pre.table = u; u += 1 << PB; pre.symbol = u; u += PRE_SYMS; pre.count = u; u += 16; pre.bits = PB; pre.alphabet = 2;
    uint8_t* lens = (uint8_t*)u;
    Bits b;
    b.in = in; b.n = in_n; b.p = 0; b.buf = 0; b.cnt = 0;
    uint32_t o = 0;
    for (;;) {
        if (!need(b, 3)) return ST_FORMAT;
        const uint32_t hdr = take(b, 3);
        const uint32_t type = hdr >> 1;
        if (type == 0) {
            take(b, b.cnt & 7);
            b.p -= (uint32_t)(b.cnt >> 3);
            b.buf = 0; b.cnt = 0;
            if (b.n - b.p < 4) return ST_FORMAT;
            const uint32_t len = in[b.p] | ((uint32_t)in[b.p + 1] << 8), nlen = in[b.p + 2] | ((uint32_t)in[b.p + 3] << 8);
            b.p += 4;
            if ((len ^ nlen) != 0xFFFF || b.n - b.p < len || out_n - o < len) return ST_FORMAT;
            for (uint32_t i = 0; i < len; i++) out[o + i] = in[b.p + i];
            o += len;
            b.p += len;
        } else if (type == 1 || type == 2) {
            int rc;
            if (type == 1) {
                int s = 0;
                for (; s < 144; s++) lens[s] = 8;
                for (; s < 256; s++) lens[s] = 9;
                for (; s < 280; s++) lens[s] = 7;
                for (; s < 288; s++) lens[s] = 8;
                rc = build_code(lens, 288, lit, false);
                if (rc) return rc;
                for (s = 0; s < 32; s++) lens[s] = 5;
                rc = build_code(lens, 32, dist, false);
                if (rc) return rc;
            } else {
                if (!need(b, 14)) return ST_FORMAT;
                const int hlit = (int)take(b, 5) + 257, hdist = (int)take(b, 5) + 1, hclen = (int)take(b, 4) + 4;
                if (hlit > 286 || hdist > 30) return ST_FORMAT;
                const uint8_t order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
                for (int i = 0; i < 19; i++) lens[i] = 0;
                for (int i = 0; i < hclen; i++) {
                    if (!need(b, 3)) return ST_FORMAT;
                    lens[order[i]] = (uint8_t)take(b, 3);
                }
                rc = build_code(lens, 19, pre, false);
                if (rc) return rc;
                const int total = hlit + hdist;
                int i = 0;
                while (i < total) {
                    const uint32_t e = decode_sym(b, pre);
                    if (!e) return ST_FORMAT;
                    const int sym = (int)(e >> 6);
                    if (sym < 16) {
                        lens[i++] = (uint8_t)sym;
                        continue;
                    }
                    uint8_t v = 0;
                    int xbits, base;
                    if (sym == 16) {
                        if (!i) return ST_FORMAT;
                        v = lens[i - 1]; xbits = 2; base = 3;
                    } else if (sym == 17) {
                        xbits = 3; base = 3;
                    } else {
                        xbits = 7; base = 11;
                    }
                    if (!need(b, xbits)) return ST_FORMAT;
                    int rep = base + (int)take(b, xbits);
                    if (i + rep > total) return ST_FORMAT;
                    while (rep--) lens[i++] = v;
                }
                if (!lens[256]) return ST_FORMAT;
                // the distance lengths sit behind the literal/length ones: build that code first, then
                // blank the tail so that the literal/length alphabet sees 288 entries
                int n_used = 0, max_len = 0;
                for (int s = 0; s < hdist; s++) {
                    n_used += lens[hlit + s] != 0;
                    if (lens[hlit + s] > max_len) max_len = lens[hlit + s];
                }
                rc = build_code(lens + hlit, hdist, dist, n_used == 0 || (n_used == 1 && max_len == 1));
                if (rc) return rc;
                for (int s = hlit; s < 288; s++) lens[s] = 0;
                rc = build_code(lens, 288, lit, false);
                if (rc) return rc;
            }
            // Symbol loop as a flat state machine: one turn either decodes one symbol or copies up to 8
            // bytes of a pending match.  On the device the 32 lanes of a warp run 32 different
            // streams; with the copy inside the symbol branch every lane would wait for the longest
            // match in the warp on every turn.
            uint32_t copy_left = 0, copy_off = 0, phase = 0;
            uint64_t pat = 0;                   // the period of a match with distance < 8, one byte per lane of the word
            for (;;) {
                if (copy_left) {
                    const uint32_t n = copy_left < 8 ? copy_left : 8;
                    uint8_t* d8 = out + o;
                    if (copy_off >= 8) {        // the loads do not depend on this turn's stores: issue them together
                        const uint8_t* s8 = d8 - copy_off;
                        uint8_t c[8];
                        for (uint32_t j = 0; j < 8; j++) c[j] = j < n ? s8[j] : 0;
                        for (uint32_t j = 0; j < 8; j++)
                            if (j < n) d8[j] = c[j];
                    } else {
                        uint32_t ph = phase;
                        for (uint32_t j = 0; j < 8; j++) {
                            if (j < n) d8[j] = (uint8_t)(pat >> (8 * ph));
                            ph = ph + 1 == copy_off ? 0 : ph + 1;
                        }
                        phase = ph;             // (advanced 8 times; only read again if copy_left stays > 0, i.e. n == 8)
                    }
                    o += n;
                    copy_left -= n;
                    continue;
                }
                const uint32_t e = decode_sym(b, lit);
                if (!e) return ST_FORMAT;
                const uint32_t kind = (e >> 4) & 3;
                if (kind == K_LIT) {
                    if (o >= out_n) return ST_FORMAT;
                    out[o++] = (uint8_t)(e >> 6);
                    continue;
                }
                if (kind == K_EOB) break;
                const int s = (int)(e >> 6);
                int x = s < 8 || s == 28 ? 0 : (s - 4) >> 2;
                uint32_t len = s < 8 ? 3u + (uint32_t)s : s == 28 ? 258u : 3u + ((4u + (uint32_t)(s & 3)) << x);
                if (!need(b, x)) return ST_FORMAT;
                len += take(b, x);
                const uint32_t d = decode_sym(b, dist);
                if (!d) return ST_FORMAT;
                const int ds = (int)(d >> 6);
                x = ds < 4 ? 0 : (ds - 2) >> 1;
                uint32_t off = ds < 4 ? 1u + (uint32_t)ds : 1u + ((2u + (uint32_t)(ds & 1)) << x);
                if (!need(b, x)) return ST_FORMAT;
                off += take(b, x);
                if (off > o || len > out_n - o) return ST_FORMAT;
                copy_left = len;
                copy_off = off;
                if (off < 8) {
                    pat = 0;
                    for (uint32_t j = 0; j < 7; j++)
                        if (j < off) pat |= (uint64_t)out[o - off + j] << (8 * j);
                    phase = 0;
                }
            }
        } else {
            return ST_FORMAT;
        }
        if (hdr & 1) return o == out_n ? ST_OK : ST_FORMAT;
    }
}

BGZF_HD uint32_t crc32_block(const uint8_t* p, uint32_t n, const uint32_t* table) {
    uint32_t c = 0xFFFFFFFFu;
    for (uint32_t i = 0; i < n; i++) c = table[(c ^ p[i]) & 0xFF] ^ (c >> 8);
    return c ^ 0xFFFFFFFFu;
}

// CRC32 of a block by the 32 lanes of a warp: lane i runs the byte loop over its slice
// [i * S, (i + 1) * S) (lane 0 starts from the standard initial state, the others from 0), moves its
// result over the bytes behind its slice with the shift operators, and the XOR of the 32 results,
// complemented, is the CRC32 of the block (CRC is linear over GF(2): crc(A || B) = shift(crc(A), |B|) ^ crc(B)).
// shift_mats[k] = the 32x32 GF(2) matrix "append 2^k zero bytes", k = 0..16 (crc32_shift_matrices, host).
constexpr int CRC_SHIFT_MATS = 17;

BGZF_HD uint32_t crc32_shift(uint32_t crc, uint32_t n_bytes, const uint32_t* shift_mats) {
    for (int k = 0; k < CRC_SHIFT_MATS; k++) {
        if (!((n_bytes >> k) & 1)) continue;
        const uint32_t* m = shift_mats + 32 * k;
        uint32_t r = 0;
        for (int bit = 0; bit < 32; bit++)
            if ((crc >> bit) & 1) r ^= m[bit];
        crc = r;
    }
    return crc;
}

// the share of lane `lane` (0..31); XOR the 32 shares and complement
BGZF_HD uint32_t crc32_lane_share(const uint8_t* p, uint32_t n, int lane, const uint32_t* table, const uint32_t* shift_mats) {
    const uint32_t S = (n + 31) / 32;
    const uint32_t lo = (uint32_t)lane * S < n ? (uint32_t)lane * S : n, hi = lo + S < n ? lo + S : n;
    uint32_t c = lane == 0 ? 0xFFFFFFFFu : 0u;
    for (uint32_t i = lo; i < hi; i++) c = table[(c ^ p[i]) & 0xFF] ^ (c >> 8);
    return crc32_shift(c, n - hi, shift_mats);
}

// ------------------------------------------------------------------------------------- records
BGZF_HD uint32_t ld32(const uint8_t* p) { return p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24); }
BGZF_HD uint32_t ld16(const uint8_t* p) { return p[0] | ((uint32_t)p[1] << 8); }

constexpr int64_t NO_START = -1;
constexpr uint32_t MAX_BLOCK_SIZE = 1u << 28;

// Does a well-formed looking alignment record start at w[p]?  (w_end = bytes in the window.)  Checks the
// fixed fields, the read name ([!-~]+ and its NUL) and walks the optional fields: they must be
// well-formed and end exactly where block_size says -- as far as the window reaches.  This is only
// the GUESS of the block-parallel split (bam_orch.h verifies the chain exactly); the stricter it
// is, the fewer files are refused.
BGZF_HD bool plausible(const uint8_t* w, int64_t p, int64_t w_end, int32_t n_ref) {
    if (p + 36 > w_end) return false;
    const uint32_t bs = ld32(w + p);
    if (bs < 32 || bs > MAX_BLOCK_SIZE) return false;
    const uint8_t* r = w + p + 4;
    const int32_t ref = (int32_t)ld32(r), pos = (int32_t)ld32(r + 4), nref = (int32_t)ld32(r + 20), npos = (int32_t)ld32(r + 24);
    if (ref < -1 || ref >= n_ref || nref < -1 || nref >= n_ref || pos < -1 || npos < -1) return false;
    const uint32_t l_name = r[8], n_cig = ld16(r + 12);
    const int32_t l_seq = (int32_t)ld32(r + 16);
    if (l_name < 1 || l_seq < 0) return false;
    const uint64_t fixed = 32ull + l_name + 4ull * n_cig + (uint64_t)((l_seq + 1) / 2) + (uint64_t)l_seq;
    if (fixed > bs) return false;
    const int64_t limit = w_end - (p + 4);              // bytes of this record the window holds
    for (uint32_t i = 0; i < l_name && 32 + (int64_t)i < limit; i++) {
        const uint8_t ch = r[32 + i];
        if (i + 1 == l_name ? ch != 0 : (ch < 0x21 || ch > 0x7E)) return false;
    }
    for (uint32_t i = 0; i < n_cig && 32 + (int64_t)l_name + 4 * (int64_t)i + 4 <= limit; i++)
        if ((ld32(r + 32 + l_name + 4 * i) & 15) > 8) return false;         // CIGAR operations are 0..8
    // optional fields: tag, type, value ... up to block_size
    int64_t a = (int64_t)fixed;
    const int64_t end = (int64_t)bs;
    while (a < end) {
        if (a + 3 > limit) return true;                 // the window ends here: consistent so far
        if (a + 3 > end) return false;
        const uint8_t ty = r[a + 2];
        a += 3;
        int64_t adv;
        if (ty == 'A' || ty == 'c' || ty == 'C') adv = 1;
        else if (ty == 's' || ty == 'S') adv = 2;
        else if (ty == 'i' || ty == 'I' || ty == 'f') adv = 4;
        else if (ty == 'Z' || ty == 'H') {
            int64_t z = a;
            while (z < end && z < limit && r[z]) z++;
            if (z >= end) return false;
            if (z >= limit) return true;
            adv = z - a + 1;
        } else if (ty == 'B') {
            if (a + 5 > end) return false;
            if (a + 5 > limit) return true;
            const uint8_t st = r[a];
            int64_t sz;
            if (st == 'c' || st == 'C') sz = 1;
            else if (st == 's' || st == 'S') sz = 2;
            else if (st == 'i' || st == 'I' || st == 'f') sz = 4;
            else return false;
            adv = 5 + sz * (int64_t)ld32(r + a + 1);
        } else return false;
        if (adv > end - a) return false;
        a += adv;
    }
    return true;
}

// First offset in [lo, hi) where a record and the one behind it look plausible (the second test is
// skipped when the window ends before the next record's header).
BGZF_HD int64_t find_start(const uint8_t* w, int64_t lo, int64_t hi, int64_t w_end, int32_t n_ref) {
    for (int64_t p = lo; p < hi; p++) {
        if (!plausible(w, p, w_end, n_ref)) continue;
        const int64_t q = p + 4 + (int64_t)ld32(w + p);
        if (q + 36 > w_end || plausible(w, q, w_end, n_ref)) return p;
    }
    return NO_START;
}

struct Hop {
    int64_t exit;       // where the chain stands once it has left [.., hi): start of the next record
    int64_t last;       // start of the last complete record counted (NO_START if none)
    uint32_t count;     // complete records that start in [start, hi)
    uint32_t bad;       // 1: a block_size below 32 on the way (the chain is broken or the guess was wrong)
};

// Hops from `start` over the records that start before hi.  A record that does not end inside the
// window is not counted: the chain stops in front of it (it is carried into the next window).
BGZF_HD Hop hop(const uint8_t* w, int64_t start, int64_t hi, int64_t w_end) {
    Hop h;
    h.exit = start; h.last = NO_START; h.count = 0; h.bad = 0;
    int64_t p = start;
    while (p < hi) {
        if (p + 4 > w_end) break;
        const uint32_t bs = ld32(w + p);
        if (bs < 32 || bs > MAX_BLOCK_SIZE) { h.bad = 1; break; }
        if (p + 4 + (int64_t)bs > w_end) break;
        h.last = p;
        h.count++;
        p += 4 + (int64_t)bs;
    }
    h.exit = p;
    return h;
}

// ---- field decoding (bamdecode.cpp parse_core / find_tags / encode_umi / mate_names_match)
constexpr int F_UNMAPPED = 1, F_DUP = 2, F_QCFAIL = 4, F_REVERSE = 8, F_NAME_MISMATCH = 16;
constexpr uint32_t CHROM_INVALID = 0xFFFF, CHROM_SC_SKIP = 0xFFFE, CHROM_SC_BAD = 0xFFFD, CELL_INVALID = 0xFFFFFFFFu;
enum { E_NONE = 0, E_FORMAT = 2, E_NO_BARCODE_TAG = 10, E_NO_UMI_TAG = 11, E_UMI = 12, E_END_NONE = 13, E_CHROM_NAME = 14, E_REF_NONE = 15 };

struct Rec {
    int32_t ref_id, pos, end;
    uint32_t l_name;            // without the NUL
    const uint8_t *name, *aux, *aux_end;
    uint8_t mapq, fbits;
    uint16_t flag;              // the SAM flag
    bool has_end, ok;
};

BGZF_HD Rec parse_core(const uint8_t* p, uint32_t n) {      // p behind block_size, n = block_size
    Rec c;
    c.ref_id = (int32_t)ld32(p);
    c.pos = (int32_t)ld32(p + 4);
    const uint32_t l_name = p[8], n_cig = ld16(p + 12), flag = ld16(p + 14);
    c.mapq = p[9];
    c.flag = (uint16_t)flag;
    const int64_t l_seq = (int32_t)ld32(p + 16);
    c.fbits = (uint8_t)(((flag >> 2) & 1) * F_UNMAPPED | ((flag >> 10) & 1) * F_DUP | ((flag >> 9) & 1) * F_QCFAIL | ((flag >> 4) & 1) * F_REVERSE);
    const uint64_t o = 32ull + l_name + 4ull * n_cig;
    c.ok = l_seq >= 0 && l_name >= 1 && o + (uint64_t)((l_seq + 1) / 2) + (uint64_t)l_seq <= n;
    c.end = -1;
    c.has_end = false;
    c.name = p + 32; c.aux = c.aux_end = p; c.l_name = 0;
    if (!c.ok) return c;
    uint32_t k = 0;
    while (k < l_name - 1 && c.name[k]) k++;
    c.l_name = k;
    c.has_end = n_cig && !(flag & 4);
    if (c.has_end) {
        const uint8_t* cg = p + 32 + l_name;
        uint32_t span = 0;
        for (uint32_t i = 0; i < n_cig; i++) {
            const uint32_t v = ld32(cg + 4 * i);
            if ((0x18Du >> (v & 15)) & 1) span += v >> 4;       // M D N = X
        }
        c.end = (int32_t)((uint32_t)c.pos + (span ? span : 1u));   // htslib bam_endpos: pos + 1 when the CIGAR consumes no reference base
    }
    c.aux = p + o + (uint64_t)((l_seq + 1) / 2) + (uint64_t)l_seq;
    c.aux_end = p + n;
    return c;
}

BGZF_HD bool mate_names_match(const Rec& a, const Rec& b) {
    uint32_t la = a.l_name, lb = b.l_name;
    while (la && a.name[la - 1] != '/') la--;
    while (lb && b.name[lb - 1] != '/') lb--;
    la = la ? la - 1 : 0;
    lb = lb ? lb - 1 : 0;
    if (la != lb) return false;
    for (uint32_t i = 0; i < la; i++) {
        const uint8_t x = a.name[i] == '/' ? '_' : a.name[i], y = b.name[i] == '/' ? '_' : b.name[i];
        if (x != y) return false;
    }
    return true;
}

struct Tag {
    const uint8_t* p;
    uint32_t n;
    int kind;                   // 0 absent, 1 string (Z, H, A), 2 other type
};

BGZF_HD bool find_tags(const Rec& c, Tag& cb, Tag& cr, Tag& ub, Tag& ur) {
    cb.kind = cr.kind = ub.kind = ur.kind = 0;
    const uint8_t *p = c.aux, *e = c.aux_end;
    while (p + 3 <= e) {
        const uint8_t t0 = p[0], t1 = p[1], ty = p[2];
        p += 3;
        uint64_t adv;
        if (ty == 'A' || ty == 'c' || ty == 'C') adv = 1;
        else if (ty == 's' || ty == 'S') adv = 2;
        else if (ty == 'i' || ty == 'I' || ty == 'f') adv = 4;
        else if (ty == 'Z' || ty == 'H') {
            const uint8_t* z = p;
            while (z < e && *z) z++;
            if (z >= e) return false;
            adv = (uint64_t)(z - p) + 1;
        } else if (ty == 'B') {
            if (p + 5 > e) return false;
            const uint8_t st = p[0];
            uint64_t sz;
            if (st == 'c' || st == 'C') sz = 1;
            else if (st == 's' || st == 'S') sz = 2;
            else if (st == 'i' || st == 'I' || st == 'f') sz = 4;
            else return false;
            adv = 5 + sz * (uint64_t)ld32(p + 1);
        } else return false;
        if (adv > (uint64_t)(e - p)) return false;
        if ((t0 == 'C' || t0 == 'U') && (t1 == 'B' || t1 == 'R')) {
            Tag v;
            v.p = p;
            v.n = 0;
            if (ty == 'Z' || ty == 'H') { v.n = (uint32_t)(adv - 1); v.kind = 1; }
            else if (ty == 'A') { v.n = 1; v.kind = 1; }
            else v.kind = 2;
            if (t0 == 'C') { if (t1 == 'B') cb = v; else cr = v; }
            else { if (t1 == 'B') ub = v; else ur = v; }
        }
        p += adv;
    }
    return true;
}

BGZF_HD bool encode_umi(const uint8_t* s, uint32_t n, uint64_t& code) {
    if (n > 21) return false;
    uint64_t c = 0;
    for (uint32_t i = 0; i < n; i++) {
        uint64_t v;
        const uint8_t ch = s[i];
        if (ch == 'A') v = 1; else if (ch == 'C') v = 2; else if (ch == 'G') v = 3; else if (ch == 'N') v = 4; else if (ch == 'T') v = 5;
        else return false;
        c = (c << 3) | v;
    }
    code = c << (3 * (21 - n));
    return true;
}

// whitelist: open addressing over (id + 1), verified against the barcode bytes
struct WhitelistView {
    const uint32_t* slot;
    const int64_t* off;
    const uint8_t* bytes;
    uint64_t mask;              // 0: no whitelist
};

BGZF_HD uint64_t wl_hash(const uint8_t* p, uint32_t n) {
    uint64_t h = 0xcbf29ce484222325ull;
    for (uint32_t i = 0; i < n; i++) h = (h ^ p[i]) * 0x100000001b3ull;
    h ^= h >> 29;
    h *= 0xbf58476d1ce4e5b9ull;
    return h ^ (h >> 32);
}

BGZF_HD uint32_t wl_find(const WhitelistView& wl, const uint8_t* p, uint32_t n) {
    if (!wl.mask) return CELL_INVALID;
    uint64_t h = wl_hash(p, n) & wl.mask;
    for (;;) {
        const uint32_t v = wl.slot[h];
        if (!v) return CELL_INVALID;
        const int64_t a = wl.off[v - 1], b = wl.off[v];
        if ((uint32_t)(b - a) == n) {
            uint32_t i = 0;
            while (i < n && wl.bytes[a + i] == p[i]) i++;
            if (i == n) return v - 1;
        }
        h = (h + 1) & wl.mask;
    }
}

// Paired end by read name (MODE_PE_NAME): the 128-bit key of a QNAME, two independent 64-bit hashes of its bytes
// (FNV-1a and a multiply-xorshift hash, each through the splitmix64 finalizer).  Mates compare keys, never bytes: for
// 10^9 distinct names the chance that any two share a key is about n^2 / 2^129 = 1.5e-21.
BGZF_HD uint64_t mix64(uint64_t h) {
    h ^= h >> 30;
    h *= 0xbf58476d1ce4e5b9ull;
    h ^= h >> 27;
    h *= 0x94d049bb133111ebull;
    return h ^ (h >> 31);
}

BGZF_HD void name_key(const uint8_t* p, uint32_t n, uint64_t& hi, uint64_t& lo) {
    uint64_t a = 0xcbf29ce484222325ull, b = 0x9e3779b97f4a7c15ull ^ n;
    for (uint32_t i = 0; i < n; i++) {
        a = (a ^ p[i]) * 0x100000001b3ull;
        b = (b + p[i] + 1) * 0xff51afd7ed558ccdull;
        b ^= b >> 29;
    }
    hi = mix64(a ^ ((uint64_t)n << 56));
    lo = mix64(b);
}

// which side of a pair a record is on: primary (0x100, 0x800 clear), paired (0x1) and exactly one of 0x40 / 0x80
enum { ROLE_EXCLUDED = 0, ROLE_READ1 = 1, ROLE_READ2 = 2 };
BGZF_HD int name_role(uint32_t flag) {
    if (!(flag & 0x1) || (flag & 0x900)) return ROLE_EXCLUDED;
    const uint32_t m = flag & 0xC0;
    return m == 0x40 ? ROLE_READ1 : m == 0x80 ? ROLE_READ2 : ROLE_EXCLUDED;
}

struct Columns {
    int32_t *start, *end;
    uint16_t* chrom;
    uint8_t *mapq, *flag;
    uint32_t* cell;
    uint64_t* umi;
    uint64_t *key_hi, *key_lo;  // MODE_PE_NAME: name_key of the QNAME (0 for excluded records)
    uint8_t* role;              // MODE_PE_NAME: name_role of the SAM flag
};

struct ParseCtx {
    const uint16_t *bulk_ids, *sc_ids;
    int32_t n_ref, n_index, qual;
    WhitelistView wl;
};

// MODE_PE_NAME_RANGE: byte ranges only (bam_orch.h decode_range): records are parsed as MODE_PE_NAME and the rows are
// held for the exchange by name owner instead of being paired (pair_name.cuh)
enum { MODE_SE = 0, MODE_PE = 1, MODE_SC = 2, MODE_PE_NAME = 3, MODE_PE_NAME_RANGE = 4 };

// Record at window offset p (complete by construction) into row k.  For MODE_PE the caller passes
// the FIRST mate and p2 = offset of the second; rows k and k + 1 are written.  MODE_PE_NAME writes the
// one-record row of MODE_SE plus the name key and the role; the pairing stage (pair_name.cuh) makes the
// pairs.  Returns E_*.
BGZF_HD int parse_record(const uint8_t* w, int64_t p, int64_t p2, int mode, const ParseCtx& pc, const Columns& o, int64_t k) {
    const Rec c = parse_core(w + p + 4, ld32(w + p));
    if (!c.ok) return E_FORMAT;
    const bool has_ref = c.ref_id >= 0 && c.ref_id < pc.n_ref;
    if (mode == MODE_PE) {
        const Rec c2 = parse_core(w + p2 + 4, ld32(w + p2));
        if (!c2.ok) return E_FORMAT;
        uint8_t f1 = c.fbits;
        const bool rejected = ((c.fbits | c2.fbits) & (F_UNMAPPED | F_DUP | F_QCFAIL)) || (int)c.mapq < pc.qual;
        if (!rejected && !mate_names_match(c, c2)) f1 |= F_NAME_MISMATCH;
        o.start[k] = c.pos; o.end[k] = c.end; o.chrom[k] = has_ref ? pc.bulk_ids[c.ref_id] : (uint16_t)CHROM_INVALID;
        o.mapq[k] = c.mapq; o.flag[k] = f1;
        const bool has_ref2 = c2.ref_id >= 0 && c2.ref_id < pc.n_ref;
        o.start[k + 1] = c2.pos; o.end[k + 1] = c2.end; o.chrom[k + 1] = has_ref2 ? pc.bulk_ids[c2.ref_id] : (uint16_t)CHROM_INVALID;
        o.mapq[k + 1] = c2.mapq; o.flag[k + 1] = c2.fbits;
        return E_NONE;
    }
    if (mode == MODE_PE_NAME) {
        o.start[k] = c.pos; o.end[k] = c.end; o.chrom[k] = has_ref ? pc.bulk_ids[c.ref_id] : (uint16_t)CHROM_INVALID;
        o.mapq[k] = c.mapq; o.flag[k] = c.fbits;
        const int role = name_role(c.flag);
        uint64_t hi = 0, lo = 0;
        if (role != ROLE_EXCLUDED) name_key(c.name, c.l_name, hi, lo);
        o.key_hi[k] = hi; o.key_lo[k] = lo; o.role[k] = (uint8_t)role;
        return E_NONE;
    }
    if (mode == MODE_SE) {
        const uint16_t ch = has_ref ? pc.bulk_ids[c.ref_id] : (uint16_t)CHROM_INVALID;
        o.start[k] = c.pos; o.end[k] = c.end; o.chrom[k] = ch; o.mapq[k] = c.mapq; o.flag[k] = c.fbits;
        if (!c.has_end && !(c.fbits & (F_UNMAPPED | F_DUP | F_QCFAIL)) && (int)c.mapq >= pc.qual && (int32_t)ch < pc.n_index) return E_END_NONE;
        return E_NONE;
    }
    o.mapq[k] = c.mapq; o.flag[k] = c.fbits;
    o.start[k] = -1; o.end[k] = -1; o.chrom[k] = (uint16_t)CHROM_INVALID; o.cell[k] = CELL_INVALID; o.umi[k] = 0;
    if ((c.fbits & (F_UNMAPPED | F_DUP | F_QCFAIL)) || (int)c.mapq < pc.qual) return E_NONE;
    Tag cb, cr, ub, ur;
    if (!find_tags(c, cb, cr, ub, ur)) return E_FORMAT;
    const Tag& bc = cb.kind ? cb : cr;
    if (!bc.kind) return E_NO_BARCODE_TAG;
    const uint32_t cid = bc.kind == 1 ? wl_find(pc.wl, bc.p, bc.n) : CELL_INVALID;
    if (cid == CELL_INVALID) return E_NONE;
    const Tag& um = ub.kind ? ub : ur;
    if (!um.kind) return E_NO_UMI_TAG;
    uint64_t code = 0;
    if (um.kind != 1 || !encode_umi(um.p, um.n, code)) return E_UMI;
    if (!has_ref) return E_REF_NONE;
    const uint16_t ch = pc.sc_ids[c.ref_id];
    if (ch == CHROM_SC_BAD) return E_CHROM_NAME;
    if (!c.has_end && ch != CHROM_SC_SKIP) return E_END_NONE;
    o.start[k] = c.pos; o.end[k] = c.end; o.chrom[k] = ch; o.cell[k] = cid; o.umi[k] = code;
    return E_NONE;
}

// Paired end over a byte range whose first record has an unknown global parity: adjacent pair i of a
// window (records at rec_off[i] and rec_off[i + 1]; record 0 of the window has range-local index g0) is
// read1 + read2 if g0 + i has the parity of the range's global offset.  Both candidates are kept: the pair
// goes to column set (g0 + i) & 1 as rows 2 (i >> 1) and 2 (i >> 1) + 1, so each set holds its pairs in
// file order.  Returns E_*.
BGZF_HD int parse_adjacent_pair(const uint8_t* w, const int64_t* rec_off, int64_t i, int64_t g0, const ParseCtx& pc, const Columns* sets) {
    return parse_record(w, rec_off[i], rec_off[i + 1], MODE_PE, pc, sets[(g0 + i) & 1], 2 * (i >> 1));
}

// rows of column set `bank` from the m records of a window that starts at range-local index g0 (m - 1 adjacent pairs)
BGZF_HD int64_t pairs_in_set(int64_t m, int64_t g0, int bank) { return m > 0 ? (m - ((bank - g0) & 1)) / 2 : 0; }

}  // namespace bgzfdev
