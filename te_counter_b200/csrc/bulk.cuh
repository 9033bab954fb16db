// Bulk counting kernels: filter (+ mate merge), point overlap, type rule, tally.
//
// Reference semantics (te_counter, te_count/te_count.py):
//   filter SE :203-218, filter + mate merge PE :76-102, candidate buckets :106-116 / :222-231,
//   point tests :118-126 / :233-241, type rule + tally :128-149 / :243-261.
//
// Closed forms used here (SURVEY.md 8a-5, 8a-6), with bs = bucket size:
//   point A  loc1 in [L, R-1]   <=>  x1 = loc1     stabs the half-open interval [L, R)
//   point B  loc2 in [L+1, R]   <=>  x2 = loc2 - 1 stabs [L, R)
//   candidate(f) <=> L//bs <= b1 <= R//bs  or  L//bs <= b2 <= R//bs,
//                    b1 = (loc1-1)//bs, b2 = (loc2+1)//bs   (the two buckets of :106-108)
//   it can only be false when loc1 == L (A) or loc2 == R (B), so the divisions are off the
//   common path.
#pragma once
#include "common.cuh"
#include "stab_build.h"

// number of features of chromosome [lo, lo+n) with L <= x, through the coarse directory
__device__ __forceinline__ int upper_bound_L(const IndexView& iv, int c, int64_t lo, int n, int x) {
    if (x < 0) return 0;                              // L >= 0 is enforced at upload
    const int64_t doff = iv.dir_off[c];
    const int ncell = (int)(iv.dir_off[c + 1] - doff);
    const int k = x >> iv.shift;
    if (k >= ncell - 1) return n;
    u32 a = __ldg(iv.dir + doff + k), b = __ldg(iv.dir + doff + k + 1);
    while (a < b) {
        u32 mid = (a + b) >> 1;
        if (__ldg(iv.L + lo + mid) <= x) a = mid + 1; else b = mid;
    }
    return (int)a;
}

__device__ __forceinline__ bool bulk_candidate(int Lk, int Rk, int loc1, int loc2, int b1, int b2,
                                               bool hitA, bool hitB, int bs) {
    if ((hitA && loc1 != Lk) || (hitB && loc2 != Rk)) return true;
    const int lb = Lk / bs, rb = Rk / bs;
    return (lb <= b1 && b1 <= rb) || (lb <= b2 && b2 <= rb);
}

// Calls f(feature_index) exactly once for every feature the reference appends to `result`
// (te_count.py:118-126); returns false as soon as f returns false.
template <class F>
__device__ __forceinline__ bool bulk_for_each_hit(const IndexView& iv, int c, int loc1, int loc2, F f) {
    const int64_t lo = iv.chrom_off[c];
    const int n = (int)(iv.chrom_off[c + 1] - lo);
    const int bs = iv.bs;
    const int b1 = floordiv(loc1 - 1, bs), b2 = floordiv(loc2 + 1, bs);
    {   // point A
        const int x = loc1;
        for (int k = upper_bound_L(iv, c, lo, n, x) - 1; k >= 0; --k) {
            if (__ldg(iv.pmaxR + lo + k) <= x) break;
            const int Rk = __ldg(iv.R + lo + k);
            if (Rk > x) {
                const int Lk = __ldg(iv.L + lo + k);
                const bool hitB = (Lk < loc2 && loc2 <= Rk);
                if (bulk_candidate(Lk, Rk, loc1, loc2, b1, b2, true, hitB, bs))
                    if (!f(lo + k)) return false;
            }
        }
    }
    {   // point B
        const int x = loc2 - 1;
        for (int k = upper_bound_L(iv, c, lo, n, x) - 1; k >= 0; --k) {
            if (__ldg(iv.pmaxR + lo + k) <= x) break;
            const int Rk = __ldg(iv.R + lo + k);
            if (Rk > x) {
                const int Lk = __ldg(iv.L + lo + k);
                if (Lk <= loc1 && loc1 < Rk) continue;          // enumerated under point A
                if (bulk_candidate(Lk, Rk, loc1, loc2, b1, b2, false, true, bs))
                    if (!f(lo + k)) return false;
            }
        }
    }
    return true;
}

#define BULK_MAX_DISTINCT 12
#define BULK_LOCI_REG 8          // hit rows a LOCI unit keeps in registers; more are found by a second walk

struct BulkStatsLocal {
    u32 units, assigned, lowq, badchrom, qcfail, crash_enh, crash_name;
};

// One thread per unit (record in SE, pair in PE), grid-stride.  Per-feature counters are int64 in
// global memory (L2-resident, 8 B x n_ensg); statistics are reduced per warp, then per CTA.
// LOCI (tec_set_option "bulk_loci", an extension outside the parity claim): a counted unit also adds 1 to every index
// row it hits, in the u64 row counters that follow the statistics (counts + n_ensg + TEC_BULK_NSTATS, upload order).
template <bool PAIRED, bool LOCI>
__global__ void __launch_bounds__(256)
bulk_count_kernel(IndexView iv, int64_t n_units, int qual, int strand_mode,
                  const int32_t* __restrict__ start, const int32_t* __restrict__ end,
                  const uint16_t* __restrict__ chrom, const uint8_t* __restrict__ mapq,
                  const uint8_t* __restrict__ flag, u64* __restrict__ counts, u64* __restrict__ stats) {
    // strand_mode != 0 is the opt-in extension of tec_set_option("bulk_strand") -- the reference raises
    // NotImplementedError for bulk --strand (te_count.py:58-59 / :183-184), so this is NOT part of the parity claim:
    // a feature on '+' or '-' is a candidate only for units whose first record lies on that strand (flag 0x10 = '-');
    // features with any other strand value stay candidates for both.  Restated in oracle/te_oracle_ext.py.
    BulkStatsLocal st = {0, 0, 0, 0, 0, 0, 0};
    u64* const loci = counts + iv.n_ensg + TEC_BULK_NSTATS;
    const u32 reject = TEC_F_UNMAPPED | TEC_F_DUP | TEC_F_QCFAIL;
    for (int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; u < n_units;
         u += (int64_t)gridDim.x * blockDim.x) {
        st.units++;
        int c, loc1, loc2;
        u32 us = 0;                                   // strand of the unit's first record (extension only)
        auto other_strand = [&](u32 w) { const u32 fs = info_strand(w); return strand_mode != 0 && fs <= 1u && fs != us; };
        if (PAIRED) {
            const uchar2 f2 = *reinterpret_cast<const uchar2*>(flag + 2 * u);
            if ((f2.x & reject) || (f2.y & reject)) { st.qcfail++; continue; }       // :81-86
            if ((int)mapq[2 * u] < qual) { st.lowq++; continue; }                      // :88 read1 only
            if (f2.x & TEC_F_NAME_MISMATCH) { st.crash_name++; continue; }             // :92-94
            us = (f2.x & TEC_F_REVERSE) ? 1u : 0u;
            c = chrom[2 * u];                                                          // :96 read1 only
            const int2 s2 = *reinterpret_cast<const int2*>(start + 2 * u);
            loc1 = s2.x;                                                               // :97
            loc2 = s2.y;                                                               // :98 mate START
        } else {
            if (flag[u] & reject) { st.qcfail++; continue; }                           // :204
            if ((int)mapq[u] < qual) { st.lowq++; continue; }                          // :208
            us = (flag[u] & TEC_F_REVERSE) ? 1u : 0u;
            c = chrom[u];
            loc1 = start[u];                                                           // :213
            loc2 = end[u];                                                             // :214
        }
        if (!chrom_in_index(iv, c)) { st.badchrom++; continue; }                       // :100 / :216

        u32 typemask = 0, nd = 0, dist[BULK_MAX_DISTINCT];
        bool overflow = false;
        u32 nrow = 0;
        int64_t rows[LOCI ? BULK_LOCI_REG : 1];
        bulk_for_each_hit(iv, c, loc1, loc2, [&](int64_t fi) {
            const u32 w = __ldg(iv.info + fi);
            if (other_strand(w)) return true;
            typemask |= 1u << info_type(w);
            const u32 e = info_ensg(w);
            bool found = false;
            for (u32 i = 0; i < nd; ++i) found |= (dist[i] == e);
            if (!found) {
                if (nd < BULK_MAX_DISTINCT) dist[nd++] = e; else overflow = true;
            }
            if (LOCI) {
#pragma unroll
                for (int j = 0; j < BULK_LOCI_REG; ++j) if ((u32)j == nrow) rows[j] = fi;     // unrolled: stays in registers
                ++nrow;
            }
            return true;
        });
        if (!typemask) continue;                                                       // :128 no result
        st.assigned++;                                                                 // :149
        const u32 counted = (1u << TEC_T_GENE) | (1u << TEC_T_TE) | (1u << TEC_T_SNRNA);
        if (!(typemask & counted)) {
            if (typemask & (1u << TEC_T_ENHANCER)) st.crash_enh++;                     // :145-147
            continue;
        }
        if (LOCI) {
            // a counted unit: +1 for every row it hits (bulk_for_each_hit lists each row once)
            if (nrow <= BULK_LOCI_REG) {
#pragma unroll
                for (int j = 0; j < BULK_LOCI_REG; ++j) if ((u32)j < nrow) atomicAdd(loci + rows[j], 1ULL);
            } else {
                bulk_for_each_hit(iv, c, loc1, loc2, [&](int64_t fi) {
                    if (!other_strand(__ldg(iv.info + fi))) atomicAdd(loci + fi, 1ULL);
                    return true;
                });
            }
        }
        if (!overflow) {
            for (u32 i = 0; i < nd; ++i) atomicAdd(counts + dist[i], 1ULL);            // one per distinct ensg
        } else {
            // more distinct ensg than the register list holds: count a hit iff no earlier hit
            // (in enumeration order) carries the same ensg -- O(h^2) re-walks, no storage
            int h = 0;
            bulk_for_each_hit(iv, c, loc1, loc2, [&](int64_t fi) {
                const u32 wi = __ldg(iv.info + fi);
                if (other_strand(wi)) { ++h; return true; }
                const u32 e = info_ensg(wi);
                int j = 0;
                bool dup = false;
                bulk_for_each_hit(iv, c, loc1, loc2, [&](int64_t fj) {
                    if (j++ >= h) return false;
                    const u32 wj = __ldg(iv.info + fj);
                    if (!other_strand(wj) && info_ensg(wj) == e) { dup = true; return false; }
                    return true;
                });
                if (!dup) atomicAdd(counts + e, 1ULL);
                ++h;
                return true;
            });
        }
    }
    // statistics: warp shuffle -> shared -> one global atomic per CTA per counter
    __shared__ u64 s_stats[TEC_BULK_NSTATS];
    if (threadIdx.x < TEC_BULK_NSTATS) s_stats[threadIdx.x] = 0;
    __syncthreads();
    u64 v[7] = {st.units, st.assigned, st.lowq, st.badchrom, st.qcfail, st.crash_enh, st.crash_name};
#pragma unroll
    for (int i = 0; i < 7; ++i) {
        const u64 s = warp_sum(v[i]);
        if ((threadIdx.x & 31) == 0 && s) atomicAdd(&s_stats[i], s);
    }
    __syncthreads();
    if (threadIdx.x < 7 && s_stats[threadIdx.x]) atomicAdd(stats + threadIdx.x, s_stats[threadIdx.x]);
}

// =====================================================================================================
// Fast path: cell table (stab_build.h) + shared-memory counters for the hottest ensg.
//
// Per unit: 16 B (PE; `end` is never read) / 12 B (SE) of streamed records (evict-first, no L1
// allocate), ONE 32-byte sector of the L2-resident cell table fetched with a single 256-bit load
// (two when the unit's points fall in different cells, one more when a crowded cell links to an
// overflow sector the point can reach), and one shared-memory or global atomic per distinct ensg.
// Units whose candidate test can fail (loc1 % bs == 0 or (loc2 + 1) % bs == 0, see the header of
// this file) or that hit more than STAB_MAXD distinct ensg are only flagged here (one ballot word per
// warp) and counted by bulk_slow_kernel with the exact search above; both are rare.
// =====================================================================================================
struct StabView {
    const u32* sectors;          // 8 words per sector, 32-byte aligned
    const uint2* cells;          // per chromosome: {first sector, number of cells}
    const u32* ovf_base;         // per 256 primary sectors: first overflow sector
    const uint8_t* slot_type;    // n_slots
    int shift;
    int all_counted;
};

#define STAB_MAXD 4
#define TEC_HOT_SLOTS 4096        // shared-memory counters when not every ensg fits (and in the slow kernel)
#define BULK_QCAP 64             // deferred-unit ring per warp (entries)
#define R_NONE 0x7FFFu           // "no point in this sector": fails the e >= r test of every entry

struct Sector { u32 w[8]; };

__device__ __forceinline__ Sector ld_sector(const u32* sectors, u32 idx) {
    Sector r;
    const u32* p = sectors + (size_t)idx * 8;
    asm volatile("ld.global.nc.L1::no_allocate.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r.w[0]), "=r"(r.w[1]), "=r"(r.w[2]), "=r"(r.w[3]), "=r"(r.w[4]), "=r"(r.w[5]), "=r"(r.w[6]), "=r"(r.w[7])
                 : "l"(p));
    return r;
}

// streamed record loads: read once, keep them out of L1 and first in line for L2 eviction
__device__ __forceinline__ u64 make_evict_first_policy() {
    u64 pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ int2 ld_stream_int2(const int32_t* p, u64 pol) {
    int2 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v2.s32 {%0,%1}, [%2], %3;" : "=r"(r.x), "=r"(r.y) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ int ld_stream_int(const int32_t* p, u64 pol) {
    int r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.s32 %0, [%1], %2;" : "=r"(r) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ u32 ld_stream_u32(const void* p, u64 pol) {
    u32 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.u32 %0, [%1], %2;" : "=r"(r) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ u32 ld_stream_u16(const void* p, u64 pol) {
    unsigned short r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.u16 %0, [%1], %2;" : "=h"(r) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ u32 ld_stream_u8(const uint8_t* p, u64 pol) {
    u32 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.u8 %0, [%1], %2;" : "=r"(r) : "l"(p), "l"(pol));
    return r;
}

// A point r (cell-relative, < 2^11, or R_NONE) prepared for the 16-bit-lane test of stab_build.h:
// bit 15 of each lane of (xg - w_s) says r >= s, of (w_e + kg) says e >= r.
struct PointK { u32 xg, kg; };
__device__ __forceinline__ PointK make_point(u32 r) {
    const u32 rr = r * 0x10001u;
    PointK p;
    p.xg = rr + 0x80008000u;
    p.kg = 0x80008000u - rr;
    return p;
}
// hit mask of a sector for points a or b.  Bit positions: entry 0 -> 15, 1 -> 31, 2 -> 14, 3 -> 30, 4 -> 13.
#define HB0 (1u << 15)
#define HB1 (1u << 31)
#define HB2 (1u << 14)
#define HB3 (1u << 30)
#define HB4 (1u << 13)
__device__ __forceinline__ u32 sector_hits(const Sector& s, const PointK a, const PointK b) {
    const u32 a0 = ((a.xg - s.w[0]) & (s.w[3] + a.kg)) | ((b.xg - s.w[0]) & (s.w[3] + b.kg));
    const u32 a1 = ((a.xg - s.w[1]) & (s.w[4] + a.kg)) | ((b.xg - s.w[1]) & (s.w[4] + b.kg));
    const u32 a2 = ((a.xg - s.w[2]) & (s.w[5] + a.kg)) | ((b.xg - s.w[2]) & (s.w[5] + b.kg));
    return (a0 & 0x80008000u) | ((a1 & 0x80008000u) >> 1) | ((a2 & 0x8000u) >> 2);
}
template <int I>
__device__ __forceinline__ u32 sector_slot_c(const Sector& s) {
    return I == 0 ? (s.w[6] & 0xFFFFu) : I == 1 ? (s.w[6] >> 16) : I == 2 ? (s.w[7] & 0xFFFFu) : I == 3 ? (s.w[7] >> 16) : (s.w[5] >> 16);
}
__device__ __forceinline__ bool sector_more(const Sector& s) { return (s.w[2] >> 16) & 1u; }
// two hit entries that both have a twin (same ensg elsewhere in the sector): the ensg may be hit twice
__device__ __forceinline__ bool sector_twin_hit(const Sector& s, u32 hit) {
    const u32 m5 = ((hit >> 13) & 7u) | ((hit >> 27) & 0x18u);          // e4, e2, e0, e3, e1
    return __popc(m5 & (s.w[2] >> 17)) >= 2;
}
__device__ __forceinline__ u32 sector_link(const Sector& s) { return s.w[2] >> 22; }
__device__ __forceinline__ u32 sector_last_s(const Sector& s) { return s.w[2] & 0xFFFFu; }

// x % 10000 == 0 (as unsigned; a negative position never hits anything in either path, so its
// answer does not matter): 10000 = 2^4 * 625, and n % (2^k * d) == 0  <=>
// rotr(n * d^-1 mod 2^32, k) <= (2^32 - 1) / (2^k * d)
__device__ __forceinline__ bool mult_of_10000(int x) {
    const u32 t = (u32)x * 0x3AFB7E91u;
    return __funnelshift_r(t, t, 4) <= 0xFFFFFFFFu / 10000u;
}

struct BulkRec {
    u32 fl, q;
    int c, loc1, loc2;
};

template <bool PAIRED>
__device__ __forceinline__ BulkRec bulk_load(u32 u, const int32_t* __restrict__ start, const int32_t* __restrict__ end,
                                             const uint16_t* __restrict__ chrom, const uint8_t* __restrict__ mapq,
                                             const uint8_t* __restrict__ flag, u64 pol) {
    BulkRec r;
    if (PAIRED) {
        r.fl = ld_stream_u16(flag + 2 * (size_t)u, pol);            // both mates' flag bytes
        r.q = ld_stream_u16(mapq + 2 * (size_t)u, pol) & 0xFFu;     // read1 only (:88)
        r.c = (int)(ld_stream_u32(chrom + 2 * (size_t)u, pol) & 0xFFFFu);   // read1 only (:96)
        const int2 s2 = ld_stream_int2(start + 2 * (size_t)u, pol);
        r.loc1 = s2.x;                                              // :97
        r.loc2 = s2.y;                                              // :98 mate START
    } else {
        r.fl = ld_stream_u8(flag + u, pol);
        r.q = ld_stream_u8(mapq + u, pol);
        r.c = (int)ld_stream_u16(chrom + u, pol);
        r.loc1 = ld_stream_int(start + u, pol);                     // :213
        r.loc2 = ld_stream_int(end + u, pol);                       // :214
    }
    return r;
}

// a unit that needs a second sector (its points straddle two cells, or it can reach the overflow
// sector), or that hit two entries of a sector holding one ensg twice: parked in the warp's ring
// and looked up 32 at a time by bulk_deferred(), so the common path stays branch-light
struct QEnt {
    u32 secA;       // sector | kind << 24   (kind 0: cell A only, 1: a second cell B)
    u32 secB;
    u32 pa;         // points in A:  ra | rb << 16   (R_NONE = none)
    u32 pb;         // points in B
};

template <int WARPS>
struct BulkShared {
    u64 stats[TEC_BULK_NSTATS];
    QEnt q[WARPS][BULK_QCAP];
    u32 qu[WARPS][BULK_QCAP];            // unit index inside the launch (for the slow flag)
};

// +1 for entry I of the sector when its hit bit is set.  Counters of the first n_hot slots live in
// shared memory; ALLHOT: every ensg does, so the global path disappears from the kernel.
template <int I, bool ALLHOT>
__device__ __forceinline__ void bump_entry(u32 hit, const Sector& s, u32 hot_addr, u32 n_hot, u64* __restrict__ counts, u32 one) {
    const u32 slot = sector_slot_c<I>(s);
    const u32 bit = I == 0 ? HB0 : I == 1 ? HB1 : I == 2 ? HB2 : I == 3 ? HB3 : HB4;
    if (ALLHOT) {
        // unconditional reduction: entries that were not hit add to a per-lane scratch word behind the
        // counters, so there is no branch (ptxas never predicates a shared-memory reduction)
        const u32 addr = (hit & bit) ? (hot_addr + slot * 4u) : (hot_addr + (n_hot + (threadIdx.x & 31)) * 4u);
        asm volatile("red.shared.add.u32 [%0], %1;" :: "r"(addr), "r"(one) : "memory");
    } else {
        asm volatile("{\n\t.reg .pred p, q, r;\n\t.reg .b32 t;\n\t"
                     "and.b32 t, %0, %1;\n\t"
                     "setp.ne.u32 p, t, 0;\n\t"
                     "setp.lt.u32 q, %2, %3;\n\t"
                     "and.pred r, p, q;\n\t"
                     "@r red.shared.add.u32 [%4], %6;\n\t"
                     "not.pred q, q;\n\t"
                     "and.pred r, p, q;\n\t"
                     "@r red.global.add.u64 [%5], %7;\n\t}"
                     :: "r"(hit), "r"(bit), "r"(slot), "r"(n_hot), "r"(hot_addr + slot * 4u), "l"(counts + slot),
                        "r"(one), "l"((u64)one) : "memory");
    }
}
template <bool ALLHOT>
__device__ __forceinline__ void bump_sector(u32 hit, const Sector& s, u32 hot_addr, u32 n_hot, u64* __restrict__ counts, u32 one) {
    bump_entry<0, ALLHOT>(hit, s, hot_addr, n_hot, counts, one);
    bump_entry<1, ALLHOT>(hit, s, hot_addr, n_hot, counts, one);
    bump_entry<2, ALLHOT>(hit, s, hot_addr, n_hot, counts, one);
    bump_entry<3, ALLHOT>(hit, s, hot_addr, n_hot, counts, one);
    bump_entry<4, ALLHOT>(hit, s, hot_addr, n_hot, counts, one);
}

// slow list: word 0 = number of flagged units, then their indices (capacity = units of the launch).
// Called by a converged warp: one atomic per warp.
__device__ __forceinline__ void flag_slow_warp(u32* __restrict__ slow_list, bool slow, u32 u, u32 lt_mask) {
    const u32 sm = __ballot_sync(0xFFFFFFFFu, slow);
    if (!sm) return;
    u32 base = 0;
    if ((threadIdx.x & 31) == 0) base = atomicAdd(slow_list, (u32)__popc(sm));
    base = __shfl_sync(0xFFFFFFFFu, base, 0);
    if (slow) slow_list[1 + base + __popc(sm & lt_mask)] = u;
}

// type rule of te_count.py:134-147 over the distinct slots of a unit; returns "count it"
__device__ __forceinline__ bool bulk_type_rule(const StabView& sv, u32 typemask, u64* __restrict__ stats) {
    const u32 counted = (1u << TEC_T_GENE) | (1u << TEC_T_TE) | (1u << TEC_T_SNRNA);
    if (typemask & counted) return true;
    if (typemask & (1u << TEC_T_ENHANCER)) atomicAdd(stats + TEC_BS_CRASH_ENHANCER, 1ULL);       // :145-147
    return false;
}

// B-entry J is dropped from hitB when a hit entry of A carries the same ensg
template <int J>
__device__ __forceinline__ u32 drop_if_in_a(u32 hitA, u32 hitB, const Sector& A, const Sector& B) {
    const u32 w = sector_slot_c<J>(B);
    const bool dup = ((hitA & HB0) && sector_slot_c<0>(A) == w) | ((hitA & HB1) && sector_slot_c<1>(A) == w) |
                     ((hitA & HB2) && sector_slot_c<2>(A) == w) | ((hitA & HB3) && sector_slot_c<3>(A) == w) |
                     ((hitA & HB4) && sector_slot_c<4>(A) == w);
    const u32 bit = J == 0 ? HB0 : J == 1 ? HB1 : J == 2 ? HB2 : J == 3 ? HB3 : HB4;
    return dup ? (hitB & ~bit) : hitB;
}

__device__ __forceinline__ u32 sector_typemask(const StabView& sv, const Sector& s, u32 hit) {
    u32 typemask = 0;
    if (hit & HB0) typemask |= 1u << __ldg(sv.slot_type + sector_slot_c<0>(s));
    if (hit & HB1) typemask |= 1u << __ldg(sv.slot_type + sector_slot_c<1>(s));
    if (hit & HB2) typemask |= 1u << __ldg(sv.slot_type + sector_slot_c<2>(s));
    if (hit & HB3) typemask |= 1u << __ldg(sv.slot_type + sector_slot_c<3>(s));
    if (hit & HB4) typemask |= 1u << __ldg(sv.slot_type + sector_slot_c<4>(s));
    return typemask;
}

__device__ __forceinline__ int points_rmax(u32 p) {
    const u32 ra = p & 0xFFFFu, rb = p >> 16;
    return max(ra == R_NONE ? -1 : (int)ra, rb == R_NONE ? -1 : (int)rb);
}

// A unit that needs exactly two sectors: two cells (kind 1), or a cell and its first overflow sector
// (kind 0).  Straight-line code for a full warp of such units; anything longer (a third sector, two
// hit entries with the same ensg inside one sector) goes to the exact kernel.
// returns 0 done, 1 exact kernel (possible double hit of one ensg), 2 needs a third sector (bulk_general)
template <bool ALLHOT>
__device__ __forceinline__ int bulk_deferred(const StabView& sv, const QEnt e, bool live,
                                             u32 hot_addr, u32 n_hot, u64* __restrict__ counts, u64* __restrict__ stats,
                                             u32& n_assigned, u32 one) {
    if (!live) return 0;
    const u32 kind = e.secA >> 24, prim = e.secA & 0xFFFFFFu;
    const Sector A = ld_sector(sv.sectors, prim);
    const u32 hitA = sector_hits(A, make_point(e.pa & 0xFFFFu), make_point(e.pa >> 16));
    const bool a_over = sector_more(A) && points_rmax(e.pa) >= (int)sector_last_s(A);
    const u32 secB = kind ? e.secB : (__ldg(sv.ovf_base + (prim >> 7)) + sector_link(A));
    const u32 pB = kind ? e.pb : e.pa;
    const Sector B = ld_sector(sv.sectors, (kind || a_over) ? secB : prim);
    u32 hitB = (kind || a_over) ? sector_hits(B, make_point(pB & 0xFFFFu), make_point(pB >> 16)) : 0u;
    if ((kind && a_over) || ((kind || a_over) && sector_more(B) && points_rmax(pB) >= (int)sector_last_s(B))) return 2;
    if (sector_twin_hit(A, hitA) || sector_twin_hit(B, hitB)) return 1;
    if (!(hitA | hitB)) return 0;                                                      // :128 no result
    n_assigned++;                                                                      // :149
    if (!sv.all_counted && !bulk_type_rule(sv, sector_typemask(sv, A, hitA) | sector_typemask(sv, B, hitB), stats)) return 0;
    hitB = drop_if_in_a<0>(hitA, hitB, A, B);
    hitB = drop_if_in_a<1>(hitA, hitB, A, B);
    hitB = drop_if_in_a<2>(hitA, hitB, A, B);
    hitB = drop_if_in_a<3>(hitA, hitB, A, B);
    hitB = drop_if_in_a<4>(hitA, hitB, A, B);
    bump_sector<ALLHOT>(hitA, A, hot_addr, n_hot, counts, one);
    bump_sector<ALLHOT>(hitB, B, hot_addr, n_hot, counts, one);
    return 0;
}

// The general case, a warp of units at a time: walk the sector chains of one or two cells and keep
// the distinct ensg in a register set.  Returns true when the set overflows (exact kernel).
#define GEN_MAXD 8
template <bool ALLHOT>
__device__ __forceinline__ bool bulk_general(const StabView& sv, const QEnt e, bool live,
                                             u32 hot_addr, u32 n_hot, u64* __restrict__ counts, u64* __restrict__ stats,
                                             u32& n_assigned, u32 one) {
    if (!live) return false;
    u32 dist[GEN_MAXD];
#pragma unroll
    for (int i = 0; i < GEN_MAXD; ++i) dist[i] = 0xFFFFFFFFu;
    u32 nd = 0;
    const int n_cell = (e.secA >> 24) ? 2 : 1;
    for (int ci = 0; ci < n_cell; ++ci) {
        const u32 prim = ci ? e.secB : (e.secA & 0xFFFFFFu);
        const u32 pp = ci ? e.pb : e.pa;
        const PointK pa = make_point(pp & 0xFFFFu), pb = make_point(pp >> 16);
        const int rmax = points_rmax(pp);
        u32 sec = prim;
        for (;;) {
            const Sector s = ld_sector(sv.sectors, sec);
            u32 hit = sector_hits(s, pa, pb);
            while (hit) {
                const u32 low = hit & (0u - hit);
                hit ^= low;
                const u32 w = (low == HB0) ? sector_slot_c<0>(s) : (low == HB1) ? sector_slot_c<1>(s) : (low == HB2) ? sector_slot_c<2>(s)
                              : (low == HB3) ? sector_slot_c<3>(s) : sector_slot_c<4>(s);
                bool found = false;
#pragma unroll
                for (int j = 0; j < GEN_MAXD; ++j) found |= (dist[j] == w);
                if (!found) {
#pragma unroll
                    for (int j = 0; j < GEN_MAXD; ++j) if ((u32)j == nd) dist[j] = w;
                    ++nd;
                }
            }
            if (!sector_more(s) || rmax < (int)sector_last_s(s)) break;
            sec = (sec == prim) ? __ldg(sv.ovf_base + (prim >> 7)) + sector_link(s) : sec + 1;
        }
    }
    if (nd > GEN_MAXD) return true;
    if (!nd) return false;                                                             // :128 no result
    n_assigned++;                                                                      // :149
    if (!sv.all_counted) {
        u32 typemask = 0;
#pragma unroll
        for (int j = 0; j < GEN_MAXD; ++j) if ((u32)j < nd) typemask |= 1u << __ldg(sv.slot_type + dist[j]);
        if (!bulk_type_rule(sv, typemask, stats)) return false;
    }
#pragma unroll
    for (int j = 0; j < GEN_MAXD; ++j) {
        if ((u32)j < nd) {
            const u32 slot = dist[j];
            if (ALLHOT || slot < n_hot) asm volatile("red.shared.add.u32 [%0], %1;" :: "r"(hot_addr + slot * 4u), "r"(one) : "memory");
            else atomicAdd(counts + slot, 1ULL);
        }
    }
    return false;
}

// One warp per 32 consecutive units, grid-stride; the next warp-tile's records are requested before
// the current one is looked up.
// NT threads per CTA; the first n_hot ensg slots are counted in dynamic shared memory (ALLHOT: all of them,
// one CTA of 1024 threads per SM; otherwise TEC_HOT_SLOTS of them, two CTAs of 512 threads per SM).
template <bool PAIRED, int NT, bool ALLHOT>
__global__ void __launch_bounds__(NT, 2048 / NT / 2)
bulk_count_cell_kernel(IndexView iv, StabView sv, int64_t n_units, int qual,
                       const int32_t* __restrict__ start, const int32_t* __restrict__ end,
                       const uint16_t* __restrict__ chrom, const uint8_t* __restrict__ mapq,
                       const uint8_t* __restrict__ flag, u64* __restrict__ counts, u64* __restrict__ stats,
                       u32* __restrict__ slow_list, u32 n_hot, QEnt* __restrict__ g_ring, u32* __restrict__ g_ring_u) {
    constexpr int BULK_WARPS = NT / 32;
    __shared__ BulkShared<BULK_WARPS> sh;
    extern __shared__ __align__(16) u32 s_hot_dyn[];
    for (u32 i = threadIdx.x; i < n_hot; i += blockDim.x) s_hot_dyn[i] = 0;
    if (threadIdx.x < TEC_BULK_NSTATS) sh.stats[threadIdx.x] = 0;
    __syncthreads();
    u32 n_assigned = 0, n_lowq = 0, n_badchrom = 0, n_qcfail = 0;
    const u32 reject = TEC_F_UNMAPPED | TEC_F_DUP | TEC_F_QCFAIL;
    const u32 reject2 = PAIRED ? (reject | (reject << 8)) : reject;
    const u64 pol = make_evict_first_policy();
    const int bs = iv.bs;
    const int shift = sv.shift;
    const u32 cmask = (1u << shift) - 1;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const u32 lt_mask = (1u << lane) - 1u;
    const u32 hot_addr = (u32)__cvta_generic_to_shared(&s_hot_dyn[0]);
    // the increment as a run-time value: a literal 1 makes ptxas pick ATOMS.POPC.INC, which needs a
    // converged warp and therefore a branch around every reduction
    const u32 one = (u32)(n_units > 0);
    QEnt* const ring = sh.q[wib];
    u32* const ring_u = sh.qu[wib];
    u32 q_head = 0, q_count = 0;                     // warp-uniform
    // second ring (global memory, rarely used): units that need a third sector
    QEnt* const ring2 = g_ring + (size_t)(blockIdx.x * BULK_WARPS + wib) * BULK_QCAP;
    u32* const ring2_u = g_ring_u + (size_t)(blockIdx.x * BULK_WARPS + wib) * BULK_QCAP;
    u32 q2_head = 0, q2_count = 0;
    // a batch of ring 1: two-sector code; what it cannot finish goes to the slow list or to ring 2
    auto run_ring1 = [&](bool all) {
        const u32 at = (q_head + lane) & (BULK_QCAP - 1);
        const QEnt e = ring[at];
        const u32 eu = ring_u[at];
        const int code = bulk_deferred<ALLHOT>(sv, e, all || (u32)lane < q_count, hot_addr, n_hot, counts, stats, n_assigned, one);
        flag_slow_warp(slow_list, code == 1, eu, lt_mask);
        const u32 gm = __ballot_sync(0xFFFFFFFFu, code == 2);
        if (gm) {
            if (code == 2) {
                const u32 at2 = (q2_head + q2_count + __popc(gm & lt_mask)) & (BULK_QCAP - 1);
                ring2[at2] = e;
                ring2_u[at2] = eu;
            }
            q2_count += __popc(gm);
            __syncwarp();
        }
    };
    auto run_ring2 = [&](bool all) {
        const u32 at = (q2_head + lane) & (BULK_QCAP - 1);
        const bool sl = bulk_general<ALLHOT>(sv, ring2[at], all || (u32)lane < q2_count, hot_addr, n_hot, counts, stats, n_assigned, one);
        flag_slow_warp(slow_list, sl, ring2_u[at], lt_mask);
    };
    const u32 n_u = (u32)n_units;                     // a launch holds < 2^28 units (TEC_LAUNCH_UNITS)
    const u32 n_tiles = (n_u + 31) >> 5;
    const u32 tile_stride = gridDim.x * BULK_WARPS;
    u32 tile = blockIdx.x * BULK_WARPS + wib;
    BulkRec cur, nxt;
    cur.fl = cur.q = 0; cur.c = cur.loc1 = cur.loc2 = 0;
    nxt = cur;
    if (tile < n_tiles && tile * 32 + lane < n_u) cur = bulk_load<PAIRED>(tile * 32 + lane, start, end, chrom, mapq, flag, pol);
    for (; tile < n_tiles; tile += tile_stride) {
        const u32 u = tile * 32 + lane;
        const u32 un = u + tile_stride * 32;
        if (un < n_u) nxt = bulk_load<PAIRED>(un, start, end, chrom, mapq, flag, pol);
        // ---- filter (te_count.py:78-102 / :203-218)
        const int c = cur.c, loc1 = cur.loc1, loc2 = cur.loc2;
        // first failing test wins, as in the reference's if / continue chain; branch-free counters
        const bool live = u < n_u;
        const bool f_qc = (cur.fl & reject2) != 0;                                         // :81-86 / :204
        const bool f_lq = (int)cur.q < qual;                                               // :88 / :208
        const bool f_nm = PAIRED && (cur.fl & TEC_F_NAME_MISMATCH);                        // :92-94
        // cells[] has one entry per chromosome plus a sentinel; chromosomes that are not keys of the
        // bucket hash (no feature) have zero cells
        const uint2 cell = __ldg(sv.cells + min((u32)c, (u32)iv.n_chrom));
        const bool f_bc = cell.y == 0;                                                     // :100 / :216
        n_qcfail += live & f_qc;
        n_lowq += live & !f_qc & f_lq;
        n_badchrom += live & !(f_qc | f_lq | f_nm) & f_bc;
        if (PAIRED && live && !(f_qc | f_lq) && f_nm) atomicAdd(stats + TEC_BS_CRASH_NAME, 1ULL);
        const bool look = live & !(f_qc | f_lq | f_nm | f_bc);
        // ---- which sector(s)
        QEnt qe;
        qe.secA = qe.secB = 0; qe.pa = qe.pb = R_NONE | (R_NONE << 16);
        bool defer = false, single = false, slow = false;
        int rmax = -1;
        if (look) {
            const bool edge = (bs == 10000) ? (mult_of_10000(loc1) | mult_of_10000(loc2 + 1))
                                            : ((loc1 % bs == 0) || ((loc2 + 1) % bs == 0));
            if (edge) slow = true;
            else {
                const int xa = loc1, xb = loc2 - 1;
                int ka = xa >> shift, kb = xb >> shift;                          // arithmetic shift: negative stays negative
                const bool va = (u32)ka < cell.y, vb = (u32)kb < cell.y;         // negative -> huge -> false
                u32 ra = (u32)xa & cmask, rb = (u32)xb & cmask;
                if (va && vb && ka != kb) {
                    // neighbouring cells: the lower cell's list reaches STAB_EXT bp into the upper one
                    if (kb == ka + 1 && rb < STAB_EXT) { kb = ka; rb += cmask + 1; }
                    else if (ka == kb + 1 && ra < STAB_EXT) { ka = kb; ra += cmask + 1; }
                }
                if (va && vb && ka != kb) {
                    qe.secA = (cell.x + (u32)ka) | (1u << 24);
                    qe.secB = cell.x + (u32)kb;
                    qe.pa = ra | (R_NONE << 16);
                    qe.pb = R_NONE | (rb << 16);
                    defer = true;
                } else if (va || vb) {
                    qe.secA = cell.x + (u32)(va ? ka : kb);
                    qe.pa = (va ? ra : R_NONE) | ((vb ? rb : R_NONE) << 16);
                    rmax = max(va ? (int)ra : -1, vb ? (int)rb : -1);
                    single = true;
                }
            }
        }
        // ---- the common case: one sector
        if (single) {
            const Sector s = ld_sector(sv.sectors, qe.secA);
            const u32 hit = sector_hits(s, make_point(qe.pa & 0xFFFFu), make_point(qe.pa >> 16));
            if (sector_more(s) && rmax >= (int)sector_last_s(s)) {
                defer = true;                                                              // the chain is walked again from A
            } else if (sector_twin_hit(s, hit)) {
                slow = true;                                                               // the same ensg may be hit twice
            } else if (hit) {                                                              // :128 result not empty
                n_assigned++;                                                              // :149
                bool count_it = true;
                if (!sv.all_counted) count_it = bulk_type_rule(sv, sector_typemask(sv, s, hit), stats);
                if (count_it) {
                    bump_sector<ALLHOT>(hit, s, hot_addr, n_hot, counts, one);
                }
            }
        }
        flag_slow_warp(slow_list, slow, (u32)u, lt_mask);
        // ---- park deferred units; look a full warp of them up when there are 32
        const u32 dm = __ballot_sync(0xFFFFFFFFu, defer);
        if (dm) {
            if (defer) {
                const u32 at = (q_head + q_count + __popc(dm & lt_mask)) & (BULK_QCAP - 1);
                ring[at] = qe;
                ring_u[at] = (u32)u;
            }
            q_count += __popc(dm);
            __syncwarp();
            if (q_count >= 32) {
                run_ring1(true);
                q_head = (q_head + 32) & (BULK_QCAP - 1);
                q_count -= 32;
                __syncwarp();
                if (q2_count >= 32) {
                    run_ring2(true);
                    q2_head = (q2_head + 32) & (BULK_QCAP - 1);
                    q2_count -= 32;
                    __syncwarp();
                }
            }
        }
        cur = nxt;
    }
    if (q_count) run_ring1(false);
    while (q2_count) {                                // at most two rounds: fewer than 64 entries
        run_ring2(false);
        const u32 done = min(q2_count, 32u);
        q2_head = (q2_head + done) & (BULK_QCAP - 1);
        q2_count -= done;
        __syncwarp();
    }
    u64 v[4] = {n_assigned, n_lowq, n_badchrom, n_qcfail};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const u64 s = warp_sum(v[i]);
        if (lane == 0 && s) atomicAdd(&sh.stats[TEC_BS_ASSIGNED + i], s);
    }
    __syncthreads();
    if (threadIdx.x >= TEC_BS_ASSIGNED && threadIdx.x < TEC_BS_ASSIGNED + 4 && sh.stats[threadIdx.x])
        atomicAdd(stats + threadIdx.x, sh.stats[threadIdx.x]);
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(stats + TEC_BS_UNITS, (u64)n_units);
    for (u32 i = threadIdx.x; i < n_hot; i += blockDim.x) {
        const u32 x = s_hot_dyn[i];
        if (x) atomicAdd(counts + i, (u64)x);
    }
}

// Units flagged by the fast kernel: bucket-edge candidates take the exact search (counters in slot
// space); units with more than STAB_MAXD distinct ensg walk the cell table again with a larger set.
// One thread per flagged unit.
#define SLOW_MAXD 8
#define SLOW_MAXD_EXACT 96
template <bool PAIRED>
__global__ void __launch_bounds__(256)
bulk_slow_kernel(IndexView iv, StabView sv, int has_stab, const int32_t* __restrict__ start, const int32_t* __restrict__ end,
                 const uint16_t* __restrict__ chrom, u64* __restrict__ counts, u64* __restrict__ stats,
                 const u32* __restrict__ slow_list) {
    // hot ensg counters privatised per CTA (a Zipf-hot TE name would otherwise serialise in one L2 slice)
    __shared__ u32 s_hot[TEC_HOT_SLOTS];
    for (int i = threadIdx.x; i < TEC_HOT_SLOTS; i += blockDim.x) s_hot[i] = 0;
    __syncthreads();
    auto bump = [&](u32 slot) {
        if (slot < TEC_HOT_SLOTS) atomicAdd(&s_hot[slot], 1u);
        else atomicAdd(counts + slot, 1ULL);
    };
    const u32 n = slow_list[0];
    const u32 counted = (1u << TEC_T_GENE) | (1u << TEC_T_TE) | (1u << TEC_T_SNRNA);
    u32 n_assigned = 0;
    for (u32 t = blockIdx.x * blockDim.x + threadIdx.x; t < n; t += gridDim.x * blockDim.x) {
        const int64_t u = slow_list[1 + t];
        int c, loc1, loc2;
        if (PAIRED) { c = chrom[2 * u]; loc1 = start[2 * u]; loc2 = start[2 * u + 1]; }
        else { c = chrom[u]; loc1 = start[u]; loc2 = end[u]; }
        const bool edge = loc1 < 0 || loc2 + 1 < 0 || (loc1 % iv.bs == 0) || ((loc2 + 1) % iv.bs == 0);
        if (has_stab && !edge) {
            // same lookup as the fast kernel, distinct slots in a register set of SLOW_MAXD
            u32 dist[SLOW_MAXD];
#pragma unroll
            for (int i = 0; i < SLOW_MAXD; ++i) dist[i] = 0xFFFFFFFFu;
            u32 nd = 0;
            const uint2 cell = __ldg(sv.cells + c);
            const int x[2] = {loc1, loc2 - 1};
            for (int p = 0; p < 2; ++p) {
                const int k = x[p] >> sv.shift;
                if ((u32)k >= cell.y) continue;
                const u32 r = (u32)x[p] & ((1u << sv.shift) - 1);
                const u32 prim = cell.x + (u32)k;
                u32 sec = prim;
                const PointK pk = make_point(r), pn = make_point(R_NONE);
                for (;;) {
                    const Sector s = ld_sector(sv.sectors, sec);
                    u32 hit = sector_hits(s, pk, pn);
                    while (hit) {
                        const u32 low = hit & (0u - hit);
                        hit ^= low;
                        const u32 e = (low == HB0) ? sector_slot_c<0>(s) : (low == HB1) ? sector_slot_c<1>(s) : (low == HB2) ? sector_slot_c<2>(s)
                                      : (low == HB3) ? sector_slot_c<3>(s) : sector_slot_c<4>(s);
                        bool found = false;
#pragma unroll
                        for (int j = 0; j < SLOW_MAXD; ++j) found |= (dist[j] == e);
                        if (!found) {
#pragma unroll
                            for (int j = 0; j < SLOW_MAXD; ++j) if ((u32)j == nd) dist[j] = e;
                            ++nd;                                                      // nd > SLOW_MAXD: overflow
                        }
                    }
                    if (!sector_more(s) || r < sector_last_s(s)) break;
                    sec = (sec == prim) ? __ldg(sv.ovf_base + (prim >> 7)) + sector_link(s) : sec + 1;
                }
            }
            if (nd <= SLOW_MAXD) {
                if (!nd) continue;                                                     // :128 no result
                n_assigned++;                                                          // :149
                u32 typemask = sv.all_counted ? counted : 0u;
                if (!sv.all_counted) {
#pragma unroll
                    for (int j = 0; j < SLOW_MAXD; ++j) if ((u32)j < nd) typemask |= 1u << __ldg(sv.slot_type + dist[j]);
                }
                if (!(typemask & counted)) {
                    if (typemask & (1u << TEC_T_ENHANCER)) atomicAdd(stats + TEC_BS_CRASH_ENHANCER, 1ULL);
                    continue;
                }
#pragma unroll
                for (int j = 0; j < SLOW_MAXD; ++j) if ((u32)j < nd) bump(dist[j]);
                continue;
            }
        }
        // one walk: type mask + the first SLOW_MAXD_EXACT distinct ensg
        u32 typemask = 0, nd = 0, dist[SLOW_MAXD_EXACT];
        bool overflow = false;
        bulk_for_each_hit(iv, c, loc1, loc2, [&](int64_t fi) {
            const u32 w = __ldg(iv.info + fi);
            typemask |= 1u << info_type(w);
            const u32 e = info_ensg(w);
            bool found = false;
            for (u32 i = 0; i < nd; ++i) found |= (dist[i] == e);
            if (!found) {
                if (nd < SLOW_MAXD_EXACT) dist[nd++] = e; else overflow = true;
            }
            return true;
        });
        if (!typemask) continue;                                                       // :128 no result
        n_assigned++;                                                                  // :149
        if (!(typemask & counted)) {
            if (typemask & (1u << TEC_T_ENHANCER)) atomicAdd(stats + TEC_BS_CRASH_ENHANCER, 1ULL);
            continue;
        }
        if (!overflow) {
            for (u32 i = 0; i < nd; ++i) bump(dist[i]);                                // one per distinct ensg
            continue;
        }
        // more distinct ensg than the list holds: count a hit iff no earlier hit (in enumeration
        // order) carries the same ensg -- O(h^2) re-walks, no storage
        int h = 0;
        bulk_for_each_hit(iv, c, loc1, loc2, [&](int64_t fi) {
            const u32 e = info_ensg(__ldg(iv.info + fi));
            int j = 0;
            bool dup = false;
            bulk_for_each_hit(iv, c, loc1, loc2, [&](int64_t fj) {
                if (j++ >= h) return false;
                if (info_ensg(__ldg(iv.info + fj)) == e) { dup = true; return false; }
                return true;
            });
            if (!dup) bump(e);
            ++h;
            return true;
        });
    }
    const u64 a_sum = warp_sum((u64)n_assigned);
    if ((threadIdx.x & 31) == 0 && a_sum) atomicAdd(stats + TEC_BS_ASSIGNED, a_sum);
    __syncthreads();
    for (int i = threadIdx.x; i < TEC_HOT_SLOTS; i += blockDim.x) {
        const u32 x = s_hot[i];
        if (x) atomicAdd(counts + i, (u64)x);
    }
}
