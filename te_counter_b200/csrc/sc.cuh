// Single-cell path: filter + whitelist, UMI collapse with the reference's bundle semantics, top-cell
// selection, Part-2 keep rule, overlap + tally, cell ranking.
//
// Reference (te_counter, te_count/te_count.py): Part 1 :372-491, Part 2 :493-575, Part 3 :577-707,
// sc_save_result :709-754.  The reference spills "bundles" of 1e7 (cell, UMI) keys to sorted text
// files and merges them with a held-line scan; nothing is spilled here, but every observable effect
// of that scheme is reproduced as sort / scan / segmented primitives (SURVEY.md 8a-9..13):
//
//   survivors      records that pass flags, MAPQ, whitelist and the '_'/'alt' skip, in file order i
//   key group      equal (cell, UMI); found by a stable LSD radix sort of i by UMI, then by cell
//   bundle         a maximal run of survivors whose number of first-in-bundle keys reaches
//                  bundle_keys; boundaries come from prev[i] (previous survivor with the same key)
//   segment        (cell, UMI, bundle): one line of one bundle file.  Its head is the first-inserted
//                  fragment (canonical rule for te_count.py:452); same chrom:strand as the head ->
//                  "already seen", anything else is added and counted in the cell's raw total
//   kept line      Part-2 held-line scan: the first line of a to-do cell in a bundle survives only if
//                  a line of a cell between the previous to-do id and this one precedes it
//   winner         of the kept lines of one (cell, UMI) only the lowest bundle's is used (:552-555)
//   fragments      per winner: the head, plus per other chrom:strand the distinct fragment whose
//                  first occurrence is latest (:603-606); each is looked up with the inclusive
//                  point tests of :645/:648 over the bucket range of :619-621
//
// Sorting and scanning use CUB device primitives as building blocks (cub::DeviceRadixSort,
// cub::DeviceScan, cub::DeviceRunLengthEncode); everything else is hand-written below.
#pragma once
#include "context.cuh"
#include <cub/cub.cuh>
#include "radix.cuh"

#define SC_NONE 0xFFFFFFFFu

struct ScState {
    int qual = 20, strand = 0;
    int64_t n_wl = 0;
    bool active = false, finalized = false;
    int64_t units = 0;
    // survivors, in file order
    u32* cell = nullptr;
    u64* umi = nullptr;
    uint4* frag = nullptr;          // {cs = chrom << 2 | strand code (0 '+', 1 '-', 2 'NA'), left, rite, 0}: one 16-byte
                                    // record, so the gather into sorted order is one random read per survivor
    int64_t n = 0, cap = 0;         // n is exact only after sc_sync_count()
    u64* d_n = nullptr;             // [0] survivors held (device): pushes do not wait for the host; [1] OR of their UMI codes, [2] of their chrom:strand words
    bool or_tracked = false;        // d_n[1..2] cover every survivor held (false after tec_sc_import_packed_dev)
    int64_t n_bound = 0;            // upper bound of n (everything pushed so far), sizes the columns
    bool n_pending = false;
    void* packed = nullptr;         // multi-GPU: survivors packed for the exchange (tec_sc_partition_dev)
    u64* gidx = nullptr;            // multi-GPU: position of each survivor in the whole job's survivor order
    int64_t gidx_cap = 0;
    bool has_gidx = false;
    tec_allreduce_fn coll = nullptr;    // multi-GPU: all-reduce over the ranks' device buffers
    void* coll_user = nullptr;
    int rank = 0, world = 1;
    u64* d_stats = nullptr;         // TEC_SC_NSTATS
    // per-push scratch
    u32* pos = nullptr;
    int64_t pos_cap = 0;
    void* cub_tmp = nullptr;
    size_t cub_cap = 0;
    // results
    int32_t* t_ensg = nullptr;
    u32* t_cell = nullptr;
    int64_t* t_count = nullptr;
    int64_t n_triples = 0;
    u32* h_cell = nullptr;          // hit cells ascending
    int64_t* h_count = nullptr;
    int64_t n_hit = 0;
    char* text = nullptr;           // dense matrix rows as text (sc_text.cuh)
    int64_t text_bytes = 0;
    int64_t stats[TEC_SC_NSTATS] = {0};
};

static void sc_free_results(tec_ctx* ctx, ScState* s) {
    ctx->cache.put(s->t_ensg); ctx->cache.put(s->t_cell); ctx->cache.put(s->t_count); ctx->cache.put(s->h_cell); ctx->cache.put(s->h_count);
    ctx->cache.put(s->text);
    s->t_ensg = nullptr; s->t_cell = nullptr; s->t_count = nullptr; s->h_cell = nullptr; s->h_count = nullptr; s->text = nullptr;
    s->n_triples = s->n_hit = s->text_bytes = 0;
}

inline void tec_ctx::free_sc() {
    if (!sc) return;
    cudaFree(sc->cell); cudaFree(sc->umi); cudaFree(sc->frag); cudaFree(sc->gidx); cudaFree(sc->d_n);
    cudaFree(sc->d_stats); cudaFree(sc->pos); cudaFree(sc->cub_tmp);
    cache.put(sc->packed);
    sc_free_results(this, sc);
    delete sc;
    sc = nullptr;
}

// every temporary of finalize goes through this and goes back to the context's block cache at the
// end (also on errors)
struct ScArena {
    DevCache& cache;
    std::vector<void*> ptrs;
    explicit ScArena(DevCache& c) : cache(c) {}
    ~ScArena() { for (void* p : ptrs) cache.put(p); }
    template <class T> cudaError_t get(T** out, size_t count) {
        void* p = nullptr;
        cudaError_t e = cache.get(&p, std::max<size_t>(count, 1) * sizeof(T));
        if (e == cudaSuccess) ptrs.push_back(p);
        *out = (T*)p;
        return e;
    }
    void release(void* p) {
        for (auto& q : ptrs) if (q == p && p) { cache.put(p); q = nullptr; }
    }
};

static int sc_cub_tmp(tec_ctx* ctx, size_t bytes) {
    ScState* s = ctx->sc;
    if (bytes <= s->cub_cap) return TEC_OK;
    TEC_CUDA(cudaStreamSynchronize(ctx->stream));
    cudaFree(s->cub_tmp);
    s->cub_tmp = nullptr;
    s->cub_cap = 0;
    TEC_CUDA(cudaMalloc(&s->cub_tmp, bytes + (bytes >> 3) + 256));
    s->cub_cap = bytes + (bytes >> 3) + 256;
    return TEC_OK;
}

struct MaxU32 { __device__ __forceinline__ u32 operator()(u32 a, u32 b) const { return a > b ? a : b; } };
struct MaxI32 { __device__ __forceinline__ int operator()(int a, int b) const { return a > b ? a : b; } };
struct SumU32 { __device__ __forceinline__ u32 operator()(u32 a, u32 b) const { return a + b; } };
// line j of the sorted order is the winner of its key group (te_count.py:552-555): head of a segment, first kept line of the key
struct ScIsWinner {
    const u32 *shead_pos, *khead_pos, *winner_at;
    __device__ __forceinline__ bool operator()(u32 j) const { return shead_pos[j] == j && winner_at[khead_pos[j]] == j; }
};

#define SC_GRID(n) (int)std::max<int64_t>(1, std::min<int64_t>(((n) + 255) / 256, (int64_t)ctx->n_sm * 16)), 256, 0, ctx->stream
#define SC_LOOP(i, n) for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (n); i += (int64_t)gridDim.x * blockDim.x)

// ------------------------------------------------------------------------------------ Part 1: filter
// te_count.py:394-438.  keep[r] = 1 for survivors; statistics by warp-aggregated atomics.
__device__ __forceinline__ u32 sc_filter_one(u32 f, u32 q, u32 cell, u32 chrom, int qual, u32& n_qc, u32& n_lowq, u32& n_badbc) {
    if (f & (TEC_F_UNMAPPED | TEC_F_DUP | TEC_F_QCFAIL)) { n_qc++; return 0u; }          // :394
    if ((int)q < qual) { n_lowq++; return 0u; }                                            // :398
    if (cell == TEC_CELL_INVALID) { n_badbc++; return 0u; }                                // :412
    return chrom != TEC_CHROM_SC_SKIP ? 1u : 0u;                                           // :432 silent skip
}
// VEC: four records per thread, one load per column (the arrays of a push are at least 16-byte aligned)
template <bool VEC>
__global__ void sc_filter_kernel(int64_t n, int qual, const uint16_t* __restrict__ chrom, const uint8_t* __restrict__ mapq,
                                 const uint8_t* __restrict__ flag, const u32* __restrict__ cell,
                                 u32* __restrict__ keep, u64* __restrict__ stats) {
    u32 n_qc = 0, n_lowq = 0, n_badbc = 0;
    if (VEC) {
        const int64_t n4 = n >> 2;
        SC_LOOP(g, n4) {
            const u32 f4 = reinterpret_cast<const u32*>(flag)[g], q4 = reinterpret_cast<const u32*>(mapq)[g];
            const uint2 c4 = reinterpret_cast<const uint2*>(chrom)[g];
            const uint4 b4 = reinterpret_cast<const uint4*>(cell)[g];
            uint4 k;
            k.x = sc_filter_one(f4 & 0xFFu, q4 & 0xFFu, b4.x, c4.x & 0xFFFFu, qual, n_qc, n_lowq, n_badbc);
            k.y = sc_filter_one((f4 >> 8) & 0xFFu, (q4 >> 8) & 0xFFu, b4.y, c4.x >> 16, qual, n_qc, n_lowq, n_badbc);
            k.z = sc_filter_one((f4 >> 16) & 0xFFu, (q4 >> 16) & 0xFFu, b4.z, c4.y & 0xFFFFu, qual, n_qc, n_lowq, n_badbc);
            k.w = sc_filter_one(f4 >> 24, q4 >> 24, b4.w, c4.y >> 16, qual, n_qc, n_lowq, n_badbc);
            reinterpret_cast<uint4*>(keep)[g] = k;
        }
        const int64_t r = (n4 << 2) + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;      // the last n % 4 records
        if (r < n) keep[r] = sc_filter_one(flag[r], mapq[r], cell[r], chrom[r], qual, n_qc, n_lowq, n_badbc);
    } else {
        SC_LOOP(r, n) keep[r] = sc_filter_one(flag[r], mapq[r], cell[r], chrom[r], qual, n_qc, n_lowq, n_badbc);
    }
    const u64 a = warp_sum(n_qc), b = warp_sum(n_lowq), c = warp_sum(n_badbc);
    if ((threadIdx.x & 31) == 0) {
        if (a) atomicAdd(stats + TEC_SS_QCFAIL, a);
        if (b) atomicAdd(stats + TEC_SS_LOWQ, b);
        if (c) atomicAdd(stats + TEC_SS_INVALID_BARCODE, c);
    }
}

// stable compaction of the survivors behind the ones already held (pos = exclusive scan of keep)
__global__ void sc_scatter_kernel(int64_t n, int strand, const u64* __restrict__ d_base, u64* __restrict__ d_or, const u32* __restrict__ keep_pos, const u32* __restrict__ keep_last,
                                  const int32_t* __restrict__ start, const int32_t* __restrict__ end,
                                  const uint16_t* __restrict__ chrom, const uint8_t* __restrict__ flag,
                                  const u32* __restrict__ cell, const u64* __restrict__ umi,
                                  u32* __restrict__ o_cell, u64* __restrict__ o_umi, uint4* __restrict__ o_frag) {
    const int64_t base = (int64_t)*d_base;
    u64 or_umi = 0;                                   // how many bits the sort keys need (tec_sc_finalize)
    u32 or_cs = 0;
    SC_LOOP(r, n) {
        const u32 p = keep_pos[r];
        const u32 nxt = (r + 1 < n) ? keep_pos[r + 1] : *keep_last;
        if (nxt == p) continue;
        const int64_t o = base + p;
        o_cell[o] = cell[r];
        const u64 u = umi[r];
        o_umi[o] = u;
        const u32 sc = strand ? ((flag[r] & TEC_F_REVERSE) ? 1u : 0u) : 2u;            // :437-438
        const u32 cs = ((u32)chrom[r] << 2) | sc;
        o_frag[o] = make_uint4(cs, (u32)start[r], (u32)end[r], 0u);                      // :434-435
        or_umi |= u;
        or_cs |= cs;
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) { or_umi |= __shfl_xor_sync(0xffffffffu, or_umi, d); or_cs |= __shfl_xor_sync(0xffffffffu, or_cs, d); }
    if ((threadIdx.x & 31) == 0) {
        if (or_umi) atomicOr(d_or, or_umi);
        if (or_cs) atomicOr(d_or + 1, (u64)or_cs);
    }
}

__global__ void sc_advance_kernel(u64* __restrict__ d_n, const u32* __restrict__ total) {
    if (threadIdx.x == 0 && blockIdx.x == 0) *d_n += *total;
}
// keep_pos holds the EXCLUSIVE scan; total = scan[n-1] + keep[n-1] is written by this helper
__global__ void sc_total_kernel(int64_t n, const u32* __restrict__ excl, const u32* __restrict__ keep_last_flag, u32* __restrict__ total) {
    if (threadIdx.x == 0 && blockIdx.x == 0) *total = excl[n - 1] + *keep_last_flag;
}

// ------------------------------------------------------------------------------------ helpers
__global__ void sc_iota_kernel(int64_t n, u32* __restrict__ v) { SC_LOOP(i, n) v[i] = (u32)i; }
// out[0] = OR of the UMI codes, out[1] = OR of the chrom:strand words (how many bits the sort keys need)
__global__ void sc_or_kernel(int64_t n, const u64* __restrict__ v, const uint4* __restrict__ frag, u64* __restrict__ out) {
    u64 acc = 0;
    u32 acc_cs = 0;
    SC_LOOP(i, n) { acc |= v[i]; acc_cs |= frag[i].x; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { acc |= __shfl_xor_sync(0xffffffffu, acc, o); acc_cs |= __shfl_xor_sync(0xffffffffu, acc_cs, o); }
    if ((threadIdx.x & 31) == 0 && acc) atomicOr(out, acc);
    if ((threadIdx.x & 31) == 0 && acc_cs) atomicOr(out + 1, (u64)acc_cs);
}

// One 64-bit sort key per survivor: cell | UMI at 2 bits per character | chrom:strand word.  Only for UMIs of exactly
// L <= 16 characters over {A, C, G, T} (3-bit codes 1, 2, 3, 5 left aligned in 63 bits, reads.py); anything else raises
// *bad and the caller takes the two-sort path.  The 21 groups are converted at once: g - 1 - (g >> 2) maps 1, 2, 3, 5
// to 0..3 without borrows, then four shift-and-mask steps close the gaps between the 2-bit fields.
__global__ void sc_pack_key_kernel(int64_t n, const u32* __restrict__ cell, const u64* __restrict__ umi, const uint4* __restrict__ frag,
                                   int L, int cs_bits, u64* __restrict__ key, u32* __restrict__ idx, u32* __restrict__ bad) {
    const u64 M1 = 0x1249249249249249ULL;
    const int drop = 3 * (21 - L);
    const u64 low = (1ULL << drop) - 1ULL;                    // L >= 1: drop <= 60
    const u64 ML = M1 & ((1ULL << (3 * L)) - 1ULL);           // L <= 16: 3 L <= 48
    bool any_bad = false;
    SC_LOOP(i, n) {
        const u64 code = umi[i];
        const u64 x = code >> drop;
        const u64 b0 = x & ML, b1 = (x >> 1) & ML, b2 = (x >> 2) & ML;
        any_bad |= ((code & low) | (code >> 63) | (ML & ~(b0 | b1 | b2)) | (b2 & ((ML & ~b0) | b1))) != 0;
        u64 y = x - ML - b2;
        y = (y & 0x30C30C30C30C30C3ULL) | ((y >> 1) & (0x30C30C30C30C30C3ULL << 2));
        y = (y & 0xF00F00F00F00F00FULL) | ((y >> 2) & (0xF00F00F00F00F00FULL << 4));
        y = (y & 0x00FF0000FF0000FFULL) | ((y >> 4) & (0x00FF0000FF0000FFULL << 8));
        y = (y & 0xFFFF00000000FFFFULL) | ((y >> 8) & (0xFFFF00000000FFFFULL << 16));
        const u64 u2 = y & 0xFFFFFFFFULL;
        key[i] = ((u64)cell[i] << (2 * L + cs_bits)) | (u2 << cs_bits) | (u64)frag[i].x;
        idx[i] = (u32)i;
    }
    if (__any_sync(0xFFFFFFFFu, any_bad) && (threadIdx.x & 31) == 0) atomicOr(bad, 1u);
}

// sorted packed keys -> the columns the rest of the pipeline reads (cell, UMI, chrom:strand word in sorted order),
// key-group heads, and prev[i] = previous survivor with the same (cell, UMI)
// SCATTER: prev[perm[j]] is written in place (a random 4-byte store per survivor).  Otherwise the value goes to
// prev[j] in sorted order and reaches its place in two coalesced steps (one radix pass on the high bits of perm,
// then sc_prev_place_kernel inside L2-sized windows).
template <bool SCATTER>
__global__ void sc_unpack_keyhead_kernel(int64_t n, const u64* __restrict__ skey, const u32* __restrict__ perm, int umi_bits, int cs_bits,
                                         u32* __restrict__ scell, u64* __restrict__ sumi, u32* __restrict__ scs,
                                         u32* __restrict__ prev, u32* __restrict__ khead_pos) {
    const u64 umi_mask = (1ULL << umi_bits) - 1ULL;           // umi_bits <= 32
    const u32 cs_mask = (u32)((1ULL << cs_bits) - 1ULL);
    SC_LOOP(j, n) {
        const u64 k = skey[j];
        const bool head = (j == 0) || ((skey[j - 1] ^ k) >> cs_bits) != 0;
        scell[j] = (u32)(k >> (umi_bits + cs_bits));
        sumi[j] = (k >> cs_bits) & umi_mask;
        scs[j] = (u32)k & cs_mask;
        const u32 pv = head ? SC_NONE : perm[j - 1];
        if (SCATTER) prev[perm[j]] = pv; else prev[j] = pv;
        khead_pos[j] = head ? (u32)j : 0u;
    }
}
// (position, value) pairs grouped by the high bits of the position: every CTA's stores fall into a few windows of
// 2^shift positions that stay in L2 until their sectors are complete
__global__ void sc_prev_place_kernel(int64_t n, const u32* __restrict__ at, const u32* __restrict__ val, u32* __restrict__ prev) {
    // grid-stride: at any moment the whole grid works inside one or two windows
    SC_LOOP(t, n) prev[at[t]] = val[t];
}
__global__ void sc_gather_cs_kernel(int64_t n, const u32* __restrict__ perm, const uint4* __restrict__ frag, u32* __restrict__ scs) {
    SC_LOOP(j, n) scs[j] = __ldg(&frag[perm[j]].x);
}
// UMI codes are 3 bits per character (reads.py: A 1, C 2, G 3, N 4, T 5, 0 = end), left aligned in 63 bits.
// When every UMI has exactly L characters over {A, C, G, T} the same order is kept by 2 bits per
// character, and the sort key shrinks from 64 to 32 bits.  Anything else raises *bad.
__global__ void sc_umi_pack2_kernel(int64_t n, const u64* __restrict__ umi, int L, u32* __restrict__ key32, u32* __restrict__ bad) {
    bool any_bad = false;
    SC_LOOP(i, n) {
        const u64 code = umi[i];
        u32 k = 0;
        bool ok = (code & ((1ULL << (3 * (21 - L))) - 1ULL)) == 0;
        for (int j = 0; j < L; ++j) {
            const u32 g = (u32)(code >> (3 * (20 - j))) & 7u;
            const u32 m = g == 1u ? 0u : g == 2u ? 1u : g == 3u ? 2u : 3u;
            ok &= (g == 1u) | (g == 2u) | (g == 3u) | (g == 5u);
            k = (k << 2) | m;
        }
        key32[i] = k;
        any_bad |= !ok;
    }
    if (__any_sync(0xFFFFFFFFu, any_bad) && (threadIdx.x & 31) == 0) atomicOr(bad, 1u);
}
template <class T>
__global__ void sc_gather_kernel(int64_t n, const u32* __restrict__ perm, const T* __restrict__ src, T* __restrict__ dst) {
    SC_LOOP(j, n) dst[j] = src[perm[j]];
}
// fragment columns in sorted (cell, umi, i) order: one pass of random reads instead of one per use
__global__ void sc_gather3_kernel(int64_t n, const u32* __restrict__ perm, const uint4* __restrict__ frag,
                                  u32* __restrict__ scs, int32_t* __restrict__ sleft, int32_t* __restrict__ srite) {
    SC_LOOP(j, n) {
        const uint4 f = __ldg(frag + perm[j]);
        scs[j] = f.x;
        sleft[j] = (int32_t)f.y;
        srite[j] = (int32_t)f.z;
    }
}
template <class T>
__global__ void sc_fill_kernel(int64_t n, T* __restrict__ v, T x) { SC_LOOP(i, n) v[i] = x; }

// sorted order j by (cell, umi, i): key-group heads and prev[i] = previous survivor with the same key
__global__ void sc_keyhead_kernel(int64_t n, const u32* __restrict__ perm, const u32* __restrict__ scell, const u64* __restrict__ sumi,
                                  u32* __restrict__ prev, u32* __restrict__ khead_pos) {
    SC_LOOP(j, n) {
        const bool head = (j == 0) || scell[j] != scell[j - 1] || sumi[j] != sumi[j - 1];
        prev[perm[j]] = head ? SC_NONE : perm[j - 1];
        khead_pos[j] = head ? (u32)j : 0u;
    }
}

// One-GPU bundle boundary search without the flag array: first occurrences per chunk of SC_BCHUNK survivors (one CTA
// per chunk), prefix sum of the few thousand chunk counts on the host, then the exact survivor inside the one chunk
// where the running count reaches bundle_keys.  Reads prev[] once (4 B per survivor) instead of flag + scan + search.
#define SC_BCHUNK 4096
__global__ void __launch_bounds__(256) sc_newkey_count_kernel(int64_t len, int64_t pos, int64_t s, const u32* __restrict__ prev, u32* __restrict__ cnt) {
    __shared__ u32 s_w[8];
    for (int64_t c = blockIdx.x; c * SC_BCHUNK < len; c += gridDim.x) {
        const int64_t k0 = c * SC_BCHUNK, k1 = min(len, k0 + SC_BCHUNK);
        u32 n = 0;
        for (int64_t k = k0 + threadIdx.x; k < k1; k += 256) {
            const u32 p = prev[pos + k];
            n += (p == SC_NONE || (int64_t)p < s) ? 1u : 0u;
        }
        n = (u32)warp_sum((u64)n);
        if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = n;
        __syncthreads();
        if (threadIdx.x == 0) cnt[c] = s_w[0] + s_w[1] + s_w[2] + s_w[3] + s_w[4] + s_w[5] + s_w[6] + s_w[7];
        __syncthreads();
    }
}
// the k in [0, len) (len <= SC_BCHUNK) whose element is the want-th first occurrence (want >= 1); one CTA of 256 threads,
// 16 consecutive elements per thread
__global__ void __launch_bounds__(256) sc_newkey_pick_kernel(int64_t len, int64_t pos, int64_t s, const u32* __restrict__ prev, u32 want, u32* __restrict__ out) {
    __shared__ u32 s_n[256];
    const int64_t k0 = (int64_t)threadIdx.x * (SC_BCHUNK / 256);
    u32 bits = 0, n = 0;
    for (int j = 0; j < SC_BCHUNK / 256; ++j) {
        if (k0 + j < len) {
            const u32 p = prev[pos + k0 + j];
            if (p == SC_NONE || (int64_t)p < s) { bits |= 1u << j; ++n; }
        }
    }
    s_n[threadIdx.x] = n;
    __syncthreads();
    if (threadIdx.x == 0) {
        u32 acc = 0;
        for (int t = 0; t < 256; ++t) { const u32 x = s_n[t]; s_n[t] = acc; acc += x; }
    }
    __syncthreads();
    const u32 before = s_n[threadIdx.x];
    if (want > before && want <= before + n) {
        u32 need = want - before;
        for (int j = 0; j < SC_BCHUNK / 256; ++j)
            if ((bits >> j) & 1u) { if (--need == 0) { *out = (u32)(k0 + j); break; } }
    }
}

// position of survivor i in the job-wide survivor order (multi-GPU: gidx; one GPU: i itself)
__device__ __forceinline__ int64_t sc_pos(const u64* __restrict__ gidx, u32 i) { return gidx ? (int64_t)gidx[i] : (int64_t)i; }

__device__ __forceinline__ int sc_bundle_of(const int64_t* __restrict__ bstart, int n_b, int64_t i) {
    int lo = 0, hi = n_b;                     // last b with bstart[b] <= i
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (bstart[mid] <= i) lo = mid; else hi = mid;
    }
    return lo;
}

// ---- multi-GPU exchange: survivors packed as 32-byte records, grouped by owner rank (cell % world),
// file order kept inside each group.  One warp owns a contiguous run of `per_warp` survivors.
struct __align__(16) ScRecord { u64 umi; u64 gidx; u32 cell; u32 cs; int32_t left; int32_t rite; };
#define SC_MAX_WORLD 8

__global__ void sc_part_count_kernel(int64_t n, int world, int64_t per_warp, int n_warps, const u32* __restrict__ cell, u32* __restrict__ counts) {
    const int lane = threadIdx.x & 31;
    for (int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < n_warps; w += (gridDim.x * blockDim.x) >> 5) {
        u32 cnt[SC_MAX_WORLD];
#pragma unroll
        for (int d = 0; d < SC_MAX_WORLD; ++d) cnt[d] = 0;
        const int64_t lo = (int64_t)w * per_warp, hi = min(n, lo + per_warp);
        for (int64_t i = lo + lane; i < hi; i += 32) {
            const int dst = (int)(cell[i] % (u32)world);
#pragma unroll
            for (int d = 0; d < SC_MAX_WORLD; ++d) cnt[d] += dst == d;
        }
#pragma unroll
        for (int d = 0; d < SC_MAX_WORLD; ++d) {
            const u32 t = (u32)warp_sum((u64)cnt[d]);
            if (lane == 0 && d < world) counts[(size_t)d * n_warps + w] = t;
        }
    }
}

__global__ void sc_part_scatter_kernel(int64_t n, int world, int64_t per_warp, int n_warps, int64_t gidx_base,
                                       const u32* __restrict__ cell, const u64* __restrict__ umi, const uint4* __restrict__ frag,
                                       const u32* __restrict__ offsets, ScRecord* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const u32 lt = (1u << lane) - 1u;
    for (int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < n_warps; w += (gridDim.x * blockDim.x) >> 5) {
        u32 off[SC_MAX_WORLD];
#pragma unroll
        for (int d = 0; d < SC_MAX_WORLD; ++d) off[d] = d < world ? offsets[(size_t)d * n_warps + w] : 0u;
        const int64_t lo = (int64_t)w * per_warp, hi = min(n, lo + per_warp);
        for (int64_t base = lo; base < hi; base += 32) {
            const int64_t i = base + lane;
            const bool live = i < hi;
            const u32 c = live ? cell[i] : 0u;
            const int dst = live ? (int)(c % (u32)world) : -1;
            u32 pos = 0;
#pragma unroll
            for (int d = 0; d < SC_MAX_WORLD; ++d) {
                const u32 m = __ballot_sync(0xFFFFFFFFu, dst == d);
                if (dst == d) pos = off[d] + __popc(m & lt);
                off[d] += __popc(m);
            }
            if (live) {
                ScRecord r;
                const uint4 f = frag[i];
                r.umi = umi[i]; r.gidx = (u64)(gidx_base + i); r.cell = c; r.cs = f.x; r.left = (int32_t)f.y; r.rite = (int32_t)f.z;
                out[pos] = r;
            }
        }
    }
}

__global__ void sc_unpack_kernel(int64_t n, const ScRecord* __restrict__ in, u32* __restrict__ cell, u64* __restrict__ umi,
                                 uint4* __restrict__ frag, u64* __restrict__ gidx) {
    SC_LOOP(i, n) {
        const ScRecord r = in[i];
        cell[i] = r.cell; umi[i] = r.umi; frag[i] = make_uint4(r.cs, (u32)r.left, (u32)r.rite, 0u); gidx[i] = r.gidx;
    }
}

// first index with gidx >= x (gidx ascending)
__global__ void sc_lower_bound_kernel(int64_t n, const u64* __restrict__ gidx, u64 x0, u64 x1, int64_t* __restrict__ out) {
    if (blockIdx.x || threadIdx.x > 1) return;
    const u64 x = threadIdx.x ? x1 : x0;
    int64_t a = 0, b = n;
    while (a < b) { const int64_t m = (a + b) >> 1; if (gidx[m] < x) a = m + 1; else b = m; }
    out[threadIdx.x] = a;
}

// multi-GPU bundle boundary search: histogram of the first-in-bundle records (bundle start S) whose
// position falls in [lo, lo + n_bins * width)
__global__ void sc_newkey_hist_kernel(const int64_t* __restrict__ range, const u64* __restrict__ gidx, const u32* __restrict__ prev, int64_t S, int64_t lo,
                                      int64_t width, int n_bins, u64* __restrict__ hist) {
    const int64_t i0 = range[0], n = range[1];          // survivors with lo <= gidx < lo + n_bins * width
    for (int64_t i = i0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t g = (int64_t)gidx[i];
        if (g < lo) continue;
        const int64_t b = (g - lo) / width;
        if (b >= n_bins) continue;
        const u32 p = prev[i];
        if (p == SC_NONE || (int64_t)gidx[p] < S) atomicAdd(hist + b, 1ULL);
    }
}

// segment heads: (cell, umi, bundle) changes
__global__ void sc_seghead_kernel(int64_t n, const u32* __restrict__ perm, const u64* __restrict__ gidx, const u32* __restrict__ khead_pos,
                                  const int64_t* __restrict__ bstart, int n_b, u32* __restrict__ bundle, u32* __restrict__ shead_pos) {
    SC_LOOP(j, n) {
        const u32 b = (u32)sc_bundle_of(bstart, n_b, sc_pos(gidx, perm[j]));
        bundle[j] = b;
        bool head = (j == 0) || khead_pos[j] == (u32)j;
        if (!head) head = (u32)sc_bundle_of(bstart, n_b, sc_pos(gidx, perm[j - 1])) != b;
        shead_pos[j] = head ? (u32)j : 0u;
    }
}

// per element: already-seen / raw counts (te_count.py:444-473), per (bundle, cell) tables
__global__ void sc_segstat_kernel(int64_t n, int64_t n_wl, const u32* __restrict__ perm, const u64* __restrict__ gidx, const u32* __restrict__ scell, const u64* __restrict__ sumi,
                                  const u32* __restrict__ cs, const u32* __restrict__ shead_pos, const u32* __restrict__ bundle,
                                  u32* __restrict__ raw, u32* __restrict__ first_i, u64* __restrict__ minumi, u32* __restrict__ present,
                                  u64* __restrict__ stats) {
    u32 n_seen = 0, n_seg = 0;
    SC_LOOP(j, n) {
        const u32 h = shead_pos[j];
        const u32 c = scell[j];
        if (h == (u32)j) {
            n_seg++;
            atomicAdd(raw + c, 1u);                                                    // :471-473
            atomicMin(first_i + c, (u32)sc_pos(gidx, perm[j]));
            const int64_t bc = (int64_t)bundle[j] * n_wl + c;
            atomicMin(minumi + bc, sumi[j]);
            present[bc] = 1u;
        } else if (cs[j] == cs[h]) {                                                  // cs in sorted order
            n_seen++;                                                                  // :452-454
        } else {
            atomicAdd(raw + c, 1u);                                                    // :459-462
        }
    }
    const u64 a = warp_sum(n_seen), b = warp_sum(n_seg);
    if ((threadIdx.x & 31) == 0) {
        if (a) atomicAdd(stats + TEC_SS_ALREADY_SEEN, a);
        if (b) atomicAdd(stats + TEC_SS_SEGMENTS, b);
    }
}

// Part 2 cell choice (te_count.py:502): key = raw count descending, first appearance ascending
__global__ void sc_cellkey_kernel(int64_t n_wl, const u32* __restrict__ raw, const u32* __restrict__ first_i, u64* __restrict__ key,
                                  u32* __restrict__ id, u64* __restrict__ stats) {
    u32 n_raw = 0;
    SC_LOOP(c, n_wl) {
        const u32 r = raw[c];
        key[c] = ((u64)(~r) << 32) | (r ? first_i[c] : 0xFFFFFFFFu);
        id[c] = (u32)c;
        n_raw += r != 0;
    }
    const u64 a = warp_sum(n_raw);
    if ((threadIdx.x & 31) == 0 && a) atomicAdd(stats + TEC_SS_RAW_BARCODES, a);
}
__global__ void sc_todo_kernel(int64_t n_take, const u64* __restrict__ skey, const u32* __restrict__ sid, u32* __restrict__ todo, int* __restrict__ todo_or_neg) {
    SC_LOOP(k, n_take) {
        if ((u32)(skey[k] >> 32) == 0xFFFFFFFFu) continue;        // raw count 0: never in self.barcodes
        todo[sid[k]] = 1u;
        todo_or_neg[sid[k]] = (int)sid[k];
    }
}

// kept lines (held-line scan of te_count.py:519-541) and the winner of each key group (:552-555)
__global__ void sc_keep_kernel(int64_t n, int64_t n_wl, const u32* __restrict__ scell, const u64* __restrict__ sumi,
                               const u32* __restrict__ shead_pos, const u32* __restrict__ khead_pos, const u32* __restrict__ bundle,
                               const u32* __restrict__ todo, const int* __restrict__ prevtodo, const u64* __restrict__ minumi,
                               const u32* __restrict__ present_excl, u32* __restrict__ winner_at, u64* __restrict__ stats) {
    u32 n_kept = 0;
    SC_LOOP(j, n) {
        if (shead_pos[j] != (u32)j) continue;
        const u32 c = scell[j];
        if (!todo[c]) continue;
        const int64_t row = (int64_t)bundle[j] * n_wl;
        bool kept = true;
        if (sumi[j] == minumi[row + c]) {
            // first line of cell c in this bundle: kept iff a line of a cell in (prevtodo, c) precedes it
            const int lo = prevtodo[c];                                                // -1: no to-do cell below c
            kept = present_excl[row + c] - present_excl[row + lo + 1] > 0;
        }
        if (kept) {
            n_kept++;
            atomicMin(winner_at + khead_pos[j], (u32)j);
        }
    }
    const u64 a = warp_sum(n_kept);
    if ((threadIdx.x & 31) == 0 && a) atomicAdd(stats + TEC_SS_VALID, a);
}

// ------------------------------------------------------------------------------------ Part 3
// number of features of the chromosome with L <= x (directory + binary search), x may be negative
__device__ __forceinline__ int sc_upper_bound_L(const IndexView& iv, int c, int64_t lo, int n, int x) { return upper_bound_L(iv, c, lo, n, x); }

// feature buckets [L//bs, R//bs] (genelist.py:367-380) meet the query's bucket range [q_lo, q_hi]
__device__ __forceinline__ bool sc_candidate(int Lk, int Rk, int q_lo, int q_hi, int bs) {
    const int lb = Lk / bs, rb = floordiv(Rk, bs);
    return lb <= rb && q_lo <= rb && lb <= q_hi;
}

// calls f(feature) for every feature the reference appends to `result` (te_count.py:617-649), at
// least once per feature
template <class F>
__device__ __forceinline__ void sc_for_each_hit(const IndexView& iv, int c, int left, int rite, F f) {
    const int64_t lo = iv.chrom_off[c];
    const int n = (int)(iv.chrom_off[c + 1] - lo);
    const int bs = iv.bs;
    const int q_lo = floordiv(left - 1, bs), q_hi = floordiv(rite, bs);                // :619-621
    if (q_hi < q_lo) return;                                                           // empty range(): `if buckets_reqd` fails
    // point A: left in [L-1, R]  <=>  L <= left+1 and R >= left
    for (int k = upper_bound_L(iv, c, lo, n, left + 1) - 1; k >= 0; --k) {
        if (__ldg(iv.pmaxR + lo + k) < left) break;
        const int Rk = __ldg(iv.R + lo + k);
        if (Rk >= left) {
            const int Lk = __ldg(iv.L + lo + k);
            if (sc_candidate(Lk, Rk, q_lo, q_hi, bs)) f(lo + k);
        }
    }
    // point B: rite in [L, R+1]  <=>  L <= rite and R >= rite-1
    for (int k = upper_bound_L(iv, c, lo, n, rite) - 1; k >= 0; --k) {
        if (__ldg(iv.pmaxR + lo + k) < rite - 1) break;
        const int Rk = __ldg(iv.R + lo + k);
        if (Rk >= rite - 1) {
            const int Lk = __ldg(iv.L + lo + k);
            if (Lk <= left + 1 && Rk >= left) continue;                                // seen under point A
            if (sc_candidate(Lk, Rk, q_lo, q_hi, bs)) f(lo + k);
        }
    }
}

#define SC_MAX_PAIRS 24
#define SC_REG_PAIRS 8

struct ScOut {
    u64* pairs;            // ensg << 32 | cell, appended
    u32* n_pairs;
    u32 cap_pairs;
    u32* cell_hits;        // per whitelist id
    u64* stats;
    u32* overflow;
};

// single-cell cell table: same layout as the bulk table (stab_build.h) over the intervals
// [L-1, R+1) -- left in [L-1, R] or rite in [L, R+1] (te_count.py:645/:648) is a stab query of that
// interval at left or at rite-1 -- with one slot per distinct (ensg, strand) pair.
struct ScTableView {
    StabView sv;                 // sectors / cells / ovf_base / shift (slot_type unused)
    const u32* pair_key;         // slot -> ensg slot << 3 | strand code
    const uint8_t* pair_type;    // slot -> TEC_T_*
    int present;
};

// Result of one fragment (cell, chrom:strand, left, rite), te_count.py:607-686: the (ensg, cell)
// increments it causes are returned to the caller, which appends them warp-aggregated.
struct FragOut {
    u32 n;                       // number of keys
    u32 key[SC_MAX_PAIRS];       // ensg ids
    bool hit, assigned, crash, spilled;
};

__device__ __forceinline__ void sc_append_direct(const ScOut& o, u64 v) {
    const u32 at = atomicAdd(o.n_pairs, 1u);
    if (at < o.cap_pairs) o.pairs[at] = v; else *o.overflow = 1u;
}

__device__ void sc_count_fragment(const IndexView& iv, const ScTableView& tv, int strand_mode, const u32* __restrict__ ensg_of_slot,
                                  u32 cell, u32 cs, int left, int rite, const ScOut& o, FragOut& out) {
    out.n = 0; out.hit = out.assigned = out.crash = out.spilled = false;
    const int c = (int)(cs >> 2);
    const u32 rs = cs & 3u;
    if (!chrom_in_index(iv, c)) return;                                                // :614
    u32 typemask = 0, np = 0;
    u32* pairs = out.key;
    bool over = false, missing = false, exact = true;
    if (tv.present && left >= 0 && left < rite) {
        // for left < rite every feature that passes a point test is also in the bucket range (:619-621)
        exact = false;
        u32 pr[SC_REG_PAIRS];                                    // distinct pairs in registers (static indexing only)
#pragma unroll
        for (int i = 0; i < SC_REG_PAIRS; ++i) pr[i] = 0xFFFFFFFFu;
        const uint2 cellr = __ldg(tv.sv.cells + c);
        const int x[2] = {left, rite - 1};
        for (int p = 0; p < 2; ++p) {
            const int k = x[p] >> tv.sv.shift;
            if ((u32)k >= cellr.y) continue;
            if (p == 1 && x[1] == x[0]) continue;
            const u32 r = (u32)x[p] & ((1u << tv.sv.shift) - 1);
            const u32 prim = cellr.x + (u32)k;
            u32 sec = prim;
            const PointK pk = make_point(r), pn = make_point(R_NONE);
            for (;;) {
                const Sector sct = ld_sector(tv.sv.sectors, sec);
                u32 hit = sector_hits(sct, pk, pn);
                while (hit) {
                    const u32 low = hit & (0u - hit);
                    hit ^= low;
                    const u32 word = (low & 0x80008000u) ? sct.w[6] : ((low & 0x40004000u) ? sct.w[7] : sct.w[5]);
                    const u32 slot = (low & 0xFFFF2000u) ? (word >> 16) : (word & 0xFFFFu);
                    const u32 key = __ldg(tv.pair_key + slot);
                    bool found = false;
#pragma unroll
                    for (int i = 0; i < SC_REG_PAIRS; ++i) found |= pr[i] == key;
                    if (!found) {
#pragma unroll
                        for (int i = 0; i < SC_REG_PAIRS; ++i) if ((u32)i == np) pr[i] = key;
                        ++np;                                    // np > SC_REG_PAIRS: overflow
                        typemask |= 1u << __ldg(tv.pair_type + slot);
                        missing |= (key & 7u) == 7u;
                    }
                }
                if (!sector_more(sct) || r < sector_last_s(sct)) break;
                sec = (sec == prim) ? __ldg(tv.sv.ovf_base + (prim >> 7)) + sector_link(sct) : sec + 1;
            }
        }
        if (np > SC_REG_PAIRS) { exact = true; typemask = 0; np = 0; missing = false; }
        else {
#pragma unroll
            for (int i = 0; i < SC_REG_PAIRS; ++i) if ((u32)i < np) pairs[i] = pr[i];
        }
    }
    if (exact) {
        sc_for_each_hit(iv, c, left, rite, [&](int64_t fi) {
            const u32 w = __ldg(iv.info + fi);
            typemask |= 1u << info_type(w);
            const u32 fs = info_strand(w);
            missing |= fs == 7u;
            const u32 key = (info_ensg(w) << 3) | fs;                                  // (ensg, strand) of :661
            bool found = false;
            for (u32 i = 0; i < np; ++i) found |= pairs[i] == key;
            if (!found) { if (np < SC_MAX_PAIRS) pairs[np++] = key; else over = true; }
        });
    }
    if (!typemask) return;
    out.hit = true;                                                                    // :653-655
    if (missing) { out.crash = true; return; }                                         // :661 KeyError
    const bool gene = typemask & (1u << TEC_T_GENE);
    if (!gene && !(typemask & ((1u << TEC_T_TE) | (1u << TEC_T_ENHANCER)))) return;    // :684
    out.assigned = true;                                                               // :686
    if (!over) {
        u32 m = 0;
        for (u32 i = 0; i < np; ++i) {
            const u32 key = pairs[i];
            if (gene && strand_mode && rs != (key & 7u)) continue;                     // :665
            pairs[m++] = ensg_of_slot[key >> 3];
        }
        out.n = m;
        return;
    }
    // more distinct pairs than the list holds: append directly, a hit iff no earlier hit has the same pair
    out.spilled = true;
    int h = 0;
    sc_for_each_hit(iv, c, left, rite, [&](int64_t fi) {
        const u32 w = __ldg(iv.info + fi);
        const u32 key = (info_ensg(w) << 3) | info_strand(w);
        int j = 0;
        bool dup = false;
        sc_for_each_hit(iv, c, left, rite, [&](int64_t fj) {
            if (j++ >= h || dup) return;
            const u32 w2 = __ldg(iv.info + fj);
            if (((info_ensg(w2) << 3) | info_strand(w2)) == key) dup = true;
        });
        if (!dup && !(gene && strand_mode && rs != (key & 7u)))
            sc_append_direct(o, ((u64)ensg_of_slot[key >> 3] << 32) | cell);
        ++h;
    });
}

// winners compacted into a dense list, so that every lane of sc_part3_kernel has a fragment to count
// one thread per winning segment; all columns are in sorted (cell, umi, i) order.  The increments of
// a warp's fragments are appended with one atomic per warp.
__global__ void sc_part3_kernel(int64_t n, int64_t n_win, const u32* __restrict__ wlist, IndexView iv, ScTableView tv, int strand_mode,
                                const u32* __restrict__ ensg_of_slot, const u32* __restrict__ scell, const u32* __restrict__ shead_pos,
                                const u32* __restrict__ cs, const u32* __restrict__ perm, const uint4* __restrict__ frag, ScOut o) {
    // the coordinates of a fragment are read where they lie (file order) through perm: only the winners' heads, and the
    // rare fragments of a line on another chrom:strand, need them
    auto left = [&](int64_t jj) { return (int)__ldg(&frag[perm[jj]].y); };
    auto rite = [&](int64_t jj) { return (int)__ldg(&frag[perm[jj]].z); };
    const int lane = threadIdx.x & 31;
    u32 n_assigned = 0, n_crash = 0;
    const int64_t n_round = ((n_win + 31) / 32) * 32;            // whole warps stay in the loop together
    SC_LOOP(w, n_round) {
        FragOut fo;
        fo.n = 0;
        const bool win = w < n_win;
        const int64_t j = win ? (int64_t)wlist[w] : 0;
        u32 cell = 0;
        if (win) {
            cell = scell[j];
            const u32 cs0 = cs[j];
            sc_count_fragment(iv, tv, strand_mode, ensg_of_slot, cell, cs0, left(j), rite(j), o, fo);
            if (fo.hit) atomicAdd(o.cell_hits + cell, 1u);
            n_assigned += fo.assigned;
            n_crash += fo.crash;
        }
        // warp-aggregated append of the head fragments' increments
        u32 incl = fo.n;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const u32 t = __shfl_up_sync(0xFFFFFFFFu, incl, d);
            if (lane >= d) incl += t;
        }
        const u32 total = __shfl_sync(0xFFFFFFFFu, incl, 31);
        if (total) {
            u32 base = 0;
            if (lane == 31) base = atomicAdd(o.n_pairs, total);
            base = __shfl_sync(0xFFFFFFFFu, base, 31) + incl - fo.n;
            for (u32 i = 0; i < fo.n; ++i) {
                if (base + i < o.cap_pairs) o.pairs[base + i] = ((u64)fo.key[i] << 32) | cell;
                else *o.overflow = 1u;
            }
        }
        if (!win) continue;
        // other chrom:strand values of the line: the distinct fragment whose first occurrence is latest
        const u32 cs0 = cs[j];
        int64_t e = j + 1;
        while (e < n && shead_pos[e] != (u32)e) ++e;
        for (int64_t a = e - 1; a > j; --a) {
            const u32 csa = cs[a];
            if (csa == cs0) continue;
            const int la = left(a), ra = rite(a);
            bool first = true;                       // first occurrence of this exact fragment?
            for (int64_t b = j + 1; b < a && first; ++b)
                first = !(cs[b] == csa && left(b) == la && rite(b) == ra);
            if (!first) continue;
            bool later = false;                      // a later first occurrence with the same chrom:strand wins
            for (int64_t b = a + 1; b < e && !later; ++b) {
                if (cs[b] != csa) continue;
                bool fb = true;
                for (int64_t d = j + 1; d < b && fb; ++d)
                    fb = !(cs[d] == csa && left(d) == left(b) && rite(d) == rite(b));
                later = fb;
            }
            if (later) continue;
            FragOut f2;
            sc_count_fragment(iv, tv, strand_mode, ensg_of_slot, cell, csa, la, ra, o, f2);
            if (f2.hit) atomicAdd(o.cell_hits + cell, 1u);
            n_assigned += f2.assigned;
            n_crash += f2.crash;
            for (u32 i = 0; i < f2.n; ++i) sc_append_direct(o, ((u64)f2.key[i] << 32) | cell);
        }
    }
    const u64 a_sum = warp_sum((u64)n_assigned), c_sum = warp_sum((u64)n_crash);
    if (lane == 0) {
        if (a_sum) atomicAdd(o.stats + TEC_SS_ASSIGNED, a_sum);
        if (c_sum) atomicAdd(o.stats + TEC_SS_CRASH_STRAND, c_sum);
    }
}

__global__ void sc_split_kernel(int64_t n, const u64* __restrict__ key, const u32* __restrict__ cnt, int32_t* __restrict__ ensg,
                                u32* __restrict__ cell, int64_t* __restrict__ count) {
    SC_LOOP(i, n) {
        ensg[i] = (int32_t)(key[i] >> 32);
        cell[i] = (u32)key[i];
        count[i] = cnt[i];
    }
}
__global__ void sc_hitcells_kernel(int64_t n_wl, const u32* __restrict__ hits, const u32* __restrict__ excl, u32* __restrict__ cell, int64_t* __restrict__ count) {
    SC_LOOP(c, n_wl) {
        if (!hits[c]) continue;
        cell[excl[c]] = (u32)c;
        count[excl[c]] = hits[c];
    }
}
__global__ void sc_nonzero_kernel(int64_t n, const u32* __restrict__ v, u32* __restrict__ f) { SC_LOOP(i, n) f[i] = v[i] != 0; }
__global__ void sc_selkey_kernel(int64_t n, const u32* __restrict__ cell, const int64_t* __restrict__ count, u64* __restrict__ key) {
    SC_LOOP(i, n) key[i] = ((u64)(~(u32)count[i]) << 32) | cell[i];
}

// ------------------------------------------------------------------------------------ ABI
extern "C" int tec_sc_begin(tec_ctx* ctx, int qual, int strand, int64_t n_whitelist) {
    if (!ctx) return TEC_ERR_ARG;
    if (!ctx->has_index) TEC_FAIL(TEC_ERR_STATE, "tec_sc_begin: no index uploaded");
    if (n_whitelist < 0 || n_whitelist >= (int64_t)0xFFFFFFFF) TEC_FAIL(TEC_ERR_ARG, "tec_sc_begin: bad whitelist size");
    TEC_CUDA(cudaSetDevice(ctx->device));
    if (!ctx->sc) ctx->sc = new ScState();
    ScState* s = ctx->sc;
    sc_free_results(ctx, s);
    s->qual = qual; s->strand = strand ? 1 : 0; s->n_wl = n_whitelist;
    s->n = 0; s->n_bound = 0; s->n_pending = false; s->units = 0; s->active = true; s->finalized = false; s->has_gidx = false;
    if (!s->d_n) TEC_CUDA(cudaMalloc(&s->d_n, 24));
    TEC_CUDA(cudaMemsetAsync(s->d_n, 0, 24, ctx->stream));
    s->or_tracked = true;
    if (!s->d_stats) TEC_CUDA(cudaMalloc(&s->d_stats, TEC_SC_NSTATS * 8));
    TEC_CUDA(cudaMemsetAsync(s->d_stats, 0, TEC_SC_NSTATS * 8, ctx->stream));
    memset(s->stats, 0, sizeof(s->stats));
    return TEC_OK;
}

template <class T>
static cudaError_t sc_grow(T** p, int64_t old_n, int64_t new_cap, cudaStream_t st) {
    T* q = nullptr;
    cudaError_t e = cudaMalloc(&q, (size_t)new_cap * sizeof(T));
    if (e != cudaSuccess) return e;
    if (old_n) e = cudaMemcpyAsync(q, *p, (size_t)old_n * sizeof(T), cudaMemcpyDeviceToDevice, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cudaFree(*p);
    *p = q;
    return e;
}

// the exact number of survivors (pushes only advance a device counter)
static int sc_sync_count(tec_ctx* ctx) {
    ScState* s = ctx->sc;
    if (!s->n_pending) return TEC_OK;
    u64 h = 0;
    TEC_CUDA(cudaMemcpyAsync(&h, s->d_n, 8, cudaMemcpyDeviceToHost, ctx->stream));
    TEC_CUDA(cudaStreamSynchronize(ctx->stream));
    s->n = (int64_t)h;
    s->n_pending = false;
    return TEC_OK;
}

static int sc_ingest_dev(tec_ctx* ctx, int64_t n, const int32_t* start, const int32_t* end, const uint16_t* chrom,
                         const uint8_t* mapq, const uint8_t* flag, const u32* cell, const u64* umi) {
    ScState* s = ctx->sc;
    if (n >= (int64_t)0x7FFFFFFF) TEC_FAIL(TEC_ERR_LIMIT, "tec_sc_push: more than 2^31 records in one push");
    if (s->n_bound + n >= (int64_t)0xFFFFFFF0) TEC_FAIL(TEC_ERR_LIMIT, "single-cell path holds at most 2^32 records per GPU");
    if (n + 1 > s->pos_cap) {
        TEC_CUDA(cudaStreamSynchronize(ctx->stream));
        cudaFree(s->pos);
        s->pos = nullptr; s->pos_cap = 0;
        TEC_CUDA(cudaMalloc(&s->pos, (size_t)(2 * n + 4) * 4));
        s->pos_cap = n + 1;
    }
    u32* keep = s->pos;                 // [n]  flags, then their exclusive scan
    u32* lastflag = s->pos + n;         // [1]  copy of keep[n-1]
    u32* total = s->pos + n + 1;        // [1]
    if (!(((uintptr_t)chrom & 7) || ((uintptr_t)mapq & 3) || ((uintptr_t)flag & 3) || ((uintptr_t)cell & 15)))
        sc_filter_kernel<true><<<SC_GRID((n + 3) / 4)>>>(n, s->qual, chrom, mapq, flag, cell, keep, s->d_stats);
    else
        sc_filter_kernel<false><<<SC_GRID(n)>>>(n, s->qual, chrom, mapq, flag, cell, keep, s->d_stats);
    ctx->launches++;
    TEC_CUDA(cudaMemcpyAsync(lastflag, keep + n - 1, 4, cudaMemcpyDeviceToDevice, ctx->stream));
    size_t tb = 0;
    TEC_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tb, keep, keep, (int)n, ctx->stream));
    int rc = sc_cub_tmp(ctx, tb);
    if (rc) return rc;
    TEC_CUDA(cub::DeviceScan::ExclusiveSum(s->cub_tmp, tb, keep, keep, (int)n, ctx->stream));
    ctx->launches += 2;
    sc_total_kernel<<<1, 32, 0, ctx->stream>>>(n, keep, lastflag, total);
    ctx->launches++;
    // columns sized for everything pushed so far (an upper bound of the survivors): no host round trip per push
    if (s->n_bound + n > s->cap) {
        int rc2 = sc_sync_count(ctx);
        if (rc2) return rc2;
        const int64_t cap = std::max<int64_t>(s->n_bound + n, s->cap + s->cap / 2 + 1024);
        TEC_CUDA(sc_grow(&s->cell, s->n, cap, ctx->stream));
        TEC_CUDA(sc_grow(&s->umi, s->n, cap, ctx->stream));
        TEC_CUDA(sc_grow(&s->frag, s->n, cap, ctx->stream));
        s->cap = cap;
    }
    sc_scatter_kernel<<<SC_GRID(n)>>>(n, s->strand, s->d_n, s->d_n + 1, keep, total, start, end, chrom, flag, cell, umi,
                                      s->cell, s->umi, s->frag);
    sc_advance_kernel<<<1, 32, 0, ctx->stream>>>(s->d_n, total);
    ctx->launches += 2;
    TEC_CUDA(cudaGetLastError());
    s->n_bound += n;
    s->n_pending = true;
    s->units += n;
    return TEC_OK;
}

extern "C" int tec_sc_push_dev(tec_ctx* ctx, int64_t n_rec, const int32_t* start, const int32_t* end,
                               const uint16_t* chrom, const uint8_t* mapq, const uint8_t* flag,
                               const uint32_t* cell, const uint64_t* umi) {
    if (!ctx) return TEC_ERR_ARG;
    if (!ctx->sc || !ctx->sc->active) TEC_FAIL(TEC_ERR_STATE, "tec_sc_push_dev: tec_sc_begin not called");
    if (n_rec < 0) TEC_FAIL(TEC_ERR_ARG, "tec_sc_push_dev: negative record count");
    if (n_rec == 0) return TEC_OK;
    if (!start || !end || !chrom || !mapq || !flag || !cell || !umi) TEC_FAIL(TEC_ERR_ARG, "tec_sc_push_dev: null array");
    TEC_CUDA(cudaSetDevice(ctx->device));
    TEC_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
    const int64_t chunk = int64_t(1) << 30;
    for (int64_t off = 0; off < n_rec; off += chunk) {
        const int64_t n = std::min(chunk, n_rec - off);
        int rc = sc_ingest_dev(ctx, n, start + off, end + off, chrom + off, mapq + off, flag + off, cell + off, (const u64*)umi + off);
        if (rc) return rc;
    }
    TEC_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
    ctx->timed = true;
    return TEC_OK;
}

extern "C" int tec_sc_push(tec_ctx* ctx, int64_t n_rec, const int32_t* start, const int32_t* end,
                           const uint16_t* chrom, const uint8_t* mapq, const uint8_t* flag,
                           const uint32_t* cell, const uint64_t* umi) {
    if (!ctx) return TEC_ERR_ARG;
    if (!ctx->sc || !ctx->sc->active) TEC_FAIL(TEC_ERR_STATE, "tec_sc_push: tec_sc_begin not called");
    if (n_rec < 0) TEC_FAIL(TEC_ERR_ARG, "tec_sc_push: negative record count");
    if (n_rec == 0) return TEC_OK;
    if (!start || !end || !chrom || !mapq || !flag || !cell || !umi) TEC_FAIL(TEC_ERR_ARG, "tec_sc_push: null array");
    TEC_CUDA(cudaSetDevice(ctx->device));
    const int64_t chunk = TEC_STAGE_RECORDS;
    int rc = ctx->ensure_stage(std::min<int64_t>(n_rec, chunk), /*sc=*/true);
    if (rc) return rc;
    for (int64_t off = 0; off < n_rec; off += chunk) {
        const int64_t n = std::min<int64_t>(chunk, n_rec - off);
        const int sl_i = ctx->stage_next;
        ctx->stage_next ^= 1;
        StageSlot& sl = ctx->stage[sl_i];
        TEC_CUDA(cudaStreamWaitEvent(ctx->copy_stream, ctx->stage_free[sl_i], 0));
        TEC_CUDA(cudaMemcpyAsync(sl.start, start + off, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->copy_stream));
        TEC_CUDA(cudaMemcpyAsync(sl.end, end + off, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->copy_stream));
        TEC_CUDA(cudaMemcpyAsync(sl.chrom, chrom + off, (size_t)n * 2, cudaMemcpyHostToDevice, ctx->copy_stream));
        TEC_CUDA(cudaMemcpyAsync(sl.mapq, mapq + off, (size_t)n, cudaMemcpyHostToDevice, ctx->copy_stream));
        TEC_CUDA(cudaMemcpyAsync(sl.flag, flag + off, (size_t)n, cudaMemcpyHostToDevice, ctx->copy_stream));
        TEC_CUDA(cudaMemcpyAsync(sl.cell, cell + off, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->copy_stream));
        TEC_CUDA(cudaMemcpyAsync(sl.umi, umi + off, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->copy_stream));
        TEC_CUDA(cudaEventRecord(ctx->stage_ready[sl_i], ctx->copy_stream));
        TEC_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->stage_ready[sl_i], 0));
        rc = sc_ingest_dev(ctx, n, sl.start, sl.end, sl.chrom, sl.mapq, sl.flag, sl.cell, sl.umi);
        if (rc) return rc;
        TEC_CUDA(cudaEventRecord(ctx->stage_free[sl_i], ctx->stream));
    }
    TEC_CUDA(cudaStreamSynchronize(ctx->copy_stream));
    return TEC_OK;
}

// all-reduce of a device buffer over the ranks (no-op on one GPU); dtype 0 u32, 1 u64, 2 i64; op 0 sum, 1 min, 2 max
static int sc_allreduce(tec_ctx* ctx, void* dev, int64_t count, int dtype, int op) {
    ScState* s = ctx->sc;
    if (s->world <= 1) return TEC_OK;
    if (!s->coll) return ctx->comm ? comm_allreduce(ctx, dev, count, dtype, op) : TEC_OK;      // NCCL on the library's stream: no host round trip
    TEC_CUDA(cudaStreamSynchronize(ctx->stream));
    if (s->coll(s->coll_user, dev, count, dtype, op) != 0) TEC_FAIL(TEC_ERR_STATE, "single-cell collective callback failed");
    return TEC_OK;
}

#define SC_HIST_BINS 16384

// bundle starts in job-wide survivor positions, identical on every rank (te_count.py:377)
static int sc_bundles_global(tec_ctx* ctx, ScArena& A, int64_t N, const u32* prev, int64_t bundle_keys, std::vector<int64_t>& bstart, int64_t& g_end) {
    ScState* s = ctx->sc;
    u64* hist = nullptr;
    TEC_CUDA(A.get(&hist, SC_HIST_BINS + 1));
    // G = number of survivors of the whole job
    u64 h_last = 0;
    if (N) TEC_CUDA(cudaMemcpyAsync(&h_last, s->gidx + N - 1, 8, cudaMemcpyDeviceToHost, ctx->stream));
    TEC_CUDA(cudaStreamSynchronize(ctx->stream));
    u64 h_end = N ? h_last + 1 : 0;
    TEC_CUDA(cudaMemcpyAsync(hist, &h_end, 8, cudaMemcpyHostToDevice, ctx->stream));
    int rc = sc_allreduce(ctx, hist, 1, 1, 2);
    if (rc) return rc;
    TEC_CUDA(cudaMemcpyAsync(&h_end, hist, 8, cudaMemcpyDeviceToHost, ctx->stream));
    TEC_CUDA(cudaStreamSynchronize(ctx->stream));
    const int64_t G = (int64_t)h_end;
    g_end = G;
    std::vector<u64> h_hist(SC_HIST_BINS);
    int64_t* d_range = nullptr;
    TEC_CUDA(A.get(&d_range, 2));
    // histogram of the first-in-bundle survivors with lo <= position < lo + span (all ranks), into h_hist
    auto histogram = [&](int64_t S, int64_t lo, int64_t span, int64_t& width) -> int {
        width = (span + SC_HIST_BINS - 1) / SC_HIST_BINS;
        TEC_CUDA(cudaMemsetAsync(hist, 0, SC_HIST_BINS * 8, ctx->stream));
        // only the local survivors inside the window are read (positions are ascending)
        sc_lower_bound_kernel<<<1, 32, 0, ctx->stream>>>(N, s->gidx, (u64)lo, (u64)(lo + span), d_range);
        const int64_t guess = std::max<int64_t>(1, std::min<int64_t>(N, span / std::max(1, s->world) * 2 + 65536));
        sc_newkey_hist_kernel<<<SC_GRID(guess)>>>(d_range, s->gidx, prev, S, lo, width, SC_HIST_BINS, hist);
        ctx->launches += 2;
        int rc2 = sc_allreduce(ctx, hist, SC_HIST_BINS, 1, 0);
        if (rc2) return rc2;
        TEC_CUDA(cudaMemcpyAsync(h_hist.data(), hist, SC_HIST_BINS * 8, cudaMemcpyDeviceToHost, ctx->stream));
        TEC_CUDA(cudaStreamSynchronize(ctx->stream));
        return TEC_OK;
    };
    int64_t S = 0, last_len = 0;
    while (S < G) {
        bstart.push_back(S);
        // a bundle is usually about as long as the one before it: look at windows of twice that length
        int64_t lo = S, need = bundle_keys;
        bool found = false;
        while (lo < G && !found) {
            int64_t span = last_len ? std::min<int64_t>(G - lo, 2 * last_len) : G - lo;
            int64_t width = 1;
            rc = histogram(S, lo, span, width);
            if (rc) return rc;
            int b = 0;
            int64_t cum = 0;
            for (; b < SC_HIST_BINS; ++b) {
                if (cum + (int64_t)h_hist[(size_t)b] >= need) break;
                cum += (int64_t)h_hist[(size_t)b];
            }
            if (b == SC_HIST_BINS) { need -= cum; lo += span; continue; }      // not in this window
            // narrow down inside bin b
            for (;;) {
                if (width == 1) {
                    const int64_t next = lo + b + 1;
                    last_len = next - S;
                    S = next;
                    found = true;
                    break;
                }
                need -= cum;
                lo += (int64_t)b * width;
                span = width;
                rc = histogram(S, lo, span, width);
                if (rc) return rc;
                cum = 0;
                for (b = 0; b < SC_HIST_BINS; ++b) {
                    if (cum + (int64_t)h_hist[(size_t)b] >= need) break;
                    cum += (int64_t)h_hist[(size_t)b];
                }
                if (b == SC_HIST_BINS) TEC_FAIL(TEC_ERR_STATE, "single-cell bundle search lost its key");
            }
        }
        if (!found) break;                                       // fewer than bundle_keys keys left: last bundle
    }
    A.release(hist);
    return TEC_OK;
}

// ---- multi-GPU plumbing (te_counter_b200/dist.py drives it)
extern "C" int tec_sc_set_collective(tec_ctx* ctx, tec_allreduce_fn fn, void* user, int rank, int world) {
    if (!ctx) return TEC_ERR_ARG;
    if (world < 1 || rank < 0 || rank >= world || (world > 1 && !fn)) TEC_FAIL(TEC_ERR_ARG, "tec_sc_set_collective: bad arguments");
    if (!ctx->sc) ctx->sc = new ScState();
    ctx->sc->coll = world > 1 ? fn : nullptr;
    ctx->sc->coll_user = user;
    ctx->sc->rank = rank;
    ctx->sc->world = world;
    return TEC_OK;
}

// number of survivors held after the pushes
extern "C" int tec_sc_survivors(tec_ctx* ctx, int64_t* n) {
    if (!ctx) return TEC_ERR_ARG;
    ScState* s = ctx->sc;
    if (!s || !s->active) TEC_FAIL(TEC_ERR_STATE, "tec_sc_survivors: tec_sc_begin not called");
    TEC_CUDA(cudaSetDevice(ctx->device));
    int rc = sc_sync_count(ctx);
    if (rc) return rc;
    if (n) *n = s->n;
    return TEC_OK;
}

template <class T> static int sc_excl_sum(tec_ctx* ctx, T* in, T* out, int64_t n);

// Pack the survivors as 32-byte records grouped by owner rank (cell % world), file order kept inside a
// group; counts[world] on the host.  The packed buffer lives until the next call / import.
extern "C" int tec_sc_partition_dev(tec_ctx* ctx, int world, int64_t gidx_base, int64_t* counts, void** records) {
    if (!ctx) return TEC_ERR_ARG;
    ScState* s = ctx->sc;
    if (!s || !s->active) TEC_FAIL(TEC_ERR_STATE, "tec_sc_partition_dev: tec_sc_begin not called");
    if (world < 1 || world > SC_MAX_WORLD || !counts || !records) TEC_FAIL(TEC_ERR_ARG, "tec_sc_partition_dev: 1..8 ranks");
    TEC_CUDA(cudaSetDevice(ctx->device));
    int rc0 = sc_sync_count(ctx);
    if (rc0) return rc0;
    const int64_t N = s->n;
    const int n_warps = (int)std::max<int64_t>(1, std::min<int64_t>((N + 1023) / 1024, (int64_t)ctx->n_sm * 64));
    const int64_t per_warp = ((N + n_warps - 1) / n_warps + 31) / 32 * 32;
    ctx->cache.put(s->packed);
    s->packed = nullptr;
    TEC_CUDA(ctx->cache.get(&s->packed, (size_t)std::max<int64_t>(N, 1) * sizeof(ScRecord)));
    u32* cnt = nullptr;
    ScArena A(ctx->cache);
    TEC_CUDA(A.get(&cnt, (size_t)world * n_warps + 1));
    TEC_CUDA(cudaMemsetAsync(cnt, 0, ((size_t)world * n_warps + 1) * 4, ctx->stream));
    const int blocks = std::max(1, std::min((n_warps + 7) / 8, ctx->n_sm * 8));
    sc_part_count_kernel<<<blocks, 256, 0, ctx->stream>>>(N, world, per_warp, n_warps, s->cell, cnt);
    int rc = sc_excl_sum(ctx, cnt, cnt, (int64_t)world * n_warps + 1);
    if (rc) return rc;
    sc_part_scatter_kernel<<<blocks, 256, 0, ctx->stream>>>(N, world, per_warp, n_warps, gidx_base, s->cell, s->umi, s->frag,
                                                           cnt, (ScRecord*)s->packed);
    ctx->launches += 4;
    std::vector<u32> h((size_t)world + 1);
    for (int d = 0; d <= world; ++d)
        TEC_CUDA(cudaMemcpyAsync(&h[(size_t)d], cnt + (size_t)d * n_warps, 4, cudaMemcpyDeviceToHost, ctx->stream));
    TEC_CUDA(cudaStreamSynchronize(ctx->stream));
    for (int d = 0; d < world; ++d) counts[d] = (int64_t)h[(size_t)d + 1] - (int64_t)h[(size_t)d];
    *records = s->packed;
    return TEC_OK;
}

// Install exchanged records (device pointer, 32 bytes each, ascending in position) as this rank's survivors.
extern "C" int tec_sc_import_packed_dev(tec_ctx* ctx, int64_t n, const void* records) {
    if (!ctx) return TEC_ERR_ARG;
    ScState* s = ctx->sc;
    if (!s || !s->active) TEC_FAIL(TEC_ERR_STATE, "tec_sc_import_packed_dev: tec_sc_begin not called");
    if (n < 0 || n >= (int64_t)0x7FFFFFF0 || (n && !records)) TEC_FAIL(TEC_ERR_ARG, "tec_sc_import_packed_dev: bad arguments");
    TEC_CUDA(cudaSetDevice(ctx->device));
    TEC_CUDA(cudaStreamSynchronize(ctx->stream));
    if (n > s->cap) {
        const int64_t cap = n + 1024;
        TEC_CUDA(sc_grow(&s->cell, 0, cap, ctx->stream));
        TEC_CUDA(sc_grow(&s->umi, 0, cap, ctx->stream));
        TEC_CUDA(sc_grow(&s->frag, 0, cap, ctx->stream));
        s->cap = cap;
    }
    if (n > s->gidx_cap) {
        TEC_CUDA(sc_grow(&s->gidx, 0, n + 1024, ctx->stream));
        s->gidx_cap = n + 1024;
    }
    if (n) sc_unpack_kernel<<<SC_GRID(n)>>>(n, (const ScRecord*)records, s->cell, s->umi, s->frag, s->gidx);
    ctx->launches++;
    TEC_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->cache.put(s->packed);
    s->packed = nullptr;
    s->n = n;
    s->n_bound = n;
    s->n_pending = false;
    TEC_CUDA(cudaMemcpy(s->d_n, &n, 8, cudaMemcpyHostToDevice));
    s->has_gidx = true;
    s->or_tracked = false;
    return TEC_OK;
}

static int ceil_log2_i64(int64_t x) { int b = 0; while ((int64_t(1) << b) < x) ++b; return b; }

template <class K, class V>
static int sc_sort_pairs(tec_ctx* ctx, K* k_in, K* k_out, V* v_in, V* v_out, int64_t n, int b0, int b1) {
    size_t tb = 0;
    TEC_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tb, k_in, k_out, v_in, v_out, (int)n, b0, b1, ctx->stream));
    int rc = sc_cub_tmp(ctx, tb);
    if (rc) return rc;
    TEC_CUDA(cub::DeviceRadixSort::SortPairs(ctx->sc->cub_tmp, tb, k_in, k_out, v_in, v_out, (int)n, b0, b1, ctx->stream));
    ctx->launches += (b1 - b0 + 7) / 8 + 2;
    return TEC_OK;
}

template <class T, class Op>
static int sc_incl_scan(tec_ctx* ctx, T* v, int64_t n, Op op) {
    size_t tb = 0;
    TEC_CUDA(cub::DeviceScan::InclusiveScan(nullptr, tb, v, v, op, (int)n, ctx->stream));
    int rc = sc_cub_tmp(ctx, tb);
    if (rc) return rc;
    TEC_CUDA(cub::DeviceScan::InclusiveScan(ctx->sc->cub_tmp, tb, v, v, op, (int)n, ctx->stream));
    ctx->launches += 2;
    return TEC_OK;
}

// T = u32, or u64 for byte offsets that can pass 4 GiB (sc_mtx.cuh)
template <class T>
static int sc_excl_sum(tec_ctx* ctx, T* in, T* out, int64_t n) {
    size_t tb = 0;
    TEC_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tb, in, out, (int)n, ctx->stream));
    int rc = sc_cub_tmp(ctx, tb);
    if (rc) return rc;
    TEC_CUDA(cub::DeviceScan::ExclusiveSum(ctx->sc->cub_tmp, tb, in, out, (int)n, ctx->stream));
    ctx->launches += 2;
    return TEC_OK;
}

extern "C" int tec_sc_finalize(tec_ctx* ctx, int64_t bundle_keys, int64_t maxcells, int64_t pad,
                               int64_t* n_triples, int64_t* n_hit_cells) {
    if (!ctx) return TEC_ERR_ARG;
    ScState* s = ctx->sc;
    if (!s || !s->active) TEC_FAIL(TEC_ERR_STATE, "tec_sc_finalize: tec_sc_begin not called");
    if (bundle_keys < 1 || maxcells < 0 || pad < 0) TEC_FAIL(TEC_ERR_ARG, "tec_sc_finalize: bad arguments");
    TEC_CUDA(cudaSetDevice(ctx->device));
    TEC_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
    sc_free_results(ctx, s);
    ScArena A(ctx->cache);
    int rc_n = sc_sync_count(ctx);
    if (rc_n) return rc_n;
    const int64_t N = s->n, W = std::max<int64_t>(s->n_wl, 1);
    if (N >= (int64_t)0x7FFFFFF0) TEC_FAIL(TEC_ERR_LIMIT, "single-cell path: more than 2^31 surviving records on one GPU");
    int64_t n_b = 0;
    u32* hits = nullptr;
    TEC_CUDA(A.get(&hits, (size_t)W));
    TEC_CUDA(cudaMemsetAsync(hits, 0, (size_t)W * 4, ctx->stream));
    u32* d_ensg_of_slot = nullptr;
    TEC_CUDA(A.get(&d_ensg_of_slot, ctx->ensg_of_slot.size()));
    if (!ctx->ensg_of_slot.empty())
        TEC_CUDA(cudaMemcpyAsync(d_ensg_of_slot, ctx->ensg_of_slot.data(), ctx->ensg_of_slot.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    u64* pairs_sorted = nullptr;
    u32 h_npairs = 0;
    ctx->sc_last_sort = ctx->sc_last_sort_passes = 0;
    if (N > 0 || s->world > 1) {          // with several ranks every rank walks the same sequence of collectives
        // ---- key groups: survivors in (cell, UMI, file position) order
        u64* d_or = s->d_n + 1;                 // kept up to date by the pushes
        if (!s->or_tracked) {
            TEC_CUDA(cudaMemsetAsync(d_or, 0, 16, ctx->stream));
            sc_or_kernel<<<SC_GRID(N)>>>(N, s->umi, s->frag, d_or);
            ctx->launches++;
        }
        u64 h_or[2] = {0, 0};
        TEC_CUDA(cudaMemcpyAsync(h_or, d_or, 16, cudaMemcpyDeviceToHost, ctx->stream));
        TEC_CUDA(cudaStreamSynchronize(ctx->stream));
        int b0 = 0, b1 = 1;
        if (h_or[0]) { b0 = __builtin_ctzll(h_or[0]); b1 = 64 - __builtin_clzll(h_or[0]); }
        const int umi_len = h_or[0] ? 21 - b0 / 3 : 0;
        const int cs_bits = h_or[1] ? 64 - __builtin_clzll(h_or[1]) : 1;
        const int cell_bits = std::max(1, ceil_log2_i64(W));
        u32 *perm = nullptr, *scell = nullptr, *scs = nullptr, *prev = nullptr, *khead = nullptr;
        u64* sumi = nullptr;
        int rc = TEC_OK;
        bool done = false;
        // (a) one packed 64-bit key per survivor, 11-bit LSD passes of csrc/radix.cuh over its cell and UMI bits; the
        //     chrom:strand word rides in the low bits, so the sorted keys ARE the sorted columns: nothing is gathered
        if (ctx->opt_sc_sort != 0 && umi_len >= 1 && umi_len <= 16 && cell_bits + 2 * umi_len + cs_bits <= 64 && N > 0) {
            u64 *ka = nullptr, *kb = nullptr;
            u32 *va = nullptr, *vb = nullptr, *d_bad = nullptr, *scratch = nullptr;
            const RdxPlan plan = rdx_plan(N, ctx->n_sm);
            TEC_CUDA(A.get(&ka, (size_t)N));
            TEC_CUDA(A.get(&va, (size_t)N));
            TEC_CUDA(A.get(&d_bad, 1));
            TEC_CUDA(cudaMemsetAsync(d_bad, 0, 4, ctx->stream));
            sc_pack_key_kernel<<<SC_GRID(N)>>>(N, s->cell, s->umi, s->frag, umi_len, cs_bits, ka, va, d_bad);
            ctx->launches += 2;
            u32 h_bad = 0;
            TEC_CUDA(cudaMemcpyAsync(&h_bad, d_bad, 4, cudaMemcpyDeviceToHost, ctx->stream));
            TEC_CUDA(cudaStreamSynchronize(ctx->stream));
            if (!h_bad) {
                TEC_CUDA(A.get(&kb, (size_t)N));
                TEC_CUDA(A.get(&vb, (size_t)N));
                TEC_CUDA(A.get(&scratch, plan.counts_bytes / 4));
                bool in_b = false;
                int n_pass = 0;
                TEC_CUDA((rdx_sort<u64, true>(ka, va, kb, vb, N, cs_bits, cs_bits + 2 * umi_len + cell_bits, ctx->n_sm, scratch, ctx->stream, &in_b, &n_pass)));
                ctx->launches += RDX_LAUNCHES_PER_PASS * n_pass;
                ctx->sc_last_sort = 1;
                ctx->sc_last_sort_passes = n_pass;
                const u64* skey = in_b ? kb : ka;
                perm = in_b ? vb : va;
                u32* free_v = in_b ? va : vb;                 // the other half of the ping-pong: free from here on
                u64* free_k = in_b ? ka : kb;
                TEC_CUDA(A.get(&scell, (size_t)N));
                TEC_CUDA(A.get(&sumi, (size_t)N));
                TEC_CUDA(A.get(&scs, (size_t)N));
                TEC_CUDA(A.get(&prev, (size_t)N));
                TEC_CUDA(A.get(&khead, (size_t)N));
                const int pos_bits = std::max(1, ceil_log2_i64(N));
                const int part_bits = std::min(RDX_MAX_BITS, pos_bits);
                if (ctx->opt_sc_prev_partition == 2 || (ctx->opt_sc_prev_partition && pos_bits > RDX_MAX_BITS + 4)) {   // 2: always (tests)
                    // prev[] in file order without 894 M random read-modify-writes of a sector: the values are written in
                    // sorted order, grouped by the top 11 bits of their position (one radix pass) and placed window by window
                    sc_unpack_keyhead_kernel<false><<<SC_GRID(N)>>>(N, skey, perm, 2 * umi_len, cs_bits, scell, sumi, scs, free_v, khead);
                    u32* at = reinterpret_cast<u32*>(free_k);
                    u32* val = at + N;
                    TEC_CUDA((rdx_pass<u32, true>(perm, free_v, at, val, N, pos_bits - part_bits, part_bits, plan, scratch, ctx->stream)));
                    sc_prev_place_kernel<<<SC_GRID(N)>>>(N, at, val, prev);
                    ctx->launches += 2 + RDX_LAUNCHES_PER_PASS;
                } else {
                    sc_unpack_keyhead_kernel<true><<<SC_GRID(N)>>>(N, skey, perm, 2 * umi_len, cs_bits, scell, sumi, scs, prev, khead);
                    ctx->launches++;
                }
                A.release(free_v); A.release(ka); A.release(kb); A.release(scratch);
                done = true;
            } else {
                A.release(ka); A.release(va);
            }
            A.release(d_bad);
        }
        // (b) any other UMI alphabet / length: stable LSD sort of i by UMI, then by cell (library sort), columns gathered
        if (!done) {
            u32 *iota = nullptr, *perm1 = nullptr, *ck = nullptr;
            u64* uk = nullptr;
            TEC_CUDA(A.get(&iota, (size_t)N));
            TEC_CUDA(A.get(&perm1, (size_t)N));
            TEC_CUDA(A.get(&uk, (size_t)N));
            sc_iota_kernel<<<SC_GRID(N)>>>(N, iota);
            // 32-bit keys when every UMI is a fixed-length string over {A, C, G, T} (2 bits per character)
            bool packed = false;
            if (ctx->opt_sc_pack_umi && umi_len >= 1 && umi_len <= 16) {
                u32 *k32 = nullptr, *k32s = nullptr, *d_bad = nullptr;
                TEC_CUDA(A.get(&k32, (size_t)N));
                TEC_CUDA(A.get(&k32s, (size_t)N));
                TEC_CUDA(A.get(&d_bad, 1));
                TEC_CUDA(cudaMemsetAsync(d_bad, 0, 4, ctx->stream));
                sc_umi_pack2_kernel<<<SC_GRID(N)>>>(N, s->umi, umi_len, k32, d_bad);
                ctx->launches++;
                u32 h_bad = 0;
                TEC_CUDA(cudaMemcpyAsync(&h_bad, d_bad, 4, cudaMemcpyDeviceToHost, ctx->stream));
                TEC_CUDA(cudaStreamSynchronize(ctx->stream));
                if (!h_bad) {
                    rc = sc_sort_pairs(ctx, k32, k32s, iota, perm1, N, 0, 2 * umi_len);
                    if (rc) return rc;
                    packed = true;
                }
                A.release(k32); A.release(k32s); A.release(d_bad);
            }
            if (!packed) {
                rc = sc_sort_pairs(ctx, s->umi, uk, iota, perm1, N, b0, b1);
                if (rc) return rc;
            }
            if (N > 0) ctx->sc_last_sort = packed ? 2 : 3;      // a rank without survivors sorts nothing
            A.release(uk); uk = nullptr;
            TEC_CUDA(A.get(&ck, (size_t)N));
            TEC_CUDA(A.get(&scell, (size_t)N));
            sc_gather_kernel<u32><<<SC_GRID(N)>>>(N, perm1, s->cell, ck);
            perm = iota;                          // reuse
            rc = sc_sort_pairs(ctx, ck, scell, perm1, perm, N, 0, cell_bits);
            if (rc) return rc;
            A.release(ck); A.release(perm1);
            TEC_CUDA(A.get(&sumi, (size_t)N));
            sc_gather_kernel<u64><<<SC_GRID(N)>>>(N, perm, s->umi, sumi);
            TEC_CUDA(A.get(&scs, (size_t)N));
            sc_gather_cs_kernel<<<SC_GRID(N)>>>(N, perm, s->frag, scs);
            TEC_CUDA(A.get(&prev, (size_t)N));
            TEC_CUDA(A.get(&khead, (size_t)N));
            sc_keyhead_kernel<<<SC_GRID(N)>>>(N, perm, scell, sumi, prev, khead);
            ctx->launches += 6;
        }
        rc = sc_incl_scan(ctx, khead, N, MaxU32());
        if (rc) return rc;
        // ---- bundle boundaries (te_count.py:377): a bundle closes after the survivor that brings
        //      its number of distinct keys to bundle_keys
        std::vector<int64_t> bstart;
        int64_t g_end = N;
        const u64* gidx = s->has_gidx ? s->gidx : nullptr;
        if (gidx) {
            rc = sc_bundles_global(ctx, A, N, prev, bundle_keys, bstart, g_end);
            if (rc) return rc;
            if (g_end >= (int64_t)0xFFFFFFF0) TEC_FAIL(TEC_ERR_LIMIT, "single-cell path: more than 2^32 surviving records in the job");
        } else {
            // windows of about the length of the bundle before (the first one: 4 x bundle_keys survivors)
            const int64_t WIN0 = std::max<int64_t>(int64_t(1) << 22, std::min<int64_t>(4 * bundle_keys, int64_t(1) << 28));
            const int64_t WMAX = int64_t(1) << 28;
            u32 *f = nullptr, *found = nullptr;
            TEC_CUDA(A.get(&f, (size_t)(WMAX / SC_BCHUNK + 1)));
            TEC_CUDA(A.get(&found, 1));
            std::vector<u32> h_cnt;
            int64_t st = 0, last_len = 0;
            while (st < N) {
                bstart.push_back(st);
                int64_t acc = 0, pos = st, next = N;
                while (pos < N) {
                    const int64_t want_len = last_len ? last_len + last_len / 4 + SC_BCHUNK : WIN0;
                    const int64_t len = std::min(std::min(want_len, WMAX), N - pos);
                    const int64_t n_chunks = (len + SC_BCHUNK - 1) / SC_BCHUNK;
                    sc_newkey_count_kernel<<<(int)std::min<int64_t>(n_chunks, (int64_t)ctx->n_sm * 8), 256, 0, ctx->stream>>>(len, pos, st, prev, f);
                    ctx->launches++;
                    h_cnt.resize((size_t)n_chunks);
                    TEC_CUDA(cudaMemcpyAsync(h_cnt.data(), f, (size_t)n_chunks * 4, cudaMemcpyDeviceToHost, ctx->stream));
                    TEC_CUDA(cudaStreamSynchronize(ctx->stream));
                    int64_t c = 0;
                    for (; c < n_chunks; ++c) {
                        if (acc + h_cnt[(size_t)c] >= bundle_keys) break;
                        acc += h_cnt[(size_t)c];
                    }
                    if (c < n_chunks) {
                        const int64_t cpos = pos + c * SC_BCHUNK, clen = std::min<int64_t>(SC_BCHUNK, pos + len - cpos);
                        sc_newkey_pick_kernel<<<1, 256, 0, ctx->stream>>>(clen, cpos, st, prev, (u32)(bundle_keys - acc), found);
                        ctx->launches++;
                        u32 k = 0;
                        TEC_CUDA(cudaMemcpyAsync(&k, found, 4, cudaMemcpyDeviceToHost, ctx->stream));
                        TEC_CUDA(cudaStreamSynchronize(ctx->stream));
                        next = cpos + k + 1;
                        break;
                    }
                    pos += len;
                }
                last_len = next - st;
                st = next;
            }
            A.release(f);
        }
        n_b = (int64_t)bstart.size();
        bstart.push_back(g_end);
        if (n_b * W > (int64_t(1) << 31)) TEC_FAIL(TEC_ERR_LIMIT, "single-cell path: bundles x whitelist exceeds 2^31 table entries");
        int64_t* d_bstart = nullptr;
        TEC_CUDA(A.get(&d_bstart, bstart.size()));
        TEC_CUDA(cudaMemcpyAsync(d_bstart, bstart.data(), bstart.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
        A.release(prev);
        // ---- segments, raw counts, per (bundle, cell) tables
        u32 *bundle = nullptr, *shead = nullptr, *raw = nullptr, *first_i = nullptr, *present = nullptr;
        u64* minumi = nullptr;
        TEC_CUDA(A.get(&bundle, (size_t)N));
        TEC_CUDA(A.get(&shead, (size_t)N));
        sc_seghead_kernel<<<SC_GRID(N)>>>(N, perm, gidx, khead, d_bstart, (int)n_b, bundle, shead);
        rc = sc_incl_scan(ctx, shead, N, MaxU32());
        if (rc) return rc;
        TEC_CUDA(A.get(&raw, (size_t)W));
        TEC_CUDA(A.get(&first_i, (size_t)W));
        TEC_CUDA(A.get(&present, (size_t)(n_b * W + 1)));
        TEC_CUDA(A.get(&minumi, (size_t)(n_b * W)));
        TEC_CUDA(cudaMemsetAsync(raw, 0, (size_t)W * 4, ctx->stream));
        TEC_CUDA(cudaMemsetAsync(first_i, 0xFF, (size_t)W * 4, ctx->stream));
        TEC_CUDA(cudaMemsetAsync(present, 0, (size_t)(n_b * W + 1) * 4, ctx->stream));
        TEC_CUDA(cudaMemsetAsync(minumi, 0xFF, (size_t)(n_b * W) * 8, ctx->stream));
        sc_segstat_kernel<<<SC_GRID(N)>>>(N, W, perm, gidx, scell, sumi, scs, shead, bundle, raw, first_i, minumi, present, s->d_stats);
        rc = sc_allreduce(ctx, raw, W, 0, 0);
        if (rc) return rc;
        rc = sc_allreduce(ctx, first_i, W, 0, 1);
        if (rc) return rc;
        rc = sc_allreduce(ctx, present, n_b * W + 1, 0, 2);
        if (rc) return rc;
        ctx->launches += 2;
        // ---- Part 2: the maxcells + pad cells with the most raw reads, ties by first appearance
        u64 *ckey = nullptr, *ckey_s = nullptr;
        u32 *cid = nullptr, *cid_s = nullptr, *todo = nullptr;
        int* prevtodo = nullptr;
        TEC_CUDA(A.get(&ckey, (size_t)W));
        TEC_CUDA(A.get(&ckey_s, (size_t)W));
        TEC_CUDA(A.get(&cid, (size_t)W));
        TEC_CUDA(A.get(&cid_s, (size_t)W));
        TEC_CUDA(A.get(&todo, (size_t)W));
        TEC_CUDA(A.get(&prevtodo, (size_t)W + 1));
        sc_cellkey_kernel<<<SC_GRID(W)>>>(W, raw, first_i, ckey, cid, s->d_stats);
        rc = sc_sort_pairs(ctx, ckey, ckey_s, cid, cid_s, W, 0, 64);
        if (rc) return rc;
        TEC_CUDA(cudaMemsetAsync(todo, 0, (size_t)W * 4, ctx->stream));
        TEC_CUDA(cudaMemsetAsync(prevtodo, 0xFF, (size_t)(W + 1) * 4, ctx->stream));      // -1
        const int64_t n_take = std::min<int64_t>(W, maxcells + pad);
        if (n_take) sc_todo_kernel<<<SC_GRID(n_take)>>>(n_take, ckey_s, cid_s, todo, prevtodo);
        // prevtodo[c] = largest to-do id < c: exclusive max-scan of (todo ? id : -1)
        {
            size_t tb = 0;
            TEC_CUDA(cub::DeviceScan::ExclusiveScan(nullptr, tb, prevtodo, prevtodo, MaxI32(), -1, (int)W, ctx->stream));
            rc = sc_cub_tmp(ctx, tb);
            if (rc) return rc;
            TEC_CUDA(cub::DeviceScan::ExclusiveScan(s->cub_tmp, tb, prevtodo, prevtodo, MaxI32(), -1, (int)W, ctx->stream));
        }
        rc = sc_excl_sum(ctx, present, present, n_b * W + 1);
        if (rc) return rc;
        u32* winner_at = nullptr;
        TEC_CUDA(A.get(&winner_at, (size_t)N));
        TEC_CUDA(cudaMemsetAsync(winner_at, 0xFF, (size_t)N * 4, ctx->stream));
        sc_keep_kernel<<<SC_GRID(N)>>>(N, W, scell, sumi, shead, khead, bundle, todo, prevtodo, minumi, present, winner_at, s->d_stats);
        ctx->launches += 5;
        // ---- Part 3: overlap + tally of the winners' fragments; retried with a larger pair list
        u32 *d_np = nullptr, *d_over = nullptr;
        TEC_CUDA(A.get(&d_np, 1));
        TEC_CUDA(A.get(&d_over, 1));
        // dense list of the winning lines
        u32 *wlist = nullptr, *d_nwin = nullptr;
        TEC_CUDA(A.get(&wlist, (size_t)std::max<int64_t>(N, 1)));
        TEC_CUDA(A.get(&d_nwin, 1));
        u32 h_nwin = 0;
        {
            // one selection pass over the positions 0..N-1 (no flag array, prefix sum and list kernel)
            ScIsWinner is_winner;
            is_winner.shead_pos = shead; is_winner.khead_pos = khead; is_winner.winner_at = winner_at;
            cub::CountingInputIterator<u32> positions(0u);
            size_t tb = 0;
            TEC_CUDA(cub::DeviceSelect::If(nullptr, tb, positions, wlist, d_nwin, (int)N, is_winner, ctx->stream));
            rc = sc_cub_tmp(ctx, tb);
            if (rc) return rc;
            TEC_CUDA(cub::DeviceSelect::If(s->cub_tmp, tb, positions, wlist, d_nwin, (int)N, is_winner, ctx->stream));
            TEC_CUDA(cudaMemcpyAsync(&h_nwin, d_nwin, 4, cudaMemcpyDeviceToHost, ctx->stream));
            TEC_CUDA(cudaStreamSynchronize(ctx->stream));
        }
        ctx->launches += 2;
        A.release(winner_at);
        u64 h_stats_before[TEC_SC_NSTATS];
        TEC_CUDA(cudaMemcpyAsync(h_stats_before, s->d_stats, sizeof(h_stats_before), cudaMemcpyDeviceToHost, ctx->stream));
        TEC_CUDA(cudaStreamSynchronize(ctx->stream));
        int64_t cap_pairs = std::min<int64_t>(std::max<int64_t>(2 * (int64_t)h_stats_before[TEC_SS_VALID] + 1024, 1 << 16), (int64_t)0xFFFFFFF0);
        u64* pairs = nullptr;
        for (;;) {
            TEC_CUDA(A.get(&pairs, (size_t)cap_pairs));
            TEC_CUDA(cudaMemsetAsync(d_np, 0, 4, ctx->stream));
            TEC_CUDA(cudaMemsetAsync(d_over, 0, 4, ctx->stream));
            TEC_CUDA(cudaMemsetAsync(hits, 0, (size_t)W * 4, ctx->stream));
            TEC_CUDA(cudaMemcpyAsync(s->d_stats, h_stats_before, sizeof(h_stats_before), cudaMemcpyHostToDevice, ctx->stream));
            ScOut o;
            o.pairs = pairs; o.n_pairs = d_np; o.cap_pairs = (u32)cap_pairs; o.cell_hits = hits; o.stats = s->d_stats; o.overflow = d_over;
            ScTableView tv;
            tv.sv = ctx->idx.sc_stab_view();
            tv.pair_key = ctx->idx.sc_pair_key; tv.pair_type = ctx->idx.sc_pair_type;
            tv.present = (ctx->idx.has_sc_stab && ctx->opt_sc_algo != 0) ? 1 : 0;
            sc_part3_kernel<<<SC_GRID(h_nwin)>>>(N, (int64_t)h_nwin, wlist, ctx->idx.view(), tv, s->strand, d_ensg_of_slot, scell, shead,
                                                 scs, perm, s->frag, o);
            ctx->launches++;
            u32 h_over = 0;
            TEC_CUDA(cudaMemcpyAsync(&h_over, d_over, 4, cudaMemcpyDeviceToHost, ctx->stream));
            TEC_CUDA(cudaMemcpyAsync(&h_npairs, d_np, 4, cudaMemcpyDeviceToHost, ctx->stream));
            TEC_CUDA(cudaStreamSynchronize(ctx->stream));
            if (!h_over) break;
            A.release(pairs);
            if (cap_pairs >= (int64_t)0xFFFFFFF0) TEC_FAIL(TEC_ERR_LIMIT, "single-cell path: more than 2^32 (feature, cell) increments");
            cap_pairs = std::min<int64_t>(std::max<int64_t>((int64_t)h_npairs + 1024, cap_pairs * 2), (int64_t)0xFFFFFFF0);
        }
        // release what Part 3 no longer needs before sorting the pair list
        A.release(wlist); A.release(minumi); A.release(present); A.release(bundle); A.release(shead); A.release(khead);
        A.release(sumi); A.release(scell); A.release(perm); A.release(scs);
        // ---- triples: sort (ensg, cell) keys, run-length encode
        if (h_npairs) {
            TEC_CUDA(A.get(&pairs_sorted, (size_t)h_npairs));
            size_t tb = 0;
            if (ctx->opt_sc_sort != 0) {
                // keys = ensg << 32 | cell: stable LSD over the cell bits, then over the ensg bits (csrc/radix.cuh, keys only;
                // the zero bits between the two fields are never visited)
                const RdxPlan plan = rdx_plan(h_npairs, ctx->n_sm);
                u32* scratch = nullptr;
                TEC_CUDA(A.get(&scratch, plan.counts_bytes / 4));
                const int cell_bits = std::max(1, ceil_log2_i64(std::max<int64_t>(W, 2)));
                const int ensg_bits = std::max(1, ceil_log2_i64(std::max<int64_t>(ctx->idx.n_ensg, 2)));
                bool in_b = false, in_b2 = false;
                int p1 = 0, p2 = 0;
                TEC_CUDA((rdx_sort<u64, false>(pairs, nullptr, pairs_sorted, nullptr, h_npairs, 0, cell_bits, ctx->n_sm, scratch, ctx->stream, &in_b, &p1)));
                u64 *k1 = in_b ? pairs_sorted : pairs, *k2 = in_b ? pairs : pairs_sorted;
                TEC_CUDA((rdx_sort<u64, false>(k1, nullptr, k2, nullptr, h_npairs, 32, 32 + ensg_bits, ctx->n_sm, scratch, ctx->stream, &in_b2, &p2)));
                u64* other = in_b2 ? k1 : k2;
                pairs_sorted = in_b2 ? k2 : k1;
                ctx->launches += RDX_LAUNCHES_PER_PASS * (p1 + p2);
                A.release(scratch);
                A.release(other);
            } else {
                const int kb = 32 + std::max(1, ceil_log2_i64(std::max<int64_t>(ctx->idx.n_ensg, 2)));
                TEC_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, tb, pairs, pairs_sorted, (int)h_npairs, 0, std::min(kb, 64), ctx->stream));
                rc = sc_cub_tmp(ctx, tb);
                if (rc) return rc;
                TEC_CUDA(cub::DeviceRadixSort::SortKeys(s->cub_tmp, tb, pairs, pairs_sorted, (int)h_npairs, 0, std::min(kb, 64), ctx->stream));
                A.release(pairs);
            }
            u64* ukeys = nullptr;
            u32 *ucnt = nullptr, *d_nruns = nullptr;
            TEC_CUDA(A.get(&ukeys, (size_t)h_npairs));
            TEC_CUDA(A.get(&ucnt, (size_t)h_npairs));
            TEC_CUDA(A.get(&d_nruns, 1));
            tb = 0;
            TEC_CUDA(cub::DeviceRunLengthEncode::Encode(nullptr, tb, pairs_sorted, ukeys, ucnt, d_nruns, (int)h_npairs, ctx->stream));
            rc = sc_cub_tmp(ctx, tb);
            if (rc) return rc;
            TEC_CUDA(cub::DeviceRunLengthEncode::Encode(s->cub_tmp, tb, pairs_sorted, ukeys, ucnt, d_nruns, (int)h_npairs, ctx->stream));
            u32 h_runs = 0;
            TEC_CUDA(cudaMemcpyAsync(&h_runs, d_nruns, 4, cudaMemcpyDeviceToHost, ctx->stream));
            TEC_CUDA(cudaStreamSynchronize(ctx->stream));
            s->n_triples = h_runs;
            TEC_CUDA(ctx->cache.get((void**)&s->t_ensg, std::max<size_t>(h_runs, 1) * 4));
            TEC_CUDA(ctx->cache.get((void**)&s->t_cell, std::max<size_t>(h_runs, 1) * 4));
            TEC_CUDA(ctx->cache.get((void**)&s->t_count, std::max<size_t>(h_runs, 1) * 8));
            if (h_runs) sc_split_kernel<<<SC_GRID(h_runs)>>>(h_runs, ukeys, ucnt, s->t_ensg, s->t_cell, s->t_count);
            ctx->launches += 8;
        }
    }
    // ---- hit cells, ascending id (self.barcodes after Part 3); with several ranks every rank gets all of them
    {
        int rc0 = sc_allreduce(ctx, hits, W, 0, 0);
        if (rc0) return rc0;
        u32 *nz = nullptr;
        TEC_CUDA(A.get(&nz, (size_t)W + 1));
        TEC_CUDA(cudaMemsetAsync(nz, 0, (size_t)(W + 1) * 4, ctx->stream));
        sc_nonzero_kernel<<<SC_GRID(W)>>>(W, hits, nz);
        int rc = sc_excl_sum(ctx, nz, nz, W + 1);
        if (rc) return rc;
        u32 h_n = 0;
        TEC_CUDA(cudaMemcpyAsync(&h_n, nz + W, 4, cudaMemcpyDeviceToHost, ctx->stream));
        TEC_CUDA(cudaStreamSynchronize(ctx->stream));
        s->n_hit = h_n;
        TEC_CUDA(ctx->cache.get((void**)&s->h_cell, std::max<size_t>(h_n, 1) * 4));
        TEC_CUDA(ctx->cache.get((void**)&s->h_count, std::max<size_t>(h_n, 1) * 8));
        if (h_n) sc_hitcells_kernel<<<SC_GRID(W)>>>(W, hits, nz, s->h_cell, s->h_count);
        ctx->launches += 2;
    }
    TEC_CUDA(cudaGetLastError());
    u64 h_stats[TEC_SC_NSTATS];
    TEC_CUDA(cudaMemcpyAsync(h_stats, s->d_stats, sizeof(h_stats), cudaMemcpyDeviceToHost, ctx->stream));
    TEC_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
    ctx->timed = true;
    TEC_CUDA(cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < TEC_SC_NSTATS; ++i) s->stats[i] = (int64_t)h_stats[i];
    s->stats[TEC_SS_UNITS] = s->units;
    s->stats[TEC_SS_BUNDLES] = n_b;
    s->stats[TEC_SS_SURVIVORS] = N;
    if (s->world > 1 && (s->coll || ctx->comm)) {
        // job-wide statistics: sums over the ranks, except the two that are already global
        u64 tmp[TEC_SC_NSTATS];
        for (int i = 0; i < TEC_SC_NSTATS; ++i) tmp[i] = (u64)s->stats[i];
        tmp[TEC_SS_RAW_BARCODES] = 0; tmp[TEC_SS_BUNDLES] = 0;
        u64* d_tmp = nullptr;
        TEC_CUDA(A.get(&d_tmp, TEC_SC_NSTATS));
        TEC_CUDA(cudaMemcpyAsync(d_tmp, tmp, sizeof(tmp), cudaMemcpyHostToDevice, ctx->stream));
        int rc1 = sc_allreduce(ctx, d_tmp, TEC_SC_NSTATS, 1, 0);
        if (rc1) return rc1;
        TEC_CUDA(cudaMemcpyAsync(tmp, d_tmp, sizeof(tmp), cudaMemcpyDeviceToHost, ctx->stream));
        TEC_CUDA(cudaStreamSynchronize(ctx->stream));
        for (int i = 0; i < TEC_SC_NSTATS; ++i)
            if (i != TEC_SS_RAW_BARCODES && i != TEC_SS_BUNDLES) s->stats[i] = (int64_t)tmp[i];
    }
    s->finalized = true;
    if (n_triples) *n_triples = s->n_triples;
    if (n_hit_cells) *n_hit_cells = s->n_hit;
    return TEC_OK;
}

extern "C" int tec_sc_fetch(tec_ctx* ctx, int32_t* ensg, uint32_t* cell, int64_t* count,
                            uint32_t* hit_cell, int64_t* hit_count, int64_t* stats) {
    if (!ctx) return TEC_ERR_ARG;
    ScState* s = ctx->sc;
    if (!s || !s->finalized) TEC_FAIL(TEC_ERR_STATE, "tec_sc_fetch: tec_sc_finalize not called");
    TEC_CUDA(cudaSetDevice(ctx->device));
    if (s->n_triples) {
        if (ensg) TEC_CUDA(cudaMemcpyAsync(ensg, s->t_ensg, (size_t)s->n_triples * 4, cudaMemcpyDeviceToHost, ctx->stream));
        if (cell) TEC_CUDA(cudaMemcpyAsync(cell, s->t_cell, (size_t)s->n_triples * 4, cudaMemcpyDeviceToHost, ctx->stream));
        if (count) TEC_CUDA(cudaMemcpyAsync(count, s->t_count, (size_t)s->n_triples * 8, cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (s->n_hit) {
        if (hit_cell) TEC_CUDA(cudaMemcpyAsync(hit_cell, s->h_cell, (size_t)s->n_hit * 4, cudaMemcpyDeviceToHost, ctx->stream));
        if (hit_count) TEC_CUDA(cudaMemcpyAsync(hit_count, s->h_count, (size_t)s->n_hit * 8, cudaMemcpyDeviceToHost, ctx->stream));
    }
    TEC_CUDA(cudaStreamSynchronize(ctx->stream));
    if (stats) memcpy(stats, s->stats, sizeof(s->stats));
    return TEC_OK;
}

// sc_save_result's rows (te_count.py:724-733): hits descending, ties by ascending id
extern "C" int tec_sc_select(tec_ctx* ctx, int64_t maxcells, uint32_t* cells_out, int64_t* n_out) {
    if (!ctx) return TEC_ERR_ARG;
    ScState* s = ctx->sc;
    if (!s || !s->finalized) TEC_FAIL(TEC_ERR_STATE, "tec_sc_select: tec_sc_finalize not called");
    if (maxcells < 0) TEC_FAIL(TEC_ERR_ARG, "tec_sc_select: negative maxcells");
    TEC_CUDA(cudaSetDevice(ctx->device));
    const int64_t n = s->n_hit, take = std::min(n, maxcells);
    if (n_out) *n_out = take;
    if (!take) return TEC_OK;
    ScArena A(ctx->cache);
    u64 *key = nullptr, *key_s = nullptr;
    u32* cell_s = nullptr;
    TEC_CUDA(A.get(&key, (size_t)n));
    TEC_CUDA(A.get(&key_s, (size_t)n));
    TEC_CUDA(A.get(&cell_s, (size_t)n));
    sc_selkey_kernel<<<SC_GRID(n)>>>(n, s->h_cell, s->h_count, key);
    int rc = sc_sort_pairs(ctx, key, key_s, s->h_cell, cell_s, n, 0, 64);
    if (rc) return rc;
    ctx->launches++;
    if (cells_out) TEC_CUDA(cudaMemcpyAsync(cells_out, cell_s, (size_t)take * 4, cudaMemcpyDeviceToHost, ctx->stream));
    TEC_CUDA(cudaStreamSynchronize(ctx->stream));
    return TEC_OK;
}
