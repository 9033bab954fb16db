// Paired end by read name (tec_bulk_begin(ctx, 2, qual); rule in include/tecount.h): the k-th read1 of a QNAME pairs
// with the k-th read2 of that QNAME in file order, wherever they lie in the file.  Per delivered batch of one-record
// rows (bgzfdev::MODE_PE_NAME rows of the device decoder, or tec_bulk_push_named):
//   1. the batch goes behind the rows left pending by earlier batches (pending rows first, the batch in file order);
//   2. row indices are stably sorted by the 128-bit name key: two stable 64-bit rdx_sort calls (radix.cuh), low word
//      first, then the high word, so rows of one name stay in file order;
//   3. name_group_kernel: one thread per run of equal keys matches its k-th read1 with its k-th read2 and writes each
//      pair as rows (read1, read2) of the unit columns, which the paired bulk kernels count (bulk_push_dev, the route
//      of the byte-range banks).  Excluded rows are counted and dropped; unmatched rows are copied, still in file order
//      within their name, into the other row set, which becomes the pending set.
// In a coordinate-sorted file the pending set holds the pairs that cross a window border and the mates on other
// chromosomes; it grows on demand up to about half the file (every read1 in front of every read2).
//
// One file over several ranks (tec_bam_count_range mode 4, tec_bulk_name_partition_dev / _import_dev / _exchange): a
// rank's byte range pairs nothing.  Its rows are held in rows[cur] in file order; the partition drops (and counts) the
// excluded ones and packs the others as 32-byte NameRecords grouped by owner rank key_lo % world, file order kept inside
// a group.  After the all-to-all an owner holds every record of its names, in file order (source ranks in rank order,
// each in file order), and one pass of steps 2 and 3 over them gives the pairs of a one-rank run.
#pragma once
#include "context.cuh"
#include "radix.cuh"
#include "bgzf_dev.h"
#include "collective.cuh"
#include "sc.cuh"                   // ScArena

#include <cub/cub.cuh>

static int bulk_push_dev(tec_ctx* ctx, int64_t n_rec, const int32_t* start, const int32_t* end,
                         const uint16_t* chrom, const uint8_t* mapq, const uint8_t* flag);

#define NAME_TPB 256

struct NameRows {
    int32_t *start = nullptr, *end = nullptr;
    uint16_t* chrom = nullptr;
    uint8_t *mapq = nullptr, *flag = nullptr, *role = nullptr;
    u64 *key_hi = nullptr, *key_lo = nullptr;
};

struct NameState {
    NameRows rows[2];               // rows[cur]: pending rows, then the batch; rows[cur ^ 1]: the next pending set
    int cur = 0;
    int64_t cap = 0;                // rows per set, sort buffer and unit column
    u64* keys[2] = {nullptr, nullptr};
    u32* vals[2] = {nullptr, nullptr};
    u32* scratch = nullptr;
    size_t scratch_bytes = 0;
    NameRows units;                 // pairs as rows (read1, read2); role / keys unused
    u64* d_cnt = nullptr;           // [0] pairs, [1] rows left pending, [2] excluded rows of the run
    u64* h_cnt = nullptr;           // pinned copy of d_cnt
    // tec_bulk_push_named: the QNAME bytes, their offsets and the SAM flags of the call
    uint8_t* d_names = nullptr;
    int64_t* d_name_off = nullptr;
    uint16_t* d_samflag = nullptr;
    size_t names_cap = 0;
    int64_t named_cap = 0;
    cudaEvent_t ev[2] = {nullptr, nullptr};
    int64_t pending = 0, peak = 0, excluded = 0;
    double ms = 0;
    void* packed = nullptr;         // NameRecords of the last tec_bulk_name_partition_dev (until the next import / partition / begin)
};

// one row in the exchange by name owner
struct __align__(16) NameRecord {
    u64 key_hi, key_lo;
    int32_t start, end;
    uint16_t chrom;
    uint8_t mapq, flag, role, pad[3];
};
static_assert(sizeof(NameRecord) == 32, "NameRecord: 32 bytes per row in the exchange");
#define NAME_MAX_WORLD 8

// ---- kernels

// tec_bulk_push_named: key and role of each record from its QNAME bytes and SAM flag
__global__ void name_key_kernel(int64_t n, const uint8_t* __restrict__ names, const int64_t* __restrict__ off,
                                const uint16_t* __restrict__ samflag, u64* __restrict__ key_hi, u64* __restrict__ key_lo,
                                uint8_t* __restrict__ role) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int r = bgzfdev::name_role(samflag[i]);
        uint64_t hi = 0, lo = 0;
        if (r != bgzfdev::ROLE_EXCLUDED) bgzfdev::name_key(names + off[i], (uint32_t)(off[i + 1] - off[i]), hi, lo);
        key_hi[i] = hi; key_lo[i] = lo; role[i] = (uint8_t)r;
    }
}

// sort input of the first pass: (low key word, row index)
__global__ void name_sort_init_kernel(int64_t n, const u64* __restrict__ key_lo, u64* __restrict__ k, u32* __restrict__ v) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        k[i] = key_lo[i];
        v[i] = (u32)i;
    }
}

// sort input of the second pass: (high key word, row index) in the order of the first pass
__global__ void name_sort_gather_kernel(int64_t n, const u32* __restrict__ v_in, const u64* __restrict__ key_hi, u64* __restrict__ k,
                                        u32* __restrict__ v) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const u32 r = v_in[i];
        k[i] = key_hi[r];
        v[i] = r;
    }
}

// row i of s into row j of d; WITH_KEYS: role and name key too (pending rows), otherwise the five columns of a unit
template <bool WITH_KEYS>
__device__ __forceinline__ void name_copy_row(const NameRows& s, u32 i, const NameRows& d, u64 j) {
    d.start[j] = s.start[i]; d.end[j] = s.end[i]; d.chrom[j] = s.chrom[i]; d.mapq[j] = s.mapq[i]; d.flag[j] = s.flag[i];
    if (WITH_KEYS) { d.role[j] = s.role[i]; d.key_hi[j] = s.key_hi[i]; d.key_lo[j] = s.key_lo[i]; }
}

// exclusive prefix of v over the warp; *tot = warp total (every lane participates)
__device__ __forceinline__ u64 name_warp_excl(u64 v, u64* tot) {
    const int lane = threadIdx.x & 31;
    u64 incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const u64 t = __shfl_up_sync(0xFFFFFFFFu, incl, d);
        if (lane >= d) incl += t;
    }
    *tot = __shfl_sync(0xFFFFFFFFu, incl, 31);
    return incl - v;
}

// One thread per run of equal keys among the non-excluded rows of sorted order `ord` (hi = sorted high words).
// cnt: [0] pairs written, [1] rows left, [2] excluded rows; stat_no_mate: the statistics slot TEC_BS_NO_MATE.
__global__ void __launch_bounds__(NAME_TPB)
name_group_kernel(int64_t n, const u32* __restrict__ ord, const u64* __restrict__ hi, NameRows rows, NameRows units, NameRows left,
                  u64* __restrict__ cnt, u64* __restrict__ stat_no_mate) {
    const int lane = threadIdx.x & 31;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t base = (int64_t)blockIdx.x * blockDim.x; base < n; base += stride) {    // uniform trip count: whole warps shuffle
        const int64_t i = base + threadIdx.x;
        u64 n_pairs = 0, n_left = 0, n_excl = 0;
        int64_t end = i;
        bool head = false;
        if (i < n) {
            const u32 r = ord[i];
            if (rows.role[r] == bgzfdev::ROLE_EXCLUDED) {
                n_excl = 1;
            } else {
                const u64 kh = hi[i], kl = rows.key_lo[r];
                head = i == 0 || hi[i - 1] != kh || rows.key_lo[ord[i - 1]] != kl || rows.role[ord[i - 1]] == bgzfdev::ROLE_EXCLUDED;
                if (head) {
                    u64 c1 = 0, c2 = 0;
                    for (end = i; end < n && hi[end] == kh && rows.key_lo[ord[end]] == kl; ++end) {
                        const int ro = rows.role[ord[end]];
                        c1 += ro == bgzfdev::ROLE_READ1;
                        c2 += ro == bgzfdev::ROLE_READ2;
                    }
                    n_pairs = c1 < c2 ? c1 : c2;
                    n_left = c1 + c2 - 2 * n_pairs;
                }
            }
        }
        u64 t_pairs, t_left, t_excl;
        u64 o_pairs = name_warp_excl(n_pairs, &t_pairs), o_left = name_warp_excl(n_left, &t_left);
        name_warp_excl(n_excl, &t_excl);
        u64 b_pairs = 0, b_left = 0;
        if (lane == 0) {
            if (t_pairs) b_pairs = atomicAdd(cnt + 0, t_pairs);
            if (t_left) b_left = atomicAdd(cnt + 1, t_left);
            if (t_excl) { atomicAdd(cnt + 2, t_excl); atomicAdd(stat_no_mate, t_excl); }
        }
        o_pairs += __shfl_sync(0xFFFFFFFFu, b_pairs, 0);
        o_left += __shfl_sync(0xFFFFFFFFu, b_left, 0);
        if (!head) continue;
        // k-th read1 with k-th read2: two cursors over the run, in sorted (= file) order
        int64_t a = i, b = i;
        while (a < end && rows.role[ord[a]] != bgzfdev::ROLE_READ1) ++a;
        while (b < end && rows.role[ord[b]] != bgzfdev::ROLE_READ2) ++b;
        while (a < end && b < end) {
            name_copy_row<false>(rows, ord[a], units, 2 * o_pairs);
            name_copy_row<false>(rows, ord[b], units, 2 * o_pairs + 1);
            ++o_pairs;
            for (++a; a < end && rows.role[ord[a]] != bgzfdev::ROLE_READ1; ++a) {}
            for (++b; b < end && rows.role[ord[b]] != bgzfdev::ROLE_READ2; ++b) {}
        }
        // what is left is of one role only: it stays pending, in file order
        const int64_t rest = a < end ? a : b;
        const int want = a < end ? bgzfdev::ROLE_READ1 : bgzfdev::ROLE_READ2;
        for (int64_t p = rest; p < end; ++p)
            if (rows.role[ord[p]] == want) name_copy_row<true>(rows, ord[p], left, o_left++);
    }
}

__global__ void name_add_kernel(u64* p, u64 v) { *p += v; }

// Partition of the held rows: one warp owns the contiguous rows [w * per_warp, (w + 1) * per_warp).  Pass 1 counts the
// rows of each owner per warp (counts[d * n_warps + w]) and adds the excluded rows to *excl and the statistics slot.
__global__ void name_part_count_kernel(int64_t n, int world, int64_t per_warp, int n_warps, const uint8_t* __restrict__ role,
                                       const u64* __restrict__ key_lo, u32* __restrict__ counts, u64* __restrict__ excl,
                                       u64* __restrict__ stat_no_mate) {
    const int lane = threadIdx.x & 31;
    for (int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < n_warps; w += (gridDim.x * blockDim.x) >> 5) {
        u32 cnt[NAME_MAX_WORLD];
#pragma unroll
        for (int d = 0; d < NAME_MAX_WORLD; ++d) cnt[d] = 0;
        u32 n_excl = 0;
        const int64_t lo = (int64_t)w * per_warp, hi = min(n, lo + per_warp);
        for (int64_t i = lo + lane; i < hi; i += 32) {
            if (role[i] == bgzfdev::ROLE_EXCLUDED) { ++n_excl; continue; }
            const int dst = (int)(key_lo[i] % (u64)world);
#pragma unroll
            for (int d = 0; d < NAME_MAX_WORLD; ++d) cnt[d] += dst == d;
        }
#pragma unroll
        for (int d = 0; d < NAME_MAX_WORLD; ++d) {
            const u32 t = (u32)warp_sum((u64)cnt[d]);
            if (lane == 0 && d < world) counts[(size_t)d * n_warps + w] = t;
        }
        const u64 t = warp_sum((u64)n_excl);
        if (lane == 0 && t) { atomicAdd(excl, t); atomicAdd(stat_no_mate, t); }
    }
}

// Pass 2 (offsets = exclusive sum of the counts): every non-excluded row into its owner's group, file order kept
__global__ void name_part_scatter_kernel(int64_t n, int world, int64_t per_warp, int n_warps, NameRows rows, const u32* __restrict__ offsets,
                                         NameRecord* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const u32 lt = (1u << lane) - 1u;
    for (int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < n_warps; w += (gridDim.x * blockDim.x) >> 5) {
        u32 off[NAME_MAX_WORLD];
#pragma unroll
        for (int d = 0; d < NAME_MAX_WORLD; ++d) off[d] = d < world ? offsets[(size_t)d * n_warps + w] : 0u;
        const int64_t lo = (int64_t)w * per_warp, hi = min(n, lo + per_warp);
        for (int64_t base = lo; base < hi; base += 32) {
            const int64_t i = base + lane;
            const bool live = i < hi && rows.role[i] != bgzfdev::ROLE_EXCLUDED;
            const u64 kl = live ? rows.key_lo[i] : 0;
            const int dst = live ? (int)(kl % (u64)world) : -1;
            u32 pos = 0;
#pragma unroll
            for (int d = 0; d < NAME_MAX_WORLD; ++d) {
                const u32 m = __ballot_sync(0xFFFFFFFFu, dst == d);
                if (dst == d) pos = off[d] + __popc(m & lt);
                off[d] += __popc(m);
            }
            if (live) {
                NameRecord r;
                r.key_hi = rows.key_hi[i]; r.key_lo = kl; r.start = rows.start[i]; r.end = rows.end[i]; r.chrom = rows.chrom[i];
                r.mapq = rows.mapq[i]; r.flag = rows.flag[i]; r.role = rows.role[i]; r.pad[0] = r.pad[1] = r.pad[2] = 0;
                out[pos] = r;
            }
        }
    }
}

// received records into rows [0, n) of d
__global__ void name_unpack_kernel(int64_t n, const NameRecord* __restrict__ in, NameRows d) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const NameRecord r = in[i];
        d.start[i] = r.start; d.end[i] = r.end; d.chrom[i] = r.chrom; d.mapq[i] = r.mapq; d.flag[i] = r.flag; d.role[i] = r.role;
        d.key_hi[i] = r.key_hi; d.key_lo[i] = r.key_lo;
    }
}

// ---- host side

inline void tec_ctx::free_name() {
    NameState* s = name;
    if (!s) return;
    auto put_rows = [&](NameRows& r) {
        cache.put(r.start); cache.put(r.end); cache.put(r.chrom); cache.put(r.mapq); cache.put(r.flag); cache.put(r.role);
        cache.put(r.key_hi); cache.put(r.key_lo);
        r = NameRows();
    };
    put_rows(s->rows[0]); put_rows(s->rows[1]); put_rows(s->units);
    for (int i = 0; i < 2; ++i) { cache.put(s->keys[i]); cache.put(s->vals[i]); }
    cache.put(s->scratch); cache.put(s->d_cnt); cache.put(s->d_names); cache.put(s->d_name_off); cache.put(s->d_samflag);
    cache.put(s->packed);
    if (s->h_cnt) cudaFreeHost(s->h_cnt);
    for (int i = 0; i < 2; ++i)
        if (s->ev[i]) cudaEventDestroy(s->ev[i]);
    delete s;
    name = nullptr;
}

// a new run: nothing pending or held, statistics of the stage back to zero (buffers are kept)
static int name_begin(tec_ctx* ctx) {
    if (!ctx->name) {
        ctx->name = new NameState();
        NameState& s = *ctx->name;
        TEC_CUDA(cudaMalloc(&s.d_cnt, 4 * 8));
        TEC_CUDA(cudaHostAlloc(&s.h_cnt, 4 * 8, cudaHostAllocDefault));
        for (int i = 0; i < 2; ++i) TEC_CUDA(cudaEventCreate(&s.ev[i]));
    }
    NameState& s = *ctx->name;
    s.pending = 0; s.peak = 0; s.excluded = 0; s.ms = 0;
    TEC_CUDA(cudaStreamSynchronize(ctx->stream));       // no copy of the exchange still reads the packed records
    ctx->cache.put(s.packed);
    s.packed = nullptr;
    TEC_CUDA(cudaMemsetAsync(s.d_cnt, 0, 4 * 8, ctx->stream));
    return TEC_OK;
}

template <class T> static int name_grow(tec_ctx* ctx, T** p, size_t bytes) {
    ctx->cache.put(*p);
    *p = nullptr;
    void* q = nullptr;
    TEC_CUDA(ctx->cache.get(&q, bytes));
    *p = (T*)q;
    return TEC_OK;
}

static int name_grow_rows(tec_ctx* ctx, NameRows& r, int64_t cap, bool keys) {
    const size_t n = (size_t)cap;
    int rc = 0;
    if ((rc = name_grow(ctx, &r.start, n * 4)) || (rc = name_grow(ctx, &r.end, n * 4)) || (rc = name_grow(ctx, &r.chrom, n * 2)) ||
        (rc = name_grow(ctx, &r.mapq, n)) || (rc = name_grow(ctx, &r.flag, n)))
        return rc;
    if (keys && ((rc = name_grow(ctx, &r.role, n)) || (rc = name_grow(ctx, &r.key_hi, n * 8)) || (rc = name_grow(ctx, &r.key_lo, n * 8)))) return rc;
    return TEC_OK;
}

// room for `need` rows in every buffer of the stage; the pending rows of rows[cur] are kept
static int name_reserve(tec_ctx* ctx, int64_t need) {
    NameState& s = *ctx->name;
    if (need >= ((int64_t)1 << 32) - (1 << 13)) TEC_FAIL(TEC_ERR_LIMIT, "pairing by read name: more than 2^32 - 2^13 rows in one pairing pass");
    if (need <= s.cap) return TEC_OK;
    const int64_t cap = std::min<int64_t>(need + (need >> 2) + 4096, ((int64_t)1 << 32) - (1 << 13) - 1);
    TEC_CUDA(cudaStreamSynchronize(ctx->stream));
    s.cap = 0;                                  // until every buffer has its new size
    NameRows old = s.rows[s.cur];
    s.rows[s.cur] = NameRows();
    int rc = 0;
    if ((rc = name_grow_rows(ctx, s.rows[s.cur], cap, true))) return rc;
    if (s.pending) {
        const size_t p = (size_t)s.pending;
        const NameRows& d = s.rows[s.cur];
        TEC_CUDA(cudaMemcpyAsync(d.start, old.start, p * 4, cudaMemcpyDeviceToDevice, ctx->stream));
        TEC_CUDA(cudaMemcpyAsync(d.end, old.end, p * 4, cudaMemcpyDeviceToDevice, ctx->stream));
        TEC_CUDA(cudaMemcpyAsync(d.chrom, old.chrom, p * 2, cudaMemcpyDeviceToDevice, ctx->stream));
        TEC_CUDA(cudaMemcpyAsync(d.mapq, old.mapq, p, cudaMemcpyDeviceToDevice, ctx->stream));
        TEC_CUDA(cudaMemcpyAsync(d.flag, old.flag, p, cudaMemcpyDeviceToDevice, ctx->stream));
        TEC_CUDA(cudaMemcpyAsync(d.role, old.role, p, cudaMemcpyDeviceToDevice, ctx->stream));
        TEC_CUDA(cudaMemcpyAsync(d.key_hi, old.key_hi, p * 8, cudaMemcpyDeviceToDevice, ctx->stream));
        TEC_CUDA(cudaMemcpyAsync(d.key_lo, old.key_lo, p * 8, cudaMemcpyDeviceToDevice, ctx->stream));
        TEC_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    for (void* q : {(void*)old.start, (void*)old.end, (void*)old.chrom, (void*)old.mapq, (void*)old.flag, (void*)old.role, (void*)old.key_hi,
                    (void*)old.key_lo})
        ctx->cache.put(q);
    if ((rc = name_grow_rows(ctx, s.rows[s.cur ^ 1], cap, true)) || (rc = name_grow_rows(ctx, s.units, cap, false))) return rc;
    for (int i = 0; i < 2; ++i)
        if ((rc = name_grow(ctx, &s.keys[i], (size_t)cap * 8)) || (rc = name_grow(ctx, &s.vals[i], (size_t)cap * 4))) return rc;
    const size_t sb = rdx_plan(cap, ctx->n_sm).counts_bytes;
    if ((rc = name_grow(ctx, &s.scratch, sb))) return rc;
    s.scratch_bytes = sb;
    s.cap = cap;
    return TEC_OK;
}

static int name_grid(tec_ctx* ctx, int64_t n) { return (int)std::max<int64_t>(1, std::min<int64_t>((n + NAME_TPB - 1) / NAME_TPB, (int64_t)ctx->n_sm * 16)); }

// steps 2 and 3 over rows[cur][0, pending + n): the batch is in place behind the pending rows (name_reserve was called)
static int name_pair_batch(tec_ctx* ctx, int64_t n) {
    NameState& s = *ctx->name;
    const int64_t m = s.pending + n;
    if (!n) return TEC_OK;
    const NameRows& rows = s.rows[s.cur];
    TEC_CUDA(cudaMemsetAsync(s.d_cnt, 0, 2 * 8, ctx->stream));
    name_sort_init_kernel<<<name_grid(ctx, m), NAME_TPB, 0, ctx->stream>>>(m, rows.key_lo, s.keys[0], s.vals[0]);
    TEC_CUDA(cudaGetLastError());
    bool in_b = false;
    TEC_CUDA((rdx_sort<u64, true>(s.keys[0], s.vals[0], s.keys[1], s.vals[1], m, 0, 64, ctx->n_sm, s.scratch, ctx->stream, &in_b)));
    int r = in_b ? 1 : 0;
    name_sort_gather_kernel<<<name_grid(ctx, m), NAME_TPB, 0, ctx->stream>>>(m, s.vals[r], rows.key_hi, s.keys[r ^ 1], s.vals[r ^ 1]);
    TEC_CUDA(cudaGetLastError());
    TEC_CUDA((rdx_sort<u64, true>(s.keys[r ^ 1], s.vals[r ^ 1], s.keys[r], s.vals[r], m, 0, 64, ctx->n_sm, s.scratch, ctx->stream, &in_b)));
    r = in_b ? r : r ^ 1;
    name_group_kernel<<<name_grid(ctx, m), NAME_TPB, 0, ctx->stream>>>(m, s.vals[r], s.keys[r], rows, s.units, s.rows[s.cur ^ 1], s.d_cnt,
                                                                      ctx->d_counts + ctx->idx.n_ensg + TEC_BS_NO_MATE);
    TEC_CUDA(cudaGetLastError());
    TEC_CUDA(cudaEventRecord(s.ev[1], ctx->stream));
    TEC_CUDA(cudaMemcpyAsync(s.h_cnt, s.d_cnt, 3 * 8, cudaMemcpyDeviceToHost, ctx->stream));
    TEC_CUDA(cudaStreamSynchronize(ctx->stream));
    float ms = 0.f;
    TEC_CUDA(cudaEventElapsedTime(&ms, s.ev[0], s.ev[1]));
    s.ms += ms;
    ctx->launches += 3 + 2 * 6 * RDX_LAUNCHES_PER_PASS;
    const int64_t pairs = (int64_t)s.h_cnt[0];
    s.pending = (int64_t)s.h_cnt[1];
    s.excluded = (int64_t)s.h_cnt[2];
    s.peak = std::max(s.peak, s.pending);
    s.cur ^= 1;
    return bulk_push_dev(ctx, 2 * pairs, s.units.start, s.units.end, s.units.chrom, s.units.mapq, s.units.flag);
}

// device rows of one batch (the MODE_PE_NAME columns of the device decoder) behind the rows of rows[cur]
static int name_append_dev(tec_ctx* ctx, int64_t n, const bgzfdev::Columns& c) {
    NameState& s = *ctx->name;
    if (int rc = name_reserve(ctx, s.pending + n)) return rc;
    TEC_CUDA(cudaEventRecord(s.ev[0], ctx->stream));
    const NameRows& d = s.rows[s.cur];
    const size_t p = (size_t)s.pending, k = (size_t)n;
    TEC_CUDA(cudaMemcpyAsync(d.start + p, c.start, k * 4, cudaMemcpyDeviceToDevice, ctx->stream));
    TEC_CUDA(cudaMemcpyAsync(d.end + p, c.end, k * 4, cudaMemcpyDeviceToDevice, ctx->stream));
    TEC_CUDA(cudaMemcpyAsync(d.chrom + p, c.chrom, k * 2, cudaMemcpyDeviceToDevice, ctx->stream));
    TEC_CUDA(cudaMemcpyAsync(d.mapq + p, c.mapq, k, cudaMemcpyDeviceToDevice, ctx->stream));
    TEC_CUDA(cudaMemcpyAsync(d.flag + p, c.flag, k, cudaMemcpyDeviceToDevice, ctx->stream));
    TEC_CUDA(cudaMemcpyAsync(d.role + p, c.role, k, cudaMemcpyDeviceToDevice, ctx->stream));
    TEC_CUDA(cudaMemcpyAsync(d.key_hi + p, c.key_hi, k * 8, cudaMemcpyDeviceToDevice, ctx->stream));
    TEC_CUDA(cudaMemcpyAsync(d.key_lo + p, c.key_lo, k * 8, cudaMemcpyDeviceToDevice, ctx->stream));
    return TEC_OK;
}

static int name_push_dev(tec_ctx* ctx, int64_t n, const bgzfdev::Columns& c) {
    if (n <= 0) return TEC_OK;
    if (int rc = name_append_dev(ctx, n, c)) return rc;
    return name_pair_batch(ctx, n);
}

// a window of a read-name byte range (MODE_PE_NAME_RANGE): the rows join the held set, unpaired and uncounted
static int name_hold_dev(tec_ctx* ctx, int64_t n, const bgzfdev::Columns& c) {
    if (n <= 0) return TEC_OK;
    if (int rc = name_append_dev(ctx, n, c)) return rc;
    ctx->name->pending += n;
    return TEC_OK;
}

// host rows with their SAM flags and QNAME bytes (tec_bulk_push_named)
static int name_push_host(tec_ctx* ctx, int64_t n, const int32_t* start, const int32_t* end, const uint16_t* chrom, const uint8_t* mapq,
                          const uint8_t* flag, const uint16_t* samflag, const int64_t* name_off, const char* names) {
    if (n <= 0) return TEC_OK;
    NameState& s = *ctx->name;
    if (int rc = name_reserve(ctx, s.pending + n)) return rc;
    const size_t nb = (size_t)name_off[n], k = (size_t)n;
    if (nb + 1 > s.names_cap) {
        TEC_CUDA(cudaStreamSynchronize(ctx->stream));
        if (int rc = name_grow(ctx, &s.d_names, nb + 1)) return rc;
        s.names_cap = nb + 1;
    }
    if (n > s.named_cap) {
        TEC_CUDA(cudaStreamSynchronize(ctx->stream));
        int rc = 0;
        if ((rc = name_grow(ctx, &s.d_name_off, (k + 1) * 8)) || (rc = name_grow(ctx, &s.d_samflag, k * 2))) return rc;
        s.named_cap = n;
    }
    TEC_CUDA(cudaEventRecord(s.ev[0], ctx->stream));
    const NameRows& d = s.rows[s.cur];
    const size_t p = (size_t)s.pending;
    TEC_CUDA(cudaMemcpyAsync(d.start + p, start, k * 4, cudaMemcpyHostToDevice, ctx->stream));
    TEC_CUDA(cudaMemcpyAsync(d.end + p, end, k * 4, cudaMemcpyHostToDevice, ctx->stream));
    TEC_CUDA(cudaMemcpyAsync(d.chrom + p, chrom, k * 2, cudaMemcpyHostToDevice, ctx->stream));
    TEC_CUDA(cudaMemcpyAsync(d.mapq + p, mapq, k, cudaMemcpyHostToDevice, ctx->stream));
    TEC_CUDA(cudaMemcpyAsync(d.flag + p, flag, k, cudaMemcpyHostToDevice, ctx->stream));
    TEC_CUDA(cudaMemcpyAsync(s.d_samflag, samflag, k * 2, cudaMemcpyHostToDevice, ctx->stream));
    TEC_CUDA(cudaMemcpyAsync(s.d_name_off, name_off, (k + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    if (nb) TEC_CUDA(cudaMemcpyAsync(s.d_names, names, nb, cudaMemcpyHostToDevice, ctx->stream));
    name_key_kernel<<<name_grid(ctx, n), NAME_TPB, 0, ctx->stream>>>(n, s.d_names, s.d_name_off, s.d_samflag, d.key_hi + p, d.key_lo + p, d.role + p);
    TEC_CUDA(cudaGetLastError());
    ctx->launches++;
    return name_pair_batch(ctx, n);              // synchronises: the caller's host buffers are free again
}

// end of the input (tec_bulk_finish, tec_bulk_allreduce): the rows still pending have no mate
static int name_flush(tec_ctx* ctx) {
    if (!ctx->name_pairing || !ctx->name || !ctx->name->pending) return TEC_OK;
    name_add_kernel<<<1, 1, 0, ctx->stream>>>(ctx->d_counts + ctx->idx.n_ensg + TEC_BS_NO_MATE, (u64)ctx->name->pending);
    TEC_CUDA(cudaGetLastError());
    ctx->launches++;
    ctx->name->pending = 0;
    return TEC_OK;
}

// ---- one file over several ranks (include/tecount.h: tec_bam_count_range mode 4, tec_bulk_name_*)

static int name_run_check(tec_ctx* ctx, const char* what) {
    if (!ctx->bulk_active || !ctx->name_pairing || !ctx->name) TEC_FAIL(TEC_ERR_STATE, std::string(what) + ": tec_bulk_begin(ctx, 2, qual) not called");
    return TEC_OK;
}

extern "C" int tec_bulk_name_partition_dev(tec_ctx* ctx, int world, int64_t* counts, void** records) {
    if (!ctx) return TEC_ERR_ARG;
    if (int rc = name_run_check(ctx, "tec_bulk_name_partition_dev")) return rc;
    if (!ctx->name_held) TEC_FAIL(TEC_ERR_STATE, "tec_bulk_name_partition_dev: no rows held (tec_bam_count_range mode 4)");
    if (world < 1 || world > NAME_MAX_WORLD || !counts || !records) TEC_FAIL(TEC_ERR_ARG, "tec_bulk_name_partition_dev: 1..8 ranks");
    TEC_CUDA(cudaSetDevice(ctx->device));
    NameState& s = *ctx->name;
    const int64_t N = s.pending;
    const int n_warps = (int)std::max<int64_t>(1, std::min<int64_t>((N + 1023) / 1024, (int64_t)ctx->n_sm * 64));
    const int64_t per_warp = ((N + n_warps - 1) / n_warps + 31) / 32 * 32;
    const int64_t n_cnt = (int64_t)world * n_warps + 1;
    TEC_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->cache.put(s.packed);
    s.packed = nullptr;
    TEC_CUDA(ctx->cache.get(&s.packed, (size_t)std::max<int64_t>(N, 1) * sizeof(NameRecord)));
    ScArena A(ctx->cache);
    u32* cnt = nullptr;
    uint8_t* tmp = nullptr;
    size_t tb = 0;
    TEC_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tb, cnt, cnt, (int)n_cnt, ctx->stream));
    TEC_CUDA(A.get(&cnt, (size_t)n_cnt));
    TEC_CUDA(A.get(&tmp, tb));
    TEC_CUDA(cudaMemsetAsync(cnt, 0, (size_t)n_cnt * 4, ctx->stream));
    const NameRows& rows = s.rows[s.cur];
    const int blocks = std::max(1, std::min((n_warps + 7) / 8, ctx->n_sm * 8));
    name_part_count_kernel<<<blocks, 256, 0, ctx->stream>>>(N, world, per_warp, n_warps, rows.role, rows.key_lo, cnt, s.d_cnt + 2,
                                                            ctx->d_counts + ctx->idx.n_ensg + TEC_BS_NO_MATE);
    TEC_CUDA(cudaGetLastError());
    TEC_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tb, cnt, cnt, (int)n_cnt, ctx->stream));
    name_part_scatter_kernel<<<blocks, 256, 0, ctx->stream>>>(N, world, per_warp, n_warps, rows, cnt, (NameRecord*)s.packed);
    TEC_CUDA(cudaGetLastError());
    ctx->launches += 4;
    std::vector<u32> h((size_t)world + 1);
    for (int d = 0; d <= world; ++d)
        TEC_CUDA(cudaMemcpyAsync(&h[(size_t)d], cnt + (size_t)d * n_warps, 4, cudaMemcpyDeviceToHost, ctx->stream));
    TEC_CUDA(cudaMemcpyAsync(s.h_cnt + 2, s.d_cnt + 2, 8, cudaMemcpyDeviceToHost, ctx->stream));
    TEC_CUDA(cudaStreamSynchronize(ctx->stream));
    for (int d = 0; d < world; ++d) counts[d] = (int64_t)h[(size_t)d + 1] - (int64_t)h[(size_t)d];
    s.excluded = (int64_t)s.h_cnt[2];
    s.pending = 0;                              // the held rows are in the packed records now
    ctx->name_held = false;
    *records = s.packed;
    return TEC_OK;
}

extern "C" int tec_bulk_name_import_dev(tec_ctx* ctx, int64_t n, const void* records) {
    if (!ctx) return TEC_ERR_ARG;
    if (int rc = name_run_check(ctx, "tec_bulk_name_import_dev")) return rc;
    if (ctx->name_held) TEC_FAIL(TEC_ERR_STATE, "tec_bulk_name_import_dev: held rows wait for tec_bulk_name_partition_dev");
    if (n < 0 || (n && !records)) TEC_FAIL(TEC_ERR_ARG, "tec_bulk_name_import_dev: bad arguments");
    TEC_CUDA(cudaSetDevice(ctx->device));
    NameState& s = *ctx->name;
    if (n) {
        if (int rc = name_reserve(ctx, s.pending + n)) return rc;
        TEC_CUDA(cudaEventRecord(s.ev[0], ctx->stream));
        NameRows d = s.rows[s.cur];
        const size_t p = (size_t)s.pending;
        d.start += p; d.end += p; d.chrom += p; d.mapq += p; d.flag += p; d.role += p; d.key_hi += p; d.key_lo += p;
        name_unpack_kernel<<<name_grid(ctx, n), NAME_TPB, 0, ctx->stream>>>(n, (const NameRecord*)records, d);
        TEC_CUDA(cudaGetLastError());
        ctx->launches++;
    }
    if (int rc = name_pair_batch(ctx, n)) return rc;  // synchronises when n > 0: the records may be freed
    TEC_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->cache.put(s.packed);
    s.packed = nullptr;
    return TEC_OK;
}

// Partition, all-gather of the send counts, grouped send / receive, import.  Every rank must call it.  The ranks agree on
// success before any record moves: the partition's status travels with the counts, and the status of the receive side's
// allocations in one more all-gather, so a rank that fails makes every rank return its status.
extern "C" int tec_bulk_name_exchange(tec_ctx* ctx, int64_t* n_owned) {
    if (!ctx) return TEC_ERR_ARG;
    if (!ctx->comm) TEC_FAIL(TEC_ERR_STATE, "tec_bulk_name_exchange: tec_comm_init not called");
    const int world = ctx->comm_world, rank = ctx->comm_rank;
    TEC_CUDA(cudaSetDevice(ctx->device));
    ncclComm_t comm = (ncclComm_t)ctx->comm;
    ScArena A(ctx->cache);
    const size_t w1 = (size_t)world + 1;
    u64* d_tab = nullptr;                       // [w1] mine: status, send counts; [world][w1] everyone's; [1] + [world] status words
    TEC_CUDA(A.get(&d_tab, w1 + (size_t)world * w1 + 1 + (size_t)world));
    u64* d_all = d_tab + w1;
    u64* d_st = d_all + (size_t)world * w1;
    // agreement: the first failing rank's status, the same on every rank
    auto agree = [&](const u64* st, size_t stride, int mine_rc, const char* step) -> int {
        for (int r = 0; r < world; ++r) {
            const int v = (int)(int64_t)st[(size_t)r * stride];
            if (!v) continue;
            if (r != rank || !mine_rc) ctx->err = std::string("tec_bulk_name_exchange: ") + step + " failed on rank " + std::to_string(r);
            return v;
        }
        return TEC_OK;
    };
    std::vector<int64_t> send((size_t)world, 0);
    void* packed = nullptr;
    const int prc = tec_bulk_name_partition_dev(ctx, world, send.data(), &packed);
    std::vector<u64> h_mine(w1), h_all((size_t)world * w1);
    h_mine[0] = (u64)(int64_t)prc;
    for (int r = 0; r < world; ++r) h_mine[(size_t)r + 1] = prc ? 0 : (u64)send[(size_t)r];
    TEC_CUDA(cudaMemcpyAsync(d_tab, h_mine.data(), w1 * 8, cudaMemcpyHostToDevice, ctx->stream));
    TEC_NCCL(g_nccl.AllGather(d_tab, d_all, w1, ncclUint64, comm, ctx->stream));
    TEC_CUDA(cudaMemcpyAsync(h_all.data(), d_all, h_all.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
    TEC_CUDA(cudaStreamSynchronize(ctx->stream));
    if (int rc = agree(h_all.data(), w1, prc, "the partition")) return rc;
    std::vector<int64_t> recv((size_t)world);
    int64_t n_recv = 0;
    for (int r = 0; r < world; ++r) { recv[(size_t)r] = (int64_t)h_all[(size_t)r * w1 + 1 + rank]; n_recv += recv[(size_t)r]; }
    // everything the receive side needs, before any record moves: the receive buffer and the pairing stage's rows
    char* dst = nullptr;
    int arc = name_reserve(ctx, ctx->name->pending + n_recv);
    if (!arc) {
        const cudaError_t e = A.get(&dst, (size_t)std::max<int64_t>(n_recv, 1) * sizeof(NameRecord));
        if (e != cudaSuccess) {
            ctx->err = std::string("tec_bulk_name_exchange: receive buffer: ") + cudaGetErrorString(e);
            arc = e == cudaErrorMemoryAllocation ? TEC_ERR_NOMEM : TEC_ERR_CUDA;
        }
    }
    std::vector<u64> h_st((size_t)world);
    const u64 mine = (u64)(int64_t)arc;
    TEC_CUDA(cudaMemcpyAsync(d_st, &mine, 8, cudaMemcpyHostToDevice, ctx->stream));
    TEC_NCCL(g_nccl.AllGather(d_st, d_st + 1, 1, ncclUint64, comm, ctx->stream));
    TEC_CUDA(cudaMemcpyAsync(h_st.data(), d_st + 1, (size_t)world * 8, cudaMemcpyDeviceToHost, ctx->stream));
    TEC_CUDA(cudaStreamSynchronize(ctx->stream));
    if (int rc = agree(h_st.data(), 1, arc, "the receive allocation")) return rc;
    // all-to-all: the received groups laid out by source rank, each in file order, are in file order
    TEC_NCCL(g_nccl.GroupStart());
    size_t so = 0, ro = 0;
    for (int r = 0; r < world; ++r) {
        const size_t sb = (size_t)send[(size_t)r] * sizeof(NameRecord), rb = (size_t)recv[(size_t)r] * sizeof(NameRecord);
        if (sb) TEC_NCCL(g_nccl.Send((const char*)packed + so, sb, ncclUint8, r, comm, ctx->stream));
        if (rb) TEC_NCCL(g_nccl.Recv(dst + ro, rb, ncclUint8, r, comm, ctx->stream));
        so += sb;
        ro += rb;
    }
    TEC_NCCL(g_nccl.GroupEnd());
    ctx->launches += 2;
    if (int rc = tec_bulk_name_import_dev(ctx, n_recv, dst)) return rc;    // synchronises: dst may go back to the cache
    if (n_owned) *n_owned = n_recv;
    return TEC_OK;
}
