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
#pragma once
#include "context.cuh"
#include "radix.cuh"
#include "bgzf_dev.h"

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
};

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
    if (s->h_cnt) cudaFreeHost(s->h_cnt);
    for (int i = 0; i < 2; ++i)
        if (s->ev[i]) cudaEventDestroy(s->ev[i]);
    delete s;
    name = nullptr;
}

// a new run: nothing pending, statistics of the stage back to zero (buffers are kept)
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

// device rows of one batch (the MODE_PE_NAME columns of the device decoder)
static int name_push_dev(tec_ctx* ctx, int64_t n, const bgzfdev::Columns& c) {
    if (n <= 0) return TEC_OK;
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
    return name_pair_batch(ctx, n);
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
