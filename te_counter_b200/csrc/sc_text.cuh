// Dense matrix rows of sc_save_result as text, built on the device (SURVEY.md 8f-2).
//
// Reference te_count/te_count.py:744-754: one line per kept cell, in the order of :724-733
// (tec_sc_select): the barcode string, then '\t' + str(count) for EVERY ensg in sorted order --
// zeros included -- and '\n'.  For 10 k cells x 40-60 k features that is ~1 GB of text of which
// all but the non-zero entries are the two bytes "\t0".
//
// Layout: the (ensg, cell, count) triples of tec_sc_finalize are re-ordered by row with one stable
// radix sort on the row number (ensg stays ascending inside a row), E = exclusive prefix sum of
// (digits - 1) over that order.  Then every byte position is known in closed form:
//   row_start(r) = bc_off[r] + r * (2 * n_ensg + 1) + E[row_ptr[r]]
//   entry j = (row r, column c) starts at row_start(r) + bc_len(r) + 2 * c + E[j] - E[row_ptr[r]]
// and one warp per item (row head or non-zero entry) writes the item and the run of "\t0" that
// follows it up to the next item, with coalesced byte stores.  HBM-bound byte work: the text is
// written once; nothing is read but the triples.
#pragma once
#include "sc.cuh"

__global__ void sc_text_rank_kernel(int64_t n_rows, const u32* __restrict__ cells, u32* __restrict__ rank, int64_t n_wl, int* __restrict__ bad) {
    SC_LOOP(r, n_rows) {
        const u32 c = cells[r];
        if ((int64_t)c >= n_wl) { *bad = 1; continue; }
        if (atomicExch(rank + c, (u32)r) != SC_NONE) *bad = 2;          // the same cell twice
    }
}

__global__ void sc_text_rowkey_kernel(int64_t n, const u32* __restrict__ t_cell, const u32* __restrict__ rank, u32 n_rows,
                                      u32* __restrict__ key, u32* __restrict__ val) {
    SC_LOOP(i, n) {
        const u32 r = rank[t_cell[i]];
        key[i] = r == SC_NONE ? n_rows : r;
        val[i] = (u32)i;
    }
}

// row_ptr[r] = first sorted position with key >= r, for r in [0, n_rows + 1]
__global__ void sc_text_rowptr_kernel(int64_t n, const u32* __restrict__ skey, u32 n_rows, u32* __restrict__ row_ptr) {
    SC_LOOP(i, n + 1) {
        const u32 lo = i == 0 ? 0u : skey[i - 1] + 1u;
        const u32 hi = i == n ? n_rows + 1u : skey[i];
        for (u32 r = lo; r <= hi && r <= n_rows + 1u; ++r) row_ptr[r] = (u32)i;
    }
}

__device__ __forceinline__ int sc_text_ndigits(u64 v) {
    int d = 1;
    while (v >= 10) { v /= 10; ++d; }
    return d;
}

__global__ void sc_text_extra_kernel(int64_t n_sel, const u32* __restrict__ sval, const int64_t* __restrict__ t_count, u32* __restrict__ extra) {
    SC_LOOP(j, n_sel + 1) extra[j] = j < n_sel ? (u32)(sc_text_ndigits((u64)t_count[sval[j]]) - 1) : 0u;
}

__device__ __forceinline__ void sc_text_zero_run(char* __restrict__ out, int64_t at, int64_t len, int lane) {
    for (int64_t o = lane; o < len; o += 32) out[at + o] = (o & 1) ? '0' : '\t';
}

__global__ void sc_text_write_kernel(int64_t n_rows, int64_t n_sel, int64_t n_ensg, const u32* __restrict__ skey, const u32* __restrict__ sval,
                                     const u32* __restrict__ row_ptr, const u32* __restrict__ E, const int32_t* __restrict__ t_ensg,
                                     const int64_t* __restrict__ t_count, const char* __restrict__ bc, const int64_t* __restrict__ bc_off,
                                     char* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t row_fixed = 2 * n_ensg + 1;
    for (int64_t it = warp; it < n_rows + n_sel; it += n_warps) {
        int64_t r, run_at, col, j_next;
        if (it < n_rows) {                                  // row head: barcode, then zeros up to the first entry
            r = it;
            const int64_t b0 = bc_off[r], bl = bc_off[r + 1] - b0;
            const int64_t rs = b0 + r * row_fixed + (int64_t)E[row_ptr[r]];
            for (int64_t o = lane; o < bl; o += 32) out[rs + o] = bc[b0 + o];
            run_at = rs + bl;
            col = -1;
            j_next = row_ptr[r];
        } else {                                            // entry: '\t', digits, then zeros up to the next entry
            const int64_t j = it - n_rows;
            r = skey[j];
            const u32 src = sval[j];
            col = t_ensg[src];
            const int64_t b0 = bc_off[r], bl = bc_off[r + 1] - b0;
            const int64_t at = b0 + r * row_fixed + bl + 2 * col + (int64_t)E[j];   // E[row_ptr[r]] cancels against row_start
            const u64 v = (u64)t_count[src];
            const int d = (int)(E[j + 1] - E[j]) + 1;
            if (lane == 0) out[at] = '\t';
            if (lane < d) {
                u64 q = v;
                for (int k = d - 1 - lane; k > 0; --k) q /= 10;
                out[at + 1 + lane] = (char)('0' + (int)(q % 10));
            }
            run_at = at + 1 + d;
            j_next = j + 1;
        }
        const bool last = j_next >= (int64_t)row_ptr[r + 1];
        const int64_t col_next = last ? n_ensg : (int64_t)t_ensg[sval[j_next]];
        const int64_t len = 2 * (col_next - col - 1);
        sc_text_zero_run(out, run_at, len, lane);
        if (last && lane == 0) out[run_at + len] = '\n';
    }
}

static void sc_text_free(tec_ctx* ctx) {
    ScState* s = ctx->sc;
    ctx->cache.put(s->text);
    s->text = nullptr;
    s->text_bytes = 0;
}

// The rows of both matrix texts (this file and sc_mtx.cuh): the rank of each listed cell (TEC_ERR_ARG for an id outside
// the whitelist or listed twice), the triples stably sorted by that rank -- unlisted cells last, ensg ascending inside a
// rank, so the listed cells' triples are ascending in (rank, ensg) -- and row_ptr[r] = first sorted position of rank r
// for r in [0, n_rows + 1].  *n_sel = row_ptr[n_rows] = triples of the listed cells.  The buffers live in A.
static int sc_text_rows(tec_ctx* ctx, ScArena& A, const char* who, int64_t n_rows, const uint32_t* cells,
                        u32** skey_out, u32** sval_out, u32** row_ptr_out, int64_t* n_sel) {
    ScState* s = ctx->sc;
    const int64_t T = s->n_triples;
    u32 *d_cells, *rank, *key, *val, *skey, *sval, *row_ptr;
    int* d_bad;
    TEC_CUDA(A.get(&d_cells, (size_t)n_rows));
    TEC_CUDA(A.get(&rank, (size_t)s->n_wl));
    TEC_CUDA(A.get(&key, (size_t)T));
    TEC_CUDA(A.get(&val, (size_t)T));
    TEC_CUDA(A.get(&skey, (size_t)T));
    TEC_CUDA(A.get(&sval, (size_t)T));
    TEC_CUDA(A.get(&row_ptr, (size_t)n_rows + 2));
    TEC_CUDA(A.get(&d_bad, 1));
    TEC_CUDA(cudaMemcpyAsync(d_cells, cells, (size_t)n_rows * 4, cudaMemcpyHostToDevice, ctx->stream));
    TEC_CUDA(cudaMemsetAsync(d_bad, 0, 4, ctx->stream));
    TEC_CUDA(cudaMemsetAsync(rank, 0xFF, (size_t)s->n_wl * 4, ctx->stream));
    sc_text_rank_kernel<<<SC_GRID(n_rows)>>>(n_rows, d_cells, rank, s->n_wl, d_bad);
    if (T) {
        sc_text_rowkey_kernel<<<SC_GRID(T)>>>(T, s->t_cell, rank, (u32)n_rows, key, val);
        int rc = sc_sort_pairs(ctx, key, skey, val, sval, T, 0, ceil_log2_i64(n_rows + 2));
        if (rc) return rc;
    }
    sc_text_rowptr_kernel<<<SC_GRID(T + 1)>>>(T, skey, (u32)n_rows, row_ptr);
    u32 h_ptr = 0;
    int h_bad = 0;
    TEC_CUDA(cudaMemcpyAsync(&h_ptr, row_ptr + n_rows, 4, cudaMemcpyDeviceToHost, ctx->stream));
    TEC_CUDA(cudaMemcpyAsync(&h_bad, d_bad, 4, cudaMemcpyDeviceToHost, ctx->stream));
    TEC_CUDA(cudaStreamSynchronize(ctx->stream));
    if (h_bad) TEC_FAIL(TEC_ERR_ARG, std::string(who) + ": cell id outside the whitelist or listed twice");
    *skey_out = skey;
    *sval_out = sval;
    *row_ptr_out = row_ptr;
    *n_sel = h_ptr;
    return TEC_OK;
}

extern "C" int tec_sc_matrix_text(tec_ctx* ctx, int64_t n_rows, const uint32_t* cells, const char* barcodes,
                                  const int64_t* bc_off, int64_t* n_bytes) {
    if (!ctx) return TEC_ERR_ARG;
    ScState* s = ctx->sc;
    if (!s || !s->finalized) TEC_FAIL(TEC_ERR_STATE, "tec_sc_matrix_text: tec_sc_finalize not called");
    if (n_rows < 0 || !n_bytes || (n_rows && (!cells || !bc_off))) TEC_FAIL(TEC_ERR_ARG, "tec_sc_matrix_text: bad arguments");
    if (n_rows >= (int64_t)SC_NONE - 1) TEC_FAIL(TEC_ERR_LIMIT, "tec_sc_matrix_text: too many rows");
    TEC_CUDA(cudaSetDevice(ctx->device));
    sc_text_free(ctx);
    *n_bytes = 0;
    if (!n_rows) return TEC_OK;
    for (int64_t r = 0; r < n_rows; ++r)
        if (bc_off[r + 1] < bc_off[r] || bc_off[0] != 0) TEC_FAIL(TEC_ERR_ARG, "tec_sc_matrix_text: barcode offsets must ascend from 0");
    const int64_t n_ensg = ctx->idx.n_ensg, bc_bytes = bc_off[n_rows];
    if (bc_bytes && !barcodes) TEC_FAIL(TEC_ERR_ARG, "tec_sc_matrix_text: null barcodes");
    ScArena A(ctx->cache);
    u32 *skey, *sval, *row_ptr, *extra, *E;
    int64_t* d_off;
    char* d_bc;
    TEC_CUDA(A.get(&d_off, (size_t)n_rows + 1));
    TEC_CUDA(A.get(&d_bc, (size_t)bc_bytes));
    TEC_CUDA(cudaMemcpyAsync(d_off, bc_off, (size_t)(n_rows + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    if (bc_bytes) TEC_CUDA(cudaMemcpyAsync(d_bc, barcodes, (size_t)bc_bytes, cudaMemcpyHostToDevice, ctx->stream));
    int64_t n_sel = 0;
    int rc = sc_text_rows(ctx, A, "tec_sc_matrix_text", n_rows, cells, &skey, &sval, &row_ptr, &n_sel);
    if (rc) return rc;
    TEC_CUDA(A.get(&extra, (size_t)n_sel + 1));
    TEC_CUDA(A.get(&E, (size_t)n_sel + 1));
    sc_text_extra_kernel<<<SC_GRID(n_sel + 1)>>>(n_sel, sval, s->t_count, extra);
    rc = sc_excl_sum(ctx, extra, E, n_sel + 1);
    if (rc) return rc;
    u32 h_extra = 0;
    TEC_CUDA(cudaMemcpyAsync(&h_extra, E + n_sel, 4, cudaMemcpyDeviceToHost, ctx->stream));
    TEC_CUDA(cudaStreamSynchronize(ctx->stream));
    const int64_t total = bc_bytes + n_rows * (2 * n_ensg + 1) + (int64_t)h_extra;
    TEC_CUDA(ctx->cache.get((void**)&s->text, (size_t)total));
    s->text_bytes = total;
    const int64_t items = n_rows + n_sel;
    const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((items + 7) / 8, (int64_t)ctx->n_sm * 16));
    sc_text_write_kernel<<<blocks, 256, 0, ctx->stream>>>(n_rows, n_sel, n_ensg, skey, sval, row_ptr, E, s->t_ensg, s->t_count,
                                                          d_bc, d_off, s->text);
    TEC_CUDA(cudaGetLastError());
    TEC_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->launches += 5;
    *n_bytes = total;
    return TEC_OK;
}

extern "C" int tec_sc_matrix_read(tec_ctx* ctx, int64_t offset, int64_t n, char* out) {
    if (!ctx) return TEC_ERR_ARG;
    ScState* s = ctx->sc;
    if (!s || !s->text) TEC_FAIL(TEC_ERR_STATE, "tec_sc_matrix_read: tec_sc_matrix_text not called");
    if (offset < 0 || n < 0 || offset + n > s->text_bytes || (n && !out)) TEC_FAIL(TEC_ERR_ARG, "tec_sc_matrix_read: range outside the text");
    TEC_CUDA(cudaSetDevice(ctx->device));
    if (n) TEC_CUDA(cudaMemcpyAsync(out, s->text + offset, (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    TEC_CUDA(cudaStreamSynchronize(ctx->stream));
    return TEC_OK;
}
