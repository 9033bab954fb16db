// The cell x feature matrix of sc_save_result as a Matrix Market coordinate file in the orientation of 10x Genomics'
// filtered_feature_bc_matrix/matrix.mtx: one row per feature (ensg id order), one column per given cell.
//
// Layout: the rows of tec_sc_matrix_text (sc_text_rows) leave the selected cells' triples ascending in (column, ensg),
// which is the entry order of the file.  len[j] = byte length of entry line j ("<ensg + 1> <k + 1> <count>\n", at most
// 3 x 20 digits + 3 bytes), E = 64-bit exclusive prefix sum of len (the text passes 4 GiB above ~150 M entries), and
// line j starts at header + E[j].  One block takes 256 consecutive lines at a time: each thread formats its line into
// shared memory at E[j] - E[first], then the block copies that contiguous run to the text with consecutive threads on
// consecutive bytes, so every warp store covers one 32-byte sector.  The text is written once; the triples are read
// once.
#pragma once
#include "sc_text.cuh"

#define SC_MTX_BANNER "%%MatrixMarket matrix coordinate integer general\n"
#define SC_MTX_TILE 256
#define SC_MTX_LINE_MAX 63          // 3 fields of up to 20 digits, 2 spaces, '\n'

__global__ void sc_mtx_len_kernel(int64_t nnz, const u32* __restrict__ skey, const u32* __restrict__ sval,
                                  const int32_t* __restrict__ t_ensg, const int64_t* __restrict__ t_count, u64* __restrict__ len) {
    SC_LOOP(j, nnz + 1) {
        if (j == nnz) { len[j] = 0; continue; }
        const u32 src = sval[j];
        len[j] = (u64)(sc_text_ndigits((u64)t_ensg[src] + 1) + sc_text_ndigits((u64)skey[j] + 1) +
                       sc_text_ndigits((u64)t_count[src]) + 3);
    }
}

// v in decimal at p[0 .. d), d = sc_text_ndigits(v)
__device__ __forceinline__ void sc_mtx_put(char* p, u64 v, int d) {
    for (int i = d - 1; i >= 0; --i) { p[i] = (char)('0' + (int)(v % 10)); v /= 10; }
}

// "<a> <b> <c>\n" at p; returns its length
__device__ __forceinline__ int sc_mtx_line(char* p, u64 a, u64 b, u64 c) {
    const int da = sc_text_ndigits(a), db = sc_text_ndigits(b), dc = sc_text_ndigits(c);
    sc_mtx_put(p, a, da);
    p[da] = ' ';
    sc_mtx_put(p + da + 1, b, db);
    p[da + 1 + db] = ' ';
    sc_mtx_put(p + da + db + 2, c, dc);
    p[da + db + dc + 2] = '\n';
    return da + db + dc + 3;
}

__global__ void __launch_bounds__(SC_MTX_TILE) sc_mtx_write_kernel(
        int64_t nnz, int64_t n_ensg, int64_t n_cols, int64_t hdr, const u32* __restrict__ skey, const u32* __restrict__ sval,
        const u64* __restrict__ E, const int32_t* __restrict__ t_ensg, const int64_t* __restrict__ t_count, char* __restrict__ out) {
    __shared__ char stage[SC_MTX_TILE * SC_MTX_LINE_MAX];
    if (blockIdx.x == 0 && threadIdx.x == 0) {                 // the two header lines; hdr = their length (host)
        const char* banner = SC_MTX_BANNER;
        const int nb = (int)sizeof(SC_MTX_BANNER) - 1;
        for (int i = 0; i < nb; ++i) out[i] = banner[i];
        sc_mtx_line(out + nb, (u64)n_ensg, (u64)n_cols, (u64)nnz);
    }
    char* body = out + hdr;
    for (int64_t j0 = (int64_t)blockIdx.x * SC_MTX_TILE; j0 < nnz; j0 += (int64_t)gridDim.x * SC_MTX_TILE) {
        const int64_t j1 = j0 + SC_MTX_TILE < nnz ? j0 + SC_MTX_TILE : nnz;
        const u64 base = E[j0];
        const int64_t j = j0 + threadIdx.x;
        if (j < j1) {
            const u32 src = sval[j];
            sc_mtx_line(stage + (E[j] - base), (u64)t_ensg[src] + 1, (u64)skey[j] + 1, (u64)t_count[src]);
        }
        __syncthreads();
        const int run = (int)(E[j1] - base);
        for (int o = threadIdx.x; o < run; o += SC_MTX_TILE) body[base + o] = stage[o];
        __syncthreads();
    }
}

static int64_t sc_mtx_ndigits_host(int64_t v) {
    int64_t d = 1;
    while (v >= 10) { v /= 10; ++d; }
    return d;
}

extern "C" int tec_sc_matrix_mtx(tec_ctx* ctx, int64_t n_cols, const uint32_t* cells, int64_t* nnz, int64_t* n_bytes) {
    if (!ctx) return TEC_ERR_ARG;
    ScState* s = ctx->sc;
    if (!s || !s->finalized) TEC_FAIL(TEC_ERR_STATE, "tec_sc_matrix_mtx: tec_sc_finalize not called");
    if (n_cols < 0 || !nnz || !n_bytes || (n_cols && !cells)) TEC_FAIL(TEC_ERR_ARG, "tec_sc_matrix_mtx: bad arguments");
    if (n_cols >= (int64_t)SC_NONE - 1) TEC_FAIL(TEC_ERR_LIMIT, "tec_sc_matrix_mtx: too many columns");
    TEC_CUDA(cudaSetDevice(ctx->device));
    sc_text_free(ctx);
    *nnz = *n_bytes = 0;
    ScArena A(ctx->cache);
    u32 *skey = nullptr, *sval = nullptr, *row_ptr = nullptr;
    int64_t n_sel = 0;
    if (n_cols) {
        int rc = sc_text_rows(ctx, A, "tec_sc_matrix_mtx", n_cols, cells, &skey, &sval, &row_ptr, &n_sel);
        if (rc) return rc;
    }
    const int64_t n_ensg = ctx->idx.n_ensg;
    const int64_t hdr = (int64_t)sizeof(SC_MTX_BANNER) - 1 + sc_mtx_ndigits_host(n_ensg) + sc_mtx_ndigits_host(n_cols) +
                        sc_mtx_ndigits_host(n_sel) + 3;
    u64 *len, *E;
    TEC_CUDA(A.get(&len, (size_t)n_sel + 1));
    TEC_CUDA(A.get(&E, (size_t)n_sel + 1));
    sc_mtx_len_kernel<<<SC_GRID(n_sel + 1)>>>(n_sel, skey, sval, s->t_ensg, s->t_count, len);
    int rc = sc_excl_sum(ctx, len, E, n_sel + 1);
    if (rc) return rc;
    u64 h_body = 0;
    TEC_CUDA(cudaMemcpyAsync(&h_body, E + n_sel, 8, cudaMemcpyDeviceToHost, ctx->stream));
    TEC_CUDA(cudaStreamSynchronize(ctx->stream));
    const int64_t total = hdr + (int64_t)h_body;
    TEC_CUDA(ctx->cache.get((void**)&s->text, (size_t)total));
    s->text_bytes = total;
    const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((n_sel + SC_MTX_TILE - 1) / SC_MTX_TILE, (int64_t)ctx->n_sm * 8));
    sc_mtx_write_kernel<<<blocks, SC_MTX_TILE, 0, ctx->stream>>>(n_sel, n_ensg, n_cols, hdr, skey, sval, E, s->t_ensg, s->t_count,
                                                                 s->text);
    TEC_CUDA(cudaGetLastError());
    TEC_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->launches += 2;
    *nnz = n_sel;
    *n_bytes = total;
    return TEC_OK;
}
