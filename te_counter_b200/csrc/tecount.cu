// libtecount.so -- C ABI implementation (see include/tecount.h).  sm_100a only, no CPU fallback.
#include "common.cuh"
#include "bulk.cuh"
#include "stab_build.h"
#include "context.cuh"
#include "collective.cuh"
#include "sc.cuh"
#include "sc_comm.cuh"
#include "sc_text.cuh"
#include "sc_mtx.cuh"
#include "bamgpu.cuh"
#include "pair_name.cuh"

#include <algorithm>
#include <cstdio>
#include <cstring>

// ------------------------------------------------------------------------------------ misc
extern "C" int tec_abi_version(void) { return TEC_ABI_VERSION; }

extern "C" const char* tec_strerror(int s) {
    switch (s) {
        case TEC_OK: return "ok";
        case TEC_ERR_CUDA: return "CUDA runtime error";
        case TEC_ERR_ARG: return "bad argument";
        case TEC_ERR_STATE: return "call out of order";
        case TEC_ERR_NOMEM: return "out of memory";
        case TEC_ERR_LIMIT: return "input exceeds a documented limit";
        case TEC_ERR_UNIMPLEMENTED: return "not implemented";
        case TEC_ERR_IO: return "file cannot be opened or read";
        case TEC_ERR_FORMAT: return "corrupt or truncated BAM / BGZF data";
        case TEC_ERR_UNSUPPORTED: return "file the device decoder refuses (decode it on the host)";
        case TEC_ERR_BAM_NO_BARCODE_TAG: return "record without CB / CR tag";
        case TEC_ERR_BAM_NO_UMI_TAG: return "record without UB / UR tag";
        case TEC_ERR_BAM_UMI: return "UMI that cannot be coded (longer than 21 characters or not ACGTN)";
        case TEC_ERR_BAM_END_NONE: return "mapped record without reference_end";
        case TEC_ERR_BAM_CHROM_NAME: return "reference name the chromosome key rule cannot take";
        case TEC_ERR_BAM_REF_NONE: return "record without a reference sequence";
        default: return "unknown status";
    }
}

extern "C" int tec_create(int device, tec_ctx** out) {
    if (!out) return TEC_ERR_ARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) return TEC_ERR_CUDA;   // no CPU fallback
    if (device < 0 || device >= n) return TEC_ERR_ARG;
    tec_ctx* ctx = new tec_ctx();
    ctx->device = device;
    auto fail = [&](int code) { tec_destroy(ctx); return code; };
    if (cudaSetDevice(device) != cudaSuccess) return fail(TEC_ERR_CUDA);
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return fail(TEC_ERR_CUDA);
    ctx->n_sm = prop.multiProcessorCount;
    ctx->smem_optin = (int)prop.sharedMemPerBlockOptin;
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) return fail(TEC_ERR_CUDA);
    if (cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) != cudaSuccess) return fail(TEC_ERR_CUDA);
    for (int i = 0; i < 2; ++i) {
        if (cudaEventCreateWithFlags(&ctx->stage_ready[i], cudaEventDisableTiming) != cudaSuccess) return fail(TEC_ERR_CUDA);
        if (cudaEventCreateWithFlags(&ctx->stage_free[i], cudaEventDisableTiming) != cudaSuccess) return fail(TEC_ERR_CUDA);
    }
    if (cudaEventCreate(&ctx->ev0) != cudaSuccess || cudaEventCreate(&ctx->ev1) != cudaSuccess) return fail(TEC_ERR_CUDA);
    *out = ctx;
    return TEC_OK;
}

extern "C" void tec_destroy(tec_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
    tec_comm_destroy(ctx);
    ctx->free_all();
    for (int i = 0; i < 2; ++i) {
        if (ctx->stage_ready[i]) cudaEventDestroy(ctx->stage_ready[i]);
        if (ctx->stage_free[i]) cudaEventDestroy(ctx->stage_free[i]);
    }
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    delete ctx;
}

extern "C" const char* tec_last_error(const tec_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

extern "C" int tec_sync(tec_ctx* ctx) {
    if (!ctx) return TEC_ERR_ARG;
    TEC_CUDA(cudaSetDevice(ctx->device));
    TEC_CUDA(cudaStreamSynchronize(ctx->copy_stream));
    TEC_CUDA(cudaStreamSynchronize(ctx->stream));
    return TEC_OK;
}

extern "C" int tec_host_alloc(tec_ctx* ctx, uint64_t bytes, void** out) {
    if (!ctx || !out) return TEC_ERR_ARG;
    TEC_CUDA(cudaSetDevice(ctx->device));
    TEC_CUDA(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault));
    return TEC_OK;
}

extern "C" int tec_host_free(tec_ctx* ctx, void* p) {
    if (!ctx) return TEC_ERR_ARG;
    TEC_CUDA(cudaFreeHost(p));
    return TEC_OK;
}

extern "C" int tec_trim(tec_ctx* ctx) {
    if (!ctx) return TEC_ERR_ARG;
    TEC_CUDA(cudaSetDevice(ctx->device));
    TEC_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->cache.trim();
    return TEC_OK;
}

extern "C" void* tec_stream(tec_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }
extern "C" float tec_last_kernel_ms(tec_ctx* ctx) {
    if (!ctx || !ctx->timed) return -1.f;
    float ms = -1.f;
    cudaSetDevice(ctx->device);
    if (cudaEventSynchronize(ctx->ev1) != cudaSuccess) return -1.f;
    if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) != cudaSuccess) return -1.f;
    return ms;
}
extern "C" int64_t tec_launch_count(const tec_ctx* ctx) { return ctx ? ctx->launches : 0; }

// ------------------------------------------------------------------------------------ index
__global__ void build_dir_kernel(const int32_t* __restrict__ L, const int64_t* __restrict__ chrom_off,
                                 const int64_t* __restrict__ dir_off, int n_chrom, int shift,
                                 u32* __restrict__ dir, int64_t n_dir) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_dir;
         i += (int64_t)gridDim.x * blockDim.x) {
        int c = 0;                                   // few chromosomes: linear scan of offsets
        while (c + 1 < n_chrom && dir_off[c + 1] <= i) ++c;
        const int64_t lo = chrom_off[c];
        const int64_t n = chrom_off[c + 1] - lo;
        const int64_t key = (i - dir_off[c]) << shift;           // first coordinate of the cell
        int64_t a = 0, b = n;                                    // #features with L < key
        while (a < b) {
            int64_t m = (a + b) >> 1;
            if ((int64_t)L[lo + m] < key) a = m + 1; else b = m;
        }
        dir[i] = (u32)a;
    }
}

extern "C" int tec_index_upload(tec_ctx* ctx, int32_t n_chrom, const int64_t* chrom_off,
                                const int32_t* L, const int32_t* R, const int32_t* ensg_id,
                                const uint8_t* type_code, const uint8_t* strand_code,
                                int32_t n_ensg, int32_t bucket_size) {
    if (!ctx) return TEC_ERR_ARG;
    if (n_chrom < 0 || n_chrom >= 0xFFF0 || !chrom_off || n_ensg < 0 || n_ensg > (1 << TEC_ENSG_BITS) || bucket_size <= 0)
        TEC_FAIL(TEC_ERR_ARG, "tec_index_upload: bad sizes");
    const int64_t nf = chrom_off[n_chrom];
    if (chrom_off[0] != 0 || nf < 0 || (nf > 0 && (!L || !R || !ensg_id || !type_code || !strand_code)))
        TEC_FAIL(TEC_ERR_ARG, "tec_index_upload: bad arrays");
    TEC_CUDA(cudaSetDevice(ctx->device));
    TEC_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->free_index();
    DevIndex& ix = ctx->idx;
    const int shift = 9;                            // 512 bp directory cells
    // slot = rank of the ensg by number of feature rows (most first): hot counters -> shared memory
    std::vector<int64_t> rows((size_t)std::max(n_ensg, 1), 0);
    for (int64_t i = 0; i < nf; ++i) {
        if (ensg_id[i] < 0 || ensg_id[i] >= n_ensg) TEC_FAIL(TEC_ERR_ARG, "tec_index_upload: ensg id out of range");
        rows[(size_t)ensg_id[i]]++;
    }
    ctx->ensg_of_slot.resize((size_t)n_ensg);
    for (int i = 0; i < n_ensg; ++i) ctx->ensg_of_slot[(size_t)i] = i;
    std::stable_sort(ctx->ensg_of_slot.begin(), ctx->ensg_of_slot.end(),
                     [&](int32_t a, int32_t b) { return rows[(size_t)a] > rows[(size_t)b]; });
    std::vector<uint32_t> slot_of((size_t)std::max(n_ensg, 1), 0);
    for (int s = 0; s < n_ensg; ++s) slot_of[(size_t)ctx->ensg_of_slot[(size_t)s]] = (uint32_t)s;
    std::vector<uint32_t> fslot((size_t)nf);
    std::vector<int32_t> pmax((size_t)nf);
    std::vector<u32> info((size_t)nf);
    std::vector<int64_t> dir_off((size_t)n_chrom + 1, 0);
    for (int c = 0; c < n_chrom; ++c) {
        const int64_t lo = chrom_off[c], hi = chrom_off[c + 1];
        if (hi < lo) TEC_FAIL(TEC_ERR_ARG, "tec_index_upload: chrom_off not monotone");
        if (hi - lo >= (int64_t)0x7FFFFFFF) TEC_FAIL(TEC_ERR_LIMIT, "tec_index_upload: chromosome with >= 2^31 features");
        int32_t run = INT32_MIN, maxL = 0;
        for (int64_t i = lo; i < hi; ++i) {
            if (L[i] < 0) TEC_FAIL(TEC_ERR_ARG, "tec_index_upload: negative feature start");
            if (R[i] > 0x7FFFFFF0) TEC_FAIL(TEC_ERR_ARG, "tec_index_upload: feature end too large");
            if (i > lo && L[i] < L[i - 1]) TEC_FAIL(TEC_ERR_ARG, "tec_index_upload: features not sorted by start within a chromosome");
            if (ensg_id[i] < 0 || ensg_id[i] >= n_ensg) TEC_FAIL(TEC_ERR_ARG, "tec_index_upload: ensg id out of range");
            if (type_code[i] > 7) TEC_FAIL(TEC_ERR_ARG, "tec_index_upload: type code out of range");
            run = std::max(run, R[i]);
            pmax[(size_t)i] = run;
            maxL = std::max(maxL, L[i]);
            fslot[(size_t)i] = slot_of[(size_t)ensg_id[i]];
            info[(size_t)i] = info_pack(fslot[(size_t)i], type_code[i], strand_code[i]);
        }
        dir_off[(size_t)c + 1] = dir_off[(size_t)c] + ((int64_t)(maxL >> shift) + 2);
    }
    // a chromosome is "in the index" iff it is a key of genelist.buckets; the key is created for every feature
    // row, before its bucket range is looked at (miniglbase/genelist.py:367-368)
    std::vector<uint8_t> chrom_valid((size_t)std::max(n_chrom, 1), 0);
    for (int c = 0; c < n_chrom; ++c) chrom_valid[(size_t)c] = chrom_off[c + 1] > chrom_off[c];
    const int64_t n_dir = dir_off[(size_t)n_chrom];
    ix.n_chrom = n_chrom; ix.n_feat = nf; ix.n_ensg = n_ensg; ix.bs = bucket_size; ix.shift = shift; ix.n_dir = n_dir;
    const size_t nfa = (size_t)std::max<int64_t>(nf, 1);
    TEC_CUDA(cudaMalloc(&ix.L, nfa * 4));
    TEC_CUDA(cudaMalloc(&ix.R, nfa * 4));
    TEC_CUDA(cudaMalloc(&ix.pmaxR, nfa * 4));
    TEC_CUDA(cudaMalloc(&ix.info, nfa * 4));
    TEC_CUDA(cudaMalloc(&ix.chrom_off, ((size_t)n_chrom + 1) * 8));
    TEC_CUDA(cudaMalloc(&ix.dir_off, ((size_t)n_chrom + 1) * 8));
    TEC_CUDA(cudaMalloc(&ix.dir, (size_t)std::max<int64_t>(n_dir, 1) * 4));
    TEC_CUDA(cudaMalloc(&ix.chrom_valid, chrom_valid.size()));
    TEC_CUDA(cudaMemcpyAsync(ix.chrom_valid, chrom_valid.data(), chrom_valid.size(), cudaMemcpyHostToDevice, ctx->stream));
    if (nf) {
        TEC_CUDA(cudaMemcpyAsync(ix.L, L, nfa * 4, cudaMemcpyHostToDevice, ctx->stream));
        TEC_CUDA(cudaMemcpyAsync(ix.R, R, nfa * 4, cudaMemcpyHostToDevice, ctx->stream));
        TEC_CUDA(cudaMemcpyAsync(ix.pmaxR, pmax.data(), nfa * 4, cudaMemcpyHostToDevice, ctx->stream));
        TEC_CUDA(cudaMemcpyAsync(ix.info, info.data(), nfa * 4, cudaMemcpyHostToDevice, ctx->stream));
    }
    TEC_CUDA(cudaMemcpyAsync(ix.chrom_off, chrom_off, ((size_t)n_chrom + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    TEC_CUDA(cudaMemcpyAsync(ix.dir_off, dir_off.data(), ((size_t)n_chrom + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    if (n_dir) {
        const int blocks = (int)std::min<int64_t>((n_dir + 255) / 256, (int64_t)ctx->n_sm * 16);
        build_dir_kernel<<<blocks, 256, 0, ctx->stream>>>(ix.L, ix.chrom_off, ix.dir_off, n_chrom, shift, ix.dir, n_dir);
        ctx->launches++;
        TEC_CUDA(cudaGetLastError());
    }
    // cell table, layout 2, for the two-pass bulk kernels (bulk2.cuh): the default bulk path
    {
        StabTable2 st;
        const int want = ctx->opt_stab_shift ? ctx->opt_stab_shift : TEC_BULK_STAB2_SHIFT;
        stab2_build(st, n_chrom, chrom_off, L, R, fslot.data(), type_code, n_ensg, want, bucket_size);
        if (st.why_not.empty()) {
            std::vector<uint2> cells((size_t)n_chrom + 1, make_uint2(0u, 0u));      // + sentinel for ids outside the index
            for (int c = 0; c < n_chrom; ++c)
                if (chrom_valid[(size_t)c])
                    cells[(size_t)c] = make_uint2((unsigned)st.cell_base[(size_t)c], (unsigned)(st.cell_base[(size_t)c + 1] - st.cell_base[(size_t)c]));
            TEC_CUDA(cudaMalloc(&ix.s2_sectors, std::max<size_t>(st.sectors.size(), 8) * 4));
            TEC_CUDA(cudaMalloc(&ix.s2_cells, cells.size() * sizeof(uint2)));
            TEC_CUDA(cudaMalloc(&ix.s2_slot_type, st.slot_type.size()));
            TEC_CUDA(cudaMalloc(&ix.s2_ovf_first, st.ovf_first.size() * 4));
            TEC_CUDA(cudaMemcpyAsync(ix.s2_sectors, st.sectors.data(), st.sectors.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
            TEC_CUDA(cudaMemcpyAsync(ix.s2_cells, cells.data(), cells.size() * sizeof(uint2), cudaMemcpyHostToDevice, ctx->stream));
            TEC_CUDA(cudaMemcpyAsync(ix.s2_slot_type, st.slot_type.data(), st.slot_type.size(), cudaMemcpyHostToDevice, ctx->stream));
            TEC_CUDA(cudaMemcpyAsync(ix.s2_ovf_first, st.ovf_first.data(), st.ovf_first.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
            TEC_CUDA(cudaStreamSynchronize(ctx->stream));
            ix.s2_shift = st.shift; ix.s2_ext = st.ext; ix.s2_all_counted = st.all_counted; ix.has_stab2 = true; ix.stab2_bytes = st.bytes();
            ix.s2_primary = st.n_primary; ix.s2_overflow = st.n_overflow; ix.s2_entries = st.n_entries;
            ix.s2_edge_cells = st.n_edge_cells; ix.s2_twin_sectors = st.n_twin_sectors;
        } else {
            ix.stab_why_not = st.why_not;
        }
    }
    // cell table, layout 1, of the round-1 kernel with in-kernel rings: only on request (bulk_algo=1)
    if (ctx->opt_bulk_algo == 1) {
        StabTable st;
        stab_build(st, n_chrom, chrom_off, L, R, fslot.data(), type_code, n_ensg, ctx->opt_stab_shift ? ctx->opt_stab_shift : TEC_BULK_STAB_SHIFT);
        if (st.why_not.empty()) {
            TEC_CUDA(cudaMalloc(&ix.st_sectors, std::max<size_t>(st.sectors.size(), 8) * 4));
            std::vector<uint2> cells((size_t)n_chrom + 1, make_uint2(0u, 0u));      // + sentinel for ids outside the index
            for (int c = 0; c < n_chrom; ++c)
                if (chrom_valid[(size_t)c])
                    cells[(size_t)c] = make_uint2((unsigned)st.cell_base[(size_t)c], (unsigned)(st.cell_base[(size_t)c + 1] - st.cell_base[(size_t)c]));
            TEC_CUDA(cudaMalloc(&ix.st_cells, cells.size() * sizeof(uint2)));
            TEC_CUDA(cudaMalloc(&ix.st_slot_type, st.slot_type.size()));
            TEC_CUDA(cudaMalloc(&ix.st_ovf_base, st.ovf_base.size() * 4));
            TEC_CUDA(cudaMemcpyAsync(ix.st_ovf_base, st.ovf_base.data(), st.ovf_base.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
            if (!st.sectors.empty())
                TEC_CUDA(cudaMemcpyAsync(ix.st_sectors, st.sectors.data(), st.sectors.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
            TEC_CUDA(cudaMemcpyAsync(ix.st_cells, cells.data(), cells.size() * sizeof(uint2), cudaMemcpyHostToDevice, ctx->stream));
            TEC_CUDA(cudaMemcpyAsync(ix.st_slot_type, st.slot_type.data(), st.slot_type.size(), cudaMemcpyHostToDevice, ctx->stream));
            TEC_CUDA(cudaStreamSynchronize(ctx->stream));
            ix.st_shift = st.shift; ix.st_all_counted = st.all_counted; ix.has_stab = true; ix.stab_bytes = st.bytes();
            ix.st_primary = st.n_primary; ix.st_overflow = st.n_overflow; ix.st_entries = st.n_entries;
        } else {
            ix.stab_why_not = st.why_not;
        }
    }
    // cell table of the single-cell Part 3: intervals [L-1, R+1), one slot per (ensg, strand) pair
    {
        std::vector<uint32_t> pkey((size_t)nf), uniq;
        for (int64_t i = 0; i < nf; ++i) pkey[(size_t)i] = (fslot[(size_t)i] << 3) | info_strand(info[(size_t)i]);
        uniq = pkey;
        std::sort(uniq.begin(), uniq.end());
        uniq.erase(std::unique(uniq.begin(), uniq.end()), uniq.end());
        if (uniq.size() <= STAB_MAX_SLOTS) {
            std::vector<uint32_t> pslot((size_t)nf);
            std::vector<int32_t> L1((size_t)nf), R1((size_t)nf);
            std::vector<uint8_t> ptype(std::max<size_t>(uniq.size(), 1), 0);
            for (int64_t i = 0; i < nf; ++i) {
                const uint32_t ps = (uint32_t)(std::lower_bound(uniq.begin(), uniq.end(), pkey[(size_t)i]) - uniq.begin());
                pslot[(size_t)i] = ps;
                ptype[ps] = type_code[i];
                L1[(size_t)i] = std::max(L[i] - 1, 0);
                // a feature whose bucket range is empty (R//bs < L//bs) is never a candidate (genelist.py:367-380)
                R1[(size_t)i] = (floordiv(R[i], bucket_size) < L[i] / bucket_size) ? L1[(size_t)i] : R[i] + 1;
            }
            StabTable st;
            stab_build(st, n_chrom, chrom_off, L1.data(), R1.data(), pslot.data(), type_code, (int)uniq.size(), ctx->opt_stab_shift ? ctx->opt_stab_shift : TEC_SC_STAB_SHIFT);
            if (st.why_not.empty()) {
                std::vector<uint2> cells((size_t)std::max(n_chrom, 1));
                for (int c = 0; c < n_chrom; ++c)
                    cells[(size_t)c] = make_uint2((unsigned)st.cell_base[(size_t)c], (unsigned)(st.cell_base[(size_t)c + 1] - st.cell_base[(size_t)c]));
                TEC_CUDA(cudaMalloc(&ix.sc_sectors, std::max<size_t>(st.sectors.size(), 8) * 4));
                TEC_CUDA(cudaMalloc(&ix.sc_cells, cells.size() * sizeof(uint2)));
                TEC_CUDA(cudaMalloc(&ix.sc_ovf_base, st.ovf_base.size() * 4));
                TEC_CUDA(cudaMalloc(&ix.sc_pair_key, std::max<size_t>(uniq.size(), 1) * 4));
                TEC_CUDA(cudaMalloc(&ix.sc_pair_type, ptype.size()));
                if (!st.sectors.empty())
                    TEC_CUDA(cudaMemcpyAsync(ix.sc_sectors, st.sectors.data(), st.sectors.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
                TEC_CUDA(cudaMemcpyAsync(ix.sc_cells, cells.data(), cells.size() * sizeof(uint2), cudaMemcpyHostToDevice, ctx->stream));
                TEC_CUDA(cudaMemcpyAsync(ix.sc_ovf_base, st.ovf_base.data(), st.ovf_base.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
                if (!uniq.empty())
                    TEC_CUDA(cudaMemcpyAsync(ix.sc_pair_key, uniq.data(), uniq.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
                TEC_CUDA(cudaMemcpyAsync(ix.sc_pair_type, ptype.data(), ptype.size(), cudaMemcpyHostToDevice, ctx->stream));
                TEC_CUDA(cudaStreamSynchronize(ctx->stream));
                ix.sc_shift = st.shift; ix.has_sc_stab = true; ix.sc_stab_bytes = st.bytes();
            }
        }
    }
    // bulk counter block; a run with loci grows it at tec_bulk_begin
    TEC_CUDA(cudaMalloc(&ctx->d_counts, ctx->bulk_words() * 8));
    ctx->counts_cap = (int64_t)ctx->bulk_words();
    TEC_CUDA(cudaMemsetAsync(ctx->d_counts, 0, ctx->bulk_words() * 8, ctx->stream));
    TEC_CUDA(cudaStreamSynchronize(ctx->stream));     // host staging vectors go out of scope
    ctx->has_index = true;
    return TEC_OK;
}

// ------------------------------------------------------------------------------------ bulk
extern "C" int tec_bulk_begin(tec_ctx* ctx, int paired, int qual) {
    if (!ctx) return TEC_ERR_ARG;
    if (!ctx->has_index) TEC_FAIL(TEC_ERR_STATE, "tec_bulk_begin: no index uploaded");
    TEC_CUDA(cudaSetDevice(ctx->device));
    ctx->paired = paired ? 1 : 0;
    ctx->name_pairing = paired == 2;
    ctx->qual = qual;
    ctx->bulk_active = false;
    ctx->name_held = false;
    ctx->loci = ctx->opt_bulk_loci != 0;
    if (ctx->name_pairing)
        if (int rc = name_begin(ctx)) return rc;
    if ((int64_t)ctx->bulk_words() > ctx->counts_cap) {
        TEC_CUDA(cudaStreamSynchronize(ctx->stream));
        cudaFree(ctx->d_counts);
        ctx->d_counts = nullptr;
        ctx->counts_cap = 0;
        TEC_CUDA(cudaMalloc(&ctx->d_counts, ctx->bulk_words() * 8));
        ctx->counts_cap = (int64_t)ctx->bulk_words();
    }
    TEC_CUDA(cudaMemsetAsync(ctx->d_counts, 0, ctx->bulk_words() * 8, ctx->stream));
    ctx->bulk_active = true;
    ctx->bank_pending = false;
    return TEC_OK;
}

// the checks of tec_bulk_push* / tec_bulk_finish / tec_bulk_allreduce: begun, no paired-end range waiting for its bank and no
// read-name range rows waiting for their partition
static int bulk_ready(tec_ctx* ctx, const char* what) {
    if (!ctx->bulk_active) TEC_FAIL(TEC_ERR_STATE, std::string(what) + ": tec_bulk_begin not called");
    if (ctx->bank_pending) TEC_FAIL(TEC_ERR_STATE, std::string(what) + ": a paired-end range count waits for tec_bulk_keep_bank");
    if (ctx->name_held) TEC_FAIL(TEC_ERR_STATE, std::string(what) + ": rows of a read-name range wait for tec_bulk_name_partition_dev");
    return TEC_OK;
}

// ... and for the pushes of records that are already pairs: not in the run of name pairing
static int bulk_ready_pairs(tec_ctx* ctx, const char* what) {
    if (int rc = bulk_ready(ctx, what)) return rc;
    if (ctx->name_pairing) TEC_FAIL(TEC_ERR_STATE, std::string(what) + ": the run pairs mates by read name (tec_bulk_push_named, tec_bam_count mode 3)");
    return TEC_OK;
}

#define TEC_LAUNCH_UNITS (int64_t(1) << 28)      // units per kernel launch (32-bit unit indices; slow list = 4 B per unit)

// the fast kernel of bulk2.cuh loads the records of two units with one instruction per column
static bool bulk2_aligned(int paired, const int32_t* start, const int32_t* end, const uint16_t* chrom, const uint8_t* mapq, const uint8_t* flag) {
    const uintptr_t a = paired ? 15 : 7, c = paired ? 7 : 3, b = paired ? 3 : 1;
    return !(((uintptr_t)start & a) || (!paired && ((uintptr_t)end & a)) || ((uintptr_t)chrom & c) || ((uintptr_t)mapq & b) || ((uintptr_t)flag & b));
}

// two-pass bulk kernels: fast kernel (two units per thread, one sector per unit), second pass over the deferred
// units, exact search on what the second pass flags
static int bulk2_launch_one(tec_ctx* ctx, int64_t n_units, const int32_t* start, const int32_t* end,
                            const uint16_t* chrom, const uint8_t* mapq, const uint8_t* flag) {
    IndexView iv = ctx->idx.view();
    Stab2View sv = ctx->idx.stab2_view();
    u64* counts = ctx->d_counts;
    u64* stats = ctx->d_counts + ctx->idx.n_ensg;
    const int64_t n_tiles = (n_units + 63) / 64;
    const size_t all_bytes = (size_t)ctx->idx.n_ensg * 4;
    const bool allhot = ctx->opt_all_hot != 0 && all_bytes + 2048 + 32 * B2_QCAP * 2 <= (size_t)ctx->smem_optin;
    // every counter in shared memory: one CTA per SM, of 1024 threads (64 registers) or, B2_MODE_DEEP, of 512 threads
    // with 128 registers and three tiles in flight per warp
    const bool deep = allhot && (ctx->opt_bulk_mode & B2_MODE_DEEP);
    const bool deep768 = deep && (ctx->opt_bulk_mode & B2_MODE_768);
    const int nt = allhot && !deep ? 1024 : deep768 ? 768 : 512;
    const u32 n_hot = allhot ? (u32)ctx->idx.n_ensg : (u32)std::min<int64_t>(TEC_HOT_SLOTS, ctx->idx.n_ensg);
    const int wpb = nt / 32;
    const size_t dyn = (size_t)n_hot * 4 + 128 + (size_t)wpb * B2_QCAP * 2;   // + one scratch word per lane, + the warps' hit queues
    const int per_sm = allhot ? 1 : ctx->opt_ctas_per_sm;
    const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((n_tiles + wpb - 1) / wpb, (int64_t)ctx->n_sm * per_sm));
    const int64_t n_warps = (int64_t)blocks * wpb;
    const int64_t seg_cap = ((n_tiles + n_warps - 1) / n_warps) * 64;
    if (n_warps * seg_cap > ctx->defer_cap || n_warps > ctx->defer_warps) {
        TEC_CUDA(cudaStreamSynchronize(ctx->stream));
        cudaFree(ctx->d_defer_list); cudaFree(ctx->d_defer_count);
        ctx->d_defer_list = nullptr; ctx->d_defer_count = nullptr; ctx->defer_cap = 0; ctx->defer_warps = 0;
        const int64_t cap = std::max<int64_t>(n_warps * seg_cap, 1 << 16), wcap = std::max<int64_t>(n_warps, 148 * 32);
        TEC_CUDA(cudaMalloc(&ctx->d_defer_list, (size_t)cap * 16));
        TEC_CUDA(cudaMalloc(&ctx->d_defer_count, (size_t)wcap * 4));
        ctx->defer_cap = cap; ctx->defer_warps = wcap;
    }
    if (n_units + 1 > ctx->slow_cap) {
        TEC_CUDA(cudaStreamSynchronize(ctx->stream));
        cudaFree(ctx->d_slow_list);
        ctx->d_slow_list = nullptr;
        ctx->slow_cap = 0;
        const int64_t cap = std::max<int64_t>(n_units + 1, 1 << 16);
        TEC_CUDA(cudaMalloc(&ctx->d_slow_list, (size_t)cap * 4));
        ctx->slow_cap = cap;
    }
    TEC_CUDA(cudaMemsetAsync(ctx->d_slow_list, 0, 4, ctx->stream));
    ctx->last_defer_n = n_warps;
#define TEC_LAUNCH_FAST2(P, NT, AH, DP)                                                                                    \
    do {                                                                                                                   \
        auto kfn = (ctx->opt_bulk_mode & B2_MODE_SCAN) ? bulk2_fast_kernel<P, NT, AH, 2, DP>                               \
                   : (ctx->opt_bulk_mode & B2_MODE_QUEUE) ? ((ctx->opt_bulk_mode & B2_MODE_TILE_DRAIN) ? bulk2_fast_kernel<P, NT, AH, 3, DP> : bulk2_fast_kernel<P, NT, AH, 1, DP>) \
                   : bulk2_fast_kernel<P, NT, AH, 0, DP>; \
        TEC_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));                        \
        kfn<<<blocks, NT, dyn, ctx->stream>>>(sv, ctx->idx.n_chrom, (u32)n_units, ctx->qual, start, end, chrom, mapq, flag, \
                                              counts, stats, (uint4*)ctx->d_defer_list, ctx->d_defer_count, (u32)seg_cap, n_hot, \
                                              (u32)ctx->opt_bulk_mode);                                                    \
    } while (0)
    if (ctx->paired) {
        if (deep768) TEC_LAUNCH_FAST2(true, 768, true, 2);
        else if (deep) TEC_LAUNCH_FAST2(true, 512, true, 3);
        else if (allhot) TEC_LAUNCH_FAST2(true, 1024, true, 0);
        else TEC_LAUNCH_FAST2(true, 512, false, 0);
    } else {
        if (deep768) TEC_LAUNCH_FAST2(false, 768, true, 2);
        else if (deep) TEC_LAUNCH_FAST2(false, 512, true, 3);
        else if (allhot) TEC_LAUNCH_FAST2(false, 1024, true, 0);
        else TEC_LAUNCH_FAST2(false, 512, false, 0);
    }
#undef TEC_LAUNCH_FAST2
    ctx->launches++;
    TEC_CUDA(cudaGetLastError());
    const int parts = std::max(1, ctx->opt_second_parts);
    const int b2 = (int)std::min<int64_t>((n_warps * parts + 7) / 8, (int64_t)ctx->n_sm * 6);
    // units that two sectors answer go through the straight-line kernel first; it leaves the rest in place
    const bool pair_pass = ctx->opt_second_mode >= 2 && sv.all_counted;
    const u32* part_count = nullptr;
    if (pair_pass) {
        if (n_warps * parts > ctx->part_cap) {
            TEC_CUDA(cudaStreamSynchronize(ctx->stream));
            cudaFree(ctx->d_part_count);
            ctx->d_part_count = nullptr; ctx->part_cap = 0;
            const int64_t cap = std::max<int64_t>(n_warps * parts, 148 * 32 * 4);
            TEC_CUDA(cudaMalloc(&ctx->d_part_count, (size_t)cap * 4));
            ctx->part_cap = cap;
        }
        if (ctx->paired)
            bulk2_pair_kernel<true><<<b2, 256, 0, ctx->stream>>>(sv, counts, stats, (uint4*)ctx->d_defer_list, ctx->d_defer_count, (u32)seg_cap,
                                                                 (u32)n_warps, (u32)parts, ctx->d_part_count, (u32)ctx->idx.n_chrom);
        else
            bulk2_pair_kernel<false><<<b2, 256, 0, ctx->stream>>>(sv, counts, stats, (uint4*)ctx->d_defer_list, ctx->d_defer_count, (u32)seg_cap,
                                                                  (u32)n_warps, (u32)parts, ctx->d_part_count, (u32)ctx->idx.n_chrom);
        ctx->launches++;
        TEC_CUDA(cudaGetLastError());
        part_count = ctx->d_part_count;
        ctx->last_part_n = n_warps * parts;
    } else {
        ctx->last_part_n = 0;
    }
#define TEC_LAUNCH_SECOND(P, SET)                                                                                              \
    bulk2_second_kernel<P, SET><<<b2, 256, 0, ctx->stream>>>(sv, counts, stats, (const uint4*)ctx->d_defer_list, ctx->d_defer_count, \
                                                             (u32)seg_cap, (u32)n_warps, (u32)parts, ctx->d_slow_list, (u32)ctx->idx.n_chrom, part_count)
    if (ctx->paired) { if (ctx->opt_second_mode) TEC_LAUNCH_SECOND(true, 1); else TEC_LAUNCH_SECOND(true, 0); }
    else { if (ctx->opt_second_mode) TEC_LAUNCH_SECOND(false, 1); else TEC_LAUNCH_SECOND(false, 0); }
#undef TEC_LAUNCH_SECOND
    ctx->launches++;
    TEC_CUDA(cudaGetLastError());
    // exact search on the units of EDGE cells / large ensg sets (has_stab = 0: no layout-1 table lookups)
    const int sblocks = (int)std::min<int64_t>((n_units + 255) / 256, (int64_t)ctx->n_sm * 4);
    StabView none = StabView();
    if (ctx->paired)
        bulk_slow_kernel<true><<<sblocks, 256, 0, ctx->stream>>>(iv, none, 0, start, end, chrom, counts, stats, ctx->d_slow_list);
    else
        bulk_slow_kernel<false><<<sblocks, 256, 0, ctx->stream>>>(iv, none, 0, start, end, chrom, counts, stats, ctx->d_slow_list);
    ctx->launches++;
    TEC_CUDA(cudaGetLastError());
    return TEC_OK;
}

static int bulk_launch_one(tec_ctx* ctx, int64_t n_units, const int32_t* start, const int32_t* end,
                           const uint16_t* chrom, const uint8_t* mapq, const uint8_t* flag) {
    IndexView iv = ctx->idx.view();
    u64* counts = ctx->d_counts;
    u64* stats = ctx->d_counts + ctx->idx.n_ensg;
    if (ctx->loci) {          // the row tally lives in the exact kernel only; it also gives the per-name counts and statistics
        const int64_t want = (n_units + 255) / 256;
        const int blocks = (int)std::min<int64_t>(want, (int64_t)ctx->n_sm * 8);
        if (ctx->paired)
            bulk_count_kernel<true, true><<<blocks, 256, 0, ctx->stream>>>(iv, n_units, ctx->qual, ctx->opt_bulk_strand, start, end, chrom, mapq, flag, counts, stats);
        else
            bulk_count_kernel<false, true><<<blocks, 256, 0, ctx->stream>>>(iv, n_units, ctx->qual, ctx->opt_bulk_strand, start, end, chrom, mapq, flag, counts, stats);
        ctx->launches++;
        TEC_CUDA(cudaGetLastError());
        return TEC_OK;
    }
    const bool use_stab2 = !ctx->opt_bulk_strand && ctx->idx.has_stab2 && (ctx->opt_bulk_algo == -1 || ctx->opt_bulk_algo == 2) &&
                           bulk2_aligned(ctx->paired, start, end, chrom, mapq, flag);
    if (use_stab2) return bulk2_launch_one(ctx, n_units, start, end, chrom, mapq, flag);
    const bool use_stab = !ctx->opt_bulk_strand && ctx->idx.has_stab && ctx->opt_bulk_algo == 1;   // the strand extension lives in the exact kernel only
    if (use_stab) {
        // fast kernel: one warp per 32 units, persistent grid; then the exact kernel on flagged units
        const int64_t n_tiles = (n_units + 31) / 32;
        if (n_units + 1 > ctx->slow_cap) {
            TEC_CUDA(cudaStreamSynchronize(ctx->stream));
            cudaFree(ctx->d_slow_list);
            ctx->d_slow_list = nullptr;
            ctx->slow_cap = 0;
            TEC_CUDA(cudaMalloc(&ctx->d_slow_list, (size_t)(n_units + 1) * 4));
            ctx->slow_cap = n_units + 1;
        }
        TEC_CUDA(cudaMemsetAsync(ctx->d_slow_list, 0, 4, ctx->stream));
        StabView sv = ctx->idx.stab_view();
        // every ensg counter in shared memory when they fit beside the rings (one 1024-thread CTA per SM);
        // otherwise the TEC_HOT_SLOTS hottest ones (two 512-thread CTAs per SM)
        const size_t all_bytes = (size_t)ctx->idx.n_ensg * 4;
        const bool allhot = ctx->opt_all_hot != 0 && all_bytes + 45 * 1024 <= (size_t)ctx->smem_optin;
        const int nt = allhot ? 1024 : 512;
        const u32 n_hot = allhot ? (u32)ctx->idx.n_ensg : (u32)std::min<int64_t>(TEC_HOT_SLOTS, ctx->idx.n_ensg);
        const size_t dyn = (size_t)n_hot * 4 + 128;            // + one scratch word per lane (bump_entry)
        const int per_sm = allhot ? 1 : ctx->opt_ctas_per_sm;
        const int blocks = (int)std::min<int64_t>((n_tiles + nt / 32 - 1) / (nt / 32), (int64_t)ctx->n_sm * per_sm);
        const int64_t ring_entries = (int64_t)blocks * (nt / 32) * BULK_QCAP;
        if (ring_entries > ctx->ring_cap) {
            TEC_CUDA(cudaStreamSynchronize(ctx->stream));
            cudaFree(ctx->d_ring); cudaFree(ctx->d_ring_u);
            ctx->d_ring = nullptr; ctx->d_ring_u = nullptr; ctx->ring_cap = 0;
            TEC_CUDA(cudaMalloc(&ctx->d_ring, (size_t)ring_entries * sizeof(QEnt)));
            TEC_CUDA(cudaMalloc(&ctx->d_ring_u, (size_t)ring_entries * 4));
            ctx->ring_cap = ring_entries;
        }
#define TEC_LAUNCH_CELL(P, NT, AH)                                                                                         \
        do {                                                                                                               \
            auto kfn = bulk_count_cell_kernel<P, NT, AH>;                                                                  \
            TEC_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));                    \
            kfn<<<blocks, NT, dyn, ctx->stream>>>(iv, sv, n_units, ctx->qual, start, end, chrom, mapq, flag, counts, stats, \
                                                  ctx->d_slow_list, n_hot, (QEnt*)ctx->d_ring, ctx->d_ring_u);            \
        } while (0)
        if (ctx->paired) { if (allhot) TEC_LAUNCH_CELL(true, 1024, true); else TEC_LAUNCH_CELL(true, 512, false); }
        else { if (allhot) TEC_LAUNCH_CELL(false, 1024, true); else TEC_LAUNCH_CELL(false, 512, false); }
#undef TEC_LAUNCH_CELL
        ctx->launches++;
        TEC_CUDA(cudaGetLastError());
        const int sblocks = (int)std::min<int64_t>((n_units + 255) / 256, (int64_t)ctx->n_sm * 8);
        if (ctx->paired)
            bulk_slow_kernel<true><<<sblocks, 256, 0, ctx->stream>>>(iv, sv, 1, start, end, chrom, counts, stats, ctx->d_slow_list);
        else
            bulk_slow_kernel<false><<<sblocks, 256, 0, ctx->stream>>>(iv, sv, 1, start, end, chrom, counts, stats, ctx->d_slow_list);
        ctx->launches++;
        TEC_CUDA(cudaGetLastError());
        return TEC_OK;
    }
    const int threads = 256;
    const int64_t want = (n_units + threads - 1) / threads;
    const int blocks = (int)std::min<int64_t>(want, (int64_t)ctx->n_sm * 8);
    if (ctx->paired)
        bulk_count_kernel<true, false><<<blocks, threads, 0, ctx->stream>>>(iv, n_units, ctx->qual, ctx->opt_bulk_strand, start, end, chrom, mapq, flag, counts, stats);
    else
        bulk_count_kernel<false, false><<<blocks, threads, 0, ctx->stream>>>(iv, n_units, ctx->qual, ctx->opt_bulk_strand, start, end, chrom, mapq, flag, counts, stats);
    ctx->launches++;
    TEC_CUDA(cudaGetLastError());
    return TEC_OK;
}

static int bulk_launch(tec_ctx* ctx, int64_t n_rec, const int32_t* start, const int32_t* end,
                       const uint16_t* chrom, const uint8_t* mapq, const uint8_t* flag) {
    const int64_t n_units = ctx->paired ? n_rec / 2 : n_rec;
    if (ctx->opt_bulk_algo == 1 && !ctx->idx.has_stab) TEC_FAIL(TEC_ERR_STATE, "bulk_algo=1 but the index has no layout-1 cell table (set the option before tec_index_upload)");
    if (ctx->opt_bulk_algo == 2 && !ctx->idx.has_stab2) TEC_FAIL(TEC_ERR_STATE, "bulk_algo=2 but the index has no cell table: " + ctx->idx.stab_why_not);
    const int64_t rpu = ctx->paired ? 2 : 1;
    for (int64_t off = 0; off < n_units; off += TEC_LAUNCH_UNITS) {
        const int64_t n = std::min<int64_t>(TEC_LAUNCH_UNITS, n_units - off);
        const int64_t r = off * rpu;
        int rc = bulk_launch_one(ctx, n, start + r, end + r, chrom + r, mapq + r, flag + r);
        if (rc) return rc;
    }
    return TEC_OK;
}

static int bulk_push_dev(tec_ctx* ctx, int64_t n_rec, const int32_t* start, const int32_t* end,
                         const uint16_t* chrom, const uint8_t* mapq, const uint8_t* flag) {
    if (n_rec < 0 || (ctx->paired && (n_rec & 1))) TEC_FAIL(TEC_ERR_ARG, "tec_bulk_push_dev: record count must be even in paired mode");
    if (n_rec == 0) return TEC_OK;
    if (!start || !end || !chrom || !mapq || !flag) TEC_FAIL(TEC_ERR_ARG, "tec_bulk_push_dev: null array");
    if (((uintptr_t)start & 7) || ((uintptr_t)end & 3) || ((uintptr_t)chrom & 3) || ((uintptr_t)mapq & 1) || ((uintptr_t)flag & 1))
        TEC_FAIL(TEC_ERR_ARG, "tec_bulk_push_dev: misaligned array");
    TEC_CUDA(cudaSetDevice(ctx->device));
    TEC_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
    int rc = bulk_launch(ctx, n_rec, start, end, chrom, mapq, flag);
    if (rc) return rc;
    TEC_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
    ctx->timed = true;
    return TEC_OK;
}

extern "C" int tec_bulk_push_dev(tec_ctx* ctx, int64_t n_rec, const int32_t* start, const int32_t* end,
                                 const uint16_t* chrom, const uint8_t* mapq, const uint8_t* flag) {
    if (!ctx) return TEC_ERR_ARG;
    if (int rc = bulk_ready_pairs(ctx, "tec_bulk_push_dev")) return rc;
    return bulk_push_dev(ctx, n_rec, start, end, chrom, mapq, flag);
}

// Host buffers: chunks are copied on the copy stream into one of two staging slots while the
// previous chunk is counted on the compute stream.
extern "C" int tec_bulk_push(tec_ctx* ctx, int64_t n_rec, const int32_t* start, const int32_t* end,
                             const uint16_t* chrom, const uint8_t* mapq, const uint8_t* flag) {
    if (!ctx) return TEC_ERR_ARG;
    if (int rc = bulk_ready_pairs(ctx, "tec_bulk_push")) return rc;
    if (n_rec < 0 || (ctx->paired && (n_rec & 1))) TEC_FAIL(TEC_ERR_ARG, "tec_bulk_push: record count must be even in paired mode");
    if (n_rec == 0) return TEC_OK;
    if (!start || !end || !chrom || !mapq || !flag) TEC_FAIL(TEC_ERR_ARG, "tec_bulk_push: null array");
    TEC_CUDA(cudaSetDevice(ctx->device));
    const int64_t chunk = TEC_STAGE_RECORDS;
    int rc = ctx->ensure_stage(std::min<int64_t>(n_rec, chunk), /*sc=*/false);
    if (rc) return rc;
    TEC_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
    for (int64_t off = 0; off < n_rec; off += chunk) {
        const int64_t n = std::min<int64_t>(chunk, n_rec - off);
        const int s = ctx->stage_next;
        ctx->stage_next ^= 1;
        StageSlot& sl = ctx->stage[s];
        TEC_CUDA(cudaStreamWaitEvent(ctx->copy_stream, ctx->stage_free[s], 0));
        TEC_CUDA(cudaMemcpyAsync(sl.start, start + off, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->copy_stream));
        // the paired-end rules never look at reference_end (te_count.py:97-98 take both mates' starts)
        if (!ctx->paired)
            TEC_CUDA(cudaMemcpyAsync(sl.end, end + off, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->copy_stream));
        TEC_CUDA(cudaMemcpyAsync(sl.chrom, chrom + off, (size_t)n * 2, cudaMemcpyHostToDevice, ctx->copy_stream));
        TEC_CUDA(cudaMemcpyAsync(sl.mapq, mapq + off, (size_t)n, cudaMemcpyHostToDevice, ctx->copy_stream));
        TEC_CUDA(cudaMemcpyAsync(sl.flag, flag + off, (size_t)n, cudaMemcpyHostToDevice, ctx->copy_stream));
        TEC_CUDA(cudaEventRecord(ctx->stage_ready[s], ctx->copy_stream));
        TEC_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->stage_ready[s], 0));
        rc = bulk_launch(ctx, n, sl.start, sl.end, sl.chrom, sl.mapq, sl.flag);
        if (rc) return rc;
        TEC_CUDA(cudaEventRecord(ctx->stage_free[s], ctx->stream));
    }
    TEC_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
    ctx->timed = true;
    // the caller may reuse its host buffers as soon as we return
    TEC_CUDA(cudaStreamSynchronize(ctx->copy_stream));
    return TEC_OK;
}

extern "C" int tec_bulk_push_named(tec_ctx* ctx, int64_t n, const int32_t* start, const int32_t* end, const uint16_t* chrom,
                                   const uint8_t* mapq, const uint8_t* flag, const uint16_t* samflag, const int64_t* name_off,
                                   const char* names) {
    if (!ctx) return TEC_ERR_ARG;
    if (int rc = bulk_ready(ctx, "tec_bulk_push_named")) return rc;
    if (!ctx->name_pairing) TEC_FAIL(TEC_ERR_STATE, "tec_bulk_push_named: tec_bulk_begin was not called with paired = 2");
    if (n < 0) TEC_FAIL(TEC_ERR_ARG, "tec_bulk_push_named: negative record count");
    if (n == 0) return TEC_OK;
    if (!start || !end || !chrom || !mapq || !flag || !samflag || !name_off || (name_off[n] > 0 && !names))
        TEC_FAIL(TEC_ERR_ARG, "tec_bulk_push_named: null array");
    if (name_off[0] != 0) TEC_FAIL(TEC_ERR_ARG, "tec_bulk_push_named: name_off[0] must be 0");
    for (int64_t i = 0; i < n; ++i)
        if (name_off[i + 1] < name_off[i] || name_off[i + 1] - name_off[i] > 254)
            TEC_FAIL(TEC_ERR_ARG, "tec_bulk_push_named: name_off must ascend by at most 254 bytes per name");
    TEC_CUDA(cudaSetDevice(ctx->device));
    return name_push_host(ctx, n, start, end, chrom, mapq, flag, samflag, name_off, names);
}

extern "C" int tec_bulk_finish(tec_ctx* ctx, int64_t* counts, int64_t* stats) {
    if (!ctx) return TEC_ERR_ARG;
    if (int rc = bulk_ready(ctx, "tec_bulk_finish")) return rc;
    TEC_CUDA(cudaSetDevice(ctx->device));
    if (int rc = name_flush(ctx)) return rc;
    const size_t ne = (size_t)ctx->idx.n_ensg;
    std::vector<int64_t> tmp(ne + TEC_BULK_NSTATS);
    TEC_CUDA(cudaMemcpyAsync(tmp.data(), ctx->d_counts, (ne + TEC_BULK_NSTATS) * 8, cudaMemcpyDeviceToHost, ctx->stream));
    TEC_CUDA(cudaStreamSynchronize(ctx->stream));
    if (counts)
        for (size_t s = 0; s < ne; ++s) counts[(size_t)ctx->ensg_of_slot[s]] = tmp[s];     // slot order -> ensg order
    if (stats) memcpy(stats, tmp.data() + ne, TEC_BULK_NSTATS * 8);
    return TEC_OK;
}

extern "C" int tec_bulk_loci(tec_ctx* ctx, int64_t* counts) {
    if (!ctx) return TEC_ERR_ARG;
    if (int rc = bulk_ready(ctx, "tec_bulk_loci")) return rc;
    if (!ctx->loci) TEC_FAIL(TEC_ERR_STATE, "tec_bulk_loci: the run did not begin with the option bulk_loci");
    if (!counts) TEC_FAIL(TEC_ERR_ARG, "tec_bulk_loci: counts is NULL");
    TEC_CUDA(cudaSetDevice(ctx->device));
    if (int rc = name_flush(ctx)) return rc;
    const size_t nf = (size_t)ctx->idx.n_feat;
    if (nf) TEC_CUDA(cudaMemcpyAsync(counts, ctx->d_counts + ctx->idx.n_ensg + TEC_BULK_NSTATS, nf * 8, cudaMemcpyDeviceToHost, ctx->stream));
    TEC_CUDA(cudaStreamSynchronize(ctx->stream));
    return TEC_OK;
}

extern "C" void* tec_bulk_counts_dev(tec_ctx* ctx) { return ctx ? (void*)ctx->d_counts : nullptr; }

extern "C" int tec_bulk_keep_bank(tec_ctx* ctx, int bank) {
    if (!ctx) return TEC_ERR_ARG;
    if (!ctx->bulk_active || !ctx->bank_pending) TEC_FAIL(TEC_ERR_STATE, "tec_bulk_keep_bank: no paired-end range count waits for it");
    if (bank != 0 && bank != 1) TEC_FAIL(TEC_ERR_ARG, "tec_bulk_keep_bank: bank must be 0 or 1");
    TEC_CUDA(cudaSetDevice(ctx->device));
    if (bank == 1)
        TEC_CUDA(cudaMemcpyAsync(ctx->d_counts, ctx->d_bank1, ctx->bulk_words() * 8, cudaMemcpyDeviceToDevice, ctx->stream));
    ctx->bank_pending = false;
    return TEC_OK;
}

extern "C" int tec_set_option(tec_ctx* ctx, const char* key, int64_t value) {
    if (!ctx || !key) return TEC_ERR_ARG;
    const std::string k(key);
    if (k == "bulk_algo") { if (value < -1 || value > 2) TEC_FAIL(TEC_ERR_ARG, "bulk_algo: -1, 0, 1 or 2"); ctx->opt_bulk_algo = (int)value; }
    else if (k == "stab_shift") { if (value && (value < 8 || value > STAB_MAX_SHIFT)) TEC_FAIL(TEC_ERR_ARG, "stab_shift: 0 (default) or 8..11"); ctx->opt_stab_shift = (int)value; }
    else if (k == "sc_algo") { if (value < -1 || value > 1) TEC_FAIL(TEC_ERR_ARG, "sc_algo: -1, 0 or 1"); ctx->opt_sc_algo = (int)value; }
    else if (k == "sc_pack_umi") { ctx->opt_sc_pack_umi = value ? 1 : 0; }
    else if (k == "all_hot") { ctx->opt_all_hot = value ? 1 : 0; }
    else if (k == "sc_sort") { if (value < 0 || value > 1) TEC_FAIL(TEC_ERR_ARG, "sc_sort: 0 library sort in two stages, 1 packed keys + csrc/radix.cuh"); ctx->opt_sc_sort = (int)value; }
    else if (k == "bulk_strand") { ctx->opt_bulk_strand = value ? 1 : 0; }     // opt-in extension, outside the parity claim (bulk.cuh)
    else if (k == "bulk_loci") { if (value < 0 || value > 1) TEC_FAIL(TEC_ERR_ARG, "bulk_loci: 0 or 1"); ctx->opt_bulk_loci = (int)value; }
    else if (k == "sc_prev_partition") { if (value < 0 || value > 2) TEC_FAIL(TEC_ERR_ARG, "sc_prev_partition: 0 random stores, 1 radix pass on large inputs, 2 always"); ctx->opt_sc_prev_partition = (int)value; }
    else if (k == "sc_sort_chunk") { if (value < 1 || value > 64) TEC_FAIL(TEC_ERR_ARG, "sc_sort_chunk: tiles per chunk of csrc/radix.cuh, 1..64"); g_rdx_chunk_tiles = (int)value; }
    else if (k == "second_parts") { if (value < 1 || value > 16) TEC_FAIL(TEC_ERR_ARG, "second_parts: 1..16"); ctx->opt_second_parts = (int)value; }
    else if (k == "second_mode") { if (value < 0 || value > 2) TEC_FAIL(TEC_ERR_ARG, "second_mode: 0 distinct ensg stored by position, 1 shifted in, 2 two-sector kernel first"); ctx->opt_second_mode = (int)value; }
    else if (k == "bulk_mode") { if (value < 0 || value > 127) TEC_FAIL(TEC_ERR_ARG, "bulk_mode: bit 0 table evict_last, bit 1 sector prefetch, bit 2 tally through the hit queue, bit 3 deep pipeline, bit 4 hit queue filled once per tile, bit 5 768-thread CTAs with two tiles in flight, bit 6 ballot queue drained once per tile"); ctx->opt_bulk_mode = (int)value; }
    else if (k == "ctas_per_sm") { if (value < 1 || value > 8) TEC_FAIL(TEC_ERR_ARG, "ctas_per_sm: 1..8"); ctx->opt_ctas_per_sm = (int)value; }
    else if (k == "bam_lanes") { if (value < 1 || value > 32) TEC_FAIL(TEC_ERR_ARG, "bam_lanes: 1..32"); ctx->opt_bam_lanes = (int)value; }
    else if (k == "bam_window_blocks") { if (value < 1 || value > (1 << 20)) TEC_FAIL(TEC_ERR_ARG, "bam_window_blocks: 1..1048576"); ctx->opt_bam_window_blocks = (int)value; }
    else TEC_FAIL(TEC_ERR_ARG, "tec_set_option: unknown key " + k);
    return TEC_OK;
}

extern "C" const char* tec_index_note(const tec_ctx* ctx) { return ctx ? ctx->idx.stab_why_not.c_str() : ""; }

extern "C" int64_t tec_get_info(tec_ctx* ctx, const char* key) {
    if (!ctx || !key) return -1;
    const std::string k(key);
    if (k == "has_stab") return (ctx->idx.has_stab || ctx->idx.has_stab2) ? 1 : 0;
    if (k == "stab_bytes") return (int64_t)(ctx->idx.has_stab2 ? ctx->idx.stab2_bytes : ctx->idx.stab_bytes);
    if (k == "has_stab2") return ctx->idx.has_stab2 ? 1 : 0;
    if (k == "stab_refused") return ctx->idx.stab_why_not.empty() ? 0 : 1;   // text: tec_index_note()
    if (k == "stab2_sector_bytes") return (ctx->idx.s2_primary + ctx->idx.s2_overflow) * 32;
    if (k == "stab2_edge_cells") return ctx->idx.s2_edge_cells;
    if (k == "stab2_twin_sectors") return ctx->idx.s2_twin_sectors;
    if (k == "last_deferred_units") {      // units the last fast-kernel launch handed to the second pass
        if (!ctx->d_defer_count || !ctx->defer_warps) return 0;
        if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) return -1;
        std::vector<u32> h((size_t)(ctx->last_defer_n > 0 ? ctx->last_defer_n : ctx->defer_warps));   // the segments the last launch used
        if (cudaMemcpy(h.data(), ctx->d_defer_count, h.size() * 4, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
        int64_t n = 0;
        for (u32 x : h) n += x;
        return n;
    }
    if (k == "last_left_units") {          // deferred units bulk2_pair_kernel left for the second pass in the last launch (-1: it did not run)
        if (!ctx->d_part_count || !ctx->last_part_n) return -1;
        if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) return -1;
        std::vector<u32> h((size_t)ctx->last_part_n);
        if (cudaMemcpy(h.data(), ctx->d_part_count, h.size() * 4, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
        int64_t n = 0;
        for (u32 x : h) n += x;
        return n;
    }
    if (k == "has_sc_stab") return ctx->idx.has_sc_stab ? 1 : 0;
    if (k == "sc_stab_bytes") return (int64_t)ctx->idx.sc_stab_bytes;
    if (k == "n_sm") return ctx->n_sm;
    if (k == "sc_last_sort") return ctx->sc_last_sort;
    if (k == "bulk_name_excluded") return ctx->name_pairing && ctx->name ? ctx->name->excluded : 0;
    if (k == "bulk_name_pending_peak") return ctx->name_pairing && ctx->name ? ctx->name->peak : 0;
    if (k == "bulk_name_ms") return ctx->name_pairing && ctx->name ? (int64_t)(ctx->name->ms + 0.5) : 0;
    if (k == "sc_last_sort_passes") return ctx->sc_last_sort_passes;
    if (k == "n_features") return ctx->idx.n_feat;
    if (k == "bulk_counter_words") return ctx->has_index ? (int64_t)ctx->bulk_words() : 0;
    if (k == "last_slow_units") {          // units the last fast-kernel launch handed to the exact kernel
        u32 n = 0;
        if (!ctx->d_slow_list) return 0;
        if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) return -1;
        if (cudaMemcpy(&n, ctx->d_slow_list, 4, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
        return (int64_t)n;
    }
    if (k == "stab_primary") return ctx->idx.has_stab2 ? ctx->idx.s2_primary : ctx->idx.st_primary;
    if (k == "stab_overflow") return ctx->idx.has_stab2 ? ctx->idx.s2_overflow : ctx->idx.st_overflow;
    if (k == "stab_entries") return ctx->idx.has_stab2 ? ctx->idx.s2_entries : ctx->idx.st_entries;
    return -1;
}

// ------------------------------------------------------------------------------------------------
// BAM file -> counting path on the device (bamgpu.cuh)
int BamGpuBackend::deliver(int64_t n, int mode) {
    if (mode == bgzfdev::MODE_PE_NAME || mode == bgzfdev::MODE_PE_NAME_RANGE) {
        const int rc = mode == bgzfdev::MODE_PE_NAME ? name_push_dev(ctx, n, col) : name_hold_dev(ctx, n, col);
        nomem = rc == TEC_ERR_NOMEM;
        return rc ? 1 : 0;
    }
    const int rc = mode == bgzfdev::MODE_SC
                       ? tec_sc_push_dev(ctx, n, col.start, col.end, col.chrom, col.mapq, col.flag, col.cell, col.umi)
                       : tec_bulk_push_dev(ctx, n, col.start, col.end, col.chrom, col.mapq, col.flag);
    return rc ? 1 : 0;
}

// column set b into counter bank b: the bulk kernels run unchanged on d_counts, which points at bank 1 for the second push
int BamGpuBackend::deliver_pairs(int64_t pairs0, int64_t pairs1) {
    for (int s = 0; s < 2; s++) {
        const int64_t n = s ? pairs1 : pairs0;
        if (!n) continue;
        if (s) std::swap(ctx->d_counts, ctx->d_bank1);
        const bgzfdev::Columns& c = pairs.s[s];
        const int rc = bulk_push_dev(ctx, 2 * n, c.start, c.end, c.chrom, c.mapq, c.flag);
        if (s) std::swap(ctx->d_counts, ctx->d_bank1);
        if (rc) return 1;
    }
    return 0;
}

static int bam_status(tec_ctx* ctx, const bamorch::Reader& r, int rc, const BamGpuBackend* be = nullptr) {
    if (rc == bamorch::OK) return TEC_OK;
    if (rc != bamorch::E_BACKEND) ctx->err = r.err;         // the backend left the CUDA text in ctx->err
    switch (rc) {
    case bamorch::E_IO: return TEC_ERR_IO;
    case bamorch::E_FORMAT: return TEC_ERR_FORMAT;
    case bamorch::E_NOT_BGZF: return TEC_ERR_UNSUPPORTED;
    case bamorch::E_UNSUPPORTED: return TEC_ERR_UNSUPPORTED;
    case bamorch::E_ARG: return TEC_ERR_ARG;
    case bamorch::E_BACKEND: return (be && be->nomem) ? TEC_ERR_NOMEM : TEC_ERR_CUDA;
    }
    if (rc <= bamorch::E_RECORD) {
        const int rec = bamorch::E_RECORD - rc;                         // bgzfdev::E_*
        if (rec == bgzfdev::E_FORMAT) return TEC_ERR_FORMAT;            // a malformed record is a format error, not a bad argument
        return -rec;                                                    // TEC_ERR_BAM_*: -10 ... -15
    }
    return TEC_ERR_FORMAT;
}

extern "C" int tec_bam_open(tec_ctx* ctx, const char* path, tec_bam** out) {
    if (!ctx || !path || !out) return TEC_ERR_ARG;
    *out = nullptr;
    tec_bam* b = new tec_bam(ctx);
    const int rc = b->reader.open_path(path);
    if (rc) {
        const int st = bam_status(ctx, b->reader, rc);
        delete b;
        return st;
    }
    *out = b;
    return TEC_OK;
}

extern "C" void tec_bam_close(tec_bam* b) { delete b; }

extern "C" int tec_bam_n_references(const tec_bam* b) { return b ? (int)b->reader.refs.size() : 0; }

extern "C" const char* tec_bam_reference_name(const tec_bam* b, int i) {
    return b && i >= 0 && (size_t)i < b->reader.refs.size() ? b->reader.refs[(size_t)i].c_str() : nullptr;
}

extern "C" int tec_bam_set_chrom_map(tec_bam* b, const uint16_t* bulk_ids, const uint16_t* sc_ids, int32_t n, int32_t n_index) {
    if (!b) return TEC_ERR_ARG;
    b->be.ctx_uploaded = false;
    return bam_status(b->ctx, b->reader, b->reader.set_chrom_map(bulk_ids, sc_ids, n, n_index));
}

extern "C" int tec_bam_set_whitelist(tec_bam* b, const char* barcodes, const int64_t* offsets, int32_t n) {
    if (!b) return TEC_ERR_ARG;
    b->be.ctx_uploaded = false;
    return bam_status(b->ctx, b->reader, b->reader.set_whitelist(barcodes, offsets, n));
}

extern "C" int tec_bam_count(tec_bam* b, int mode, int qual, int64_t* n_records) {
    if (!b) return TEC_ERR_ARG;
    tec_ctx* ctx = b->ctx;
    if (n_records) *n_records = 0;
    if (mode < 0 || mode > 3)
        TEC_FAIL(TEC_ERR_ARG, "tec_bam_count: mode must be 0 (single end), 1 (paired end), 2 (single cell) or 3 (paired end by read name)");
    if (mode == bgzfdev::MODE_SC) {
        if (!ctx->sc || !ctx->sc->active) TEC_FAIL(TEC_ERR_STATE, "tec_bam_count: tec_sc_begin not called");
    } else if (!ctx->bulk_active || (ctx->name_pairing ? 3 : ctx->paired ? 1 : 0) != mode) {
        TEC_FAIL(TEC_ERR_STATE, "tec_bam_count: tec_bulk_begin not called for this mode");
    } else if (int st = bulk_ready(ctx, "tec_bam_count")) {
        return st;
    }
    TEC_CUDA(cudaSetDevice(ctx->device));
    int64_t n = 0;
    const int rc = bamorch::decode_all(b->reader, b->be, mode, qual, ctx->opt_bam_window_blocks, &n);
    if (n_records) *n_records = n;
    return bam_status(ctx, b->reader, rc, &b->be);
}

extern "C" int tec_bam_count_range(tec_bam* b, int mode, int qual, int64_t byte_lo, int64_t byte_hi, int64_t* out) {
    if (!b) return TEC_ERR_ARG;
    tec_ctx* ctx = b->ctx;
    if (!out) TEC_FAIL(TEC_ERR_ARG, "tec_bam_count_range: out must hold TEC_BAM_RANGE_WORDS values");
    for (int i = 0; i < TEC_BAM_RANGE_WORDS; i++) out[i] = 0;
    if (mode < 0 || mode > 4 || mode == bgzfdev::MODE_PE_NAME)
        TEC_FAIL(TEC_ERR_ARG, "tec_bam_count_range: mode must be 0 (single end), 1 (paired end), 2 (single cell) or 4 (paired end by read "
                              "name, rows held for the exchange)");
    if (byte_lo < 0 || byte_hi < byte_lo) TEC_FAIL(TEC_ERR_ARG, "tec_bam_count_range: bad byte range");
    if (mode == bgzfdev::MODE_SC) {
        if (!ctx->sc || !ctx->sc->active) TEC_FAIL(TEC_ERR_STATE, "tec_bam_count_range: tec_sc_begin not called");
    } else if (mode == bgzfdev::MODE_PE_NAME_RANGE) {
        if (!ctx->bulk_active || !ctx->name_pairing) TEC_FAIL(TEC_ERR_STATE, "tec_bam_count_range: mode 4 needs tec_bulk_begin(ctx, 2, qual)");
        if (ctx->name->pending && !ctx->name_held)
            TEC_FAIL(TEC_ERR_STATE, "tec_bam_count_range: mode 4 after records were pushed into this run");
    } else if (!ctx->bulk_active || (ctx->paired ? 1 : 0) != mode || ctx->name_pairing) {
        TEC_FAIL(TEC_ERR_STATE, "tec_bam_count_range: tec_bulk_begin not called for this mode");
    } else if (int st = bulk_ready(ctx, "tec_bam_count_range")) {
        return st;
    }
    TEC_CUDA(cudaSetDevice(ctx->device));
    b->edge[0].clear();
    b->edge[1].clear();
    if (mode == bgzfdev::MODE_PE) {
        // bank 1 starts as a copy of the running count; bank 0 is the running count itself
        const size_t bytes = ctx->bulk_words() * 8;
        if (ctx->bank1_cap < (int64_t)ctx->bulk_words()) {
            TEC_CUDA(cudaStreamSynchronize(ctx->stream));
            cudaFree(ctx->d_bank1);
            ctx->d_bank1 = nullptr;
            ctx->bank1_cap = 0;
            TEC_CUDA(cudaMalloc(&ctx->d_bank1, bytes));
            ctx->bank1_cap = (int64_t)ctx->bulk_words();
        }
        TEC_CUDA(cudaMemcpyAsync(ctx->d_bank1, ctx->d_counts, bytes, cudaMemcpyDeviceToDevice, ctx->stream));
        ctx->bank_pending = true;
    }
    if (mode == bgzfdev::MODE_PE_NAME_RANGE) ctx->name_held = true;
    bamorch::RangeResult r;
    const int rc = bamorch::decode_range(b->reader, b->be, mode, qual, ctx->opt_bam_window_blocks, (uint64_t)byte_lo, (uint64_t)byte_hi, &r);
    out[0] = r.n_records; out[1] = r.start_block; out[2] = r.start_off; out[3] = r.exit_block; out[4] = r.exit_off;
    out[5] = (int64_t)b->reader.file.size;
    b->edge[0].swap(r.first_rec);
    b->edge[1].swap(r.last_rec);
    return bam_status(ctx, b->reader, rc, &b->be);
}

extern "C" int tec_bam_range_record(const tec_bam* b, int which, void* buf, int64_t cap, int64_t* len) {
    if (!b || !len || (which != 0 && which != 1)) return TEC_ERR_ARG;
    const std::vector<uint8_t>& e = b->edge[which];
    *len = (int64_t)e.size();
    if (!buf) return TEC_OK;
    if (cap < *len) {
        b->ctx->err = "tec_bam_range_record: the buffer is smaller than the record";
        return TEC_ERR_ARG;
    }
    if (!e.empty()) memcpy(buf, e.data(), e.size());
    return TEC_OK;
}

extern "C" int tec_bam_pair_columns(tec_bam* b, const void* rec1, int64_t n1, const void* rec2, int64_t n2, int qual,
                                    int32_t* start, int32_t* end, uint16_t* chrom, uint8_t* mapq, uint8_t* flag) {
    if (!b || !rec1 || !rec2 || !start || !end || !chrom || !mapq || !flag) return TEC_ERR_ARG;
    tec_ctx* ctx = b->ctx;
    const int rc = bamorch::parse_pair(b->reader, (const uint8_t*)rec1, n1, (const uint8_t*)rec2, n2, qual, start, end, chrom, mapq, flag);
    return bam_status(ctx, b->reader, rc);
}

extern "C" int64_t tec_bam_info(const tec_bam* b, int what) {
    if (!b) return 0;
    switch (what) {
    case 0: return b->be.n_declined;
    case 1: return (int64_t)(b->be.ms_load * 1e3);
    case 2: return (int64_t)(b->be.ms_inflate * 1e3);
    case 3: return (int64_t)(b->be.ms_chain * 1e3);
    case 4: return (int64_t)(b->be.ms_parse * 1e3);
    }
    return 0;
}

