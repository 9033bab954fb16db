// BAM file -> counting path without the host cores in the middle (SURVEY.md 8f-1, device side).
//
// The compressed BGZF blocks of a window (tens of thousands of blocks) go to the device as they
// are in the file; three passes with ONE THREAD PER BGZF BLOCK do the rest (routines in bgzf_dev.h,
// window loop and exact chain check in bam_orch.h, both also run on the CPU by the tests):
//   bam_inflate_kernel   raw DEFLATE + CRC32 of every block into one contiguous window in HBM
//   bam_chain_kernel     first record start per block (guess) + hop to the end of the block
//   bam_list_kernel      record offsets of the window in file order (thread per block, one load per record)
//   bam_parse_kernel     one thread per record: fields into the SoA columns tec_*_push_dev takes
// A block is independent work with a long serial dependency chain (Huffman decoding), so the
// parallelism is across blocks: the window is sized so that every SM has a few hundred of them
// in flight and the latency of one chain hides behind the others.  Decode tables live in a
// per-block scratch slice in global memory (2.9 KB, L2-resident for the blocks in flight).
// Blocks the inflate refuses are inflated by zlib on the host and patched in; record layouts the
// chain check refuses make the whole call return TEC_ERR_UNSUPPORTED (use libtecbam).
#pragma once
#include "bam_orch.h"
#include "context.cuh"

#include <thread>

#define BAM_TPB 64
#define TEC_BAM_CHUNK (size_t(128) << 20)

__global__ void bam_inflate_kernel(int nb, const bamorch::BlockDesc* __restrict__ bl, const uint8_t* __restrict__ comp, uint8_t* __restrict__ ubuf,
                                   uint8_t* __restrict__ scratch, const uint32_t* __restrict__ crc_table, const uint32_t* __restrict__ crc_mats,
                                   int32_t* __restrict__ status, int lanes) {
    // `lanes` streams per warp: 32 independent Huffman streams in one warp diverge on every symbol, fewer
    // streams per warp trade idle lanes for less serialisation (option bam_lanes)
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (lanes == 1) {
        // one block per warp: lane 0 decodes, then all 32 lanes share the CRC32 of the inflated bytes
        if (warp >= nb) return;
        const bamorch::BlockDesc d = bl[warp];
        uint8_t* out = ubuf + d.out_off;
        int st = 0;
        // the decode tables of the warp's block live in shared memory (2.9 KB per warp): a lookup per symbol
        extern __shared__ __align__(16) uint8_t bam_smem[];
        if (lane == 0) st = bgzfdev::inflate_block(comp + d.in_off, d.in_len, out, d.out_len, bam_smem + (threadIdx.x >> 5) * bgzfdev::SCRATCH_STRIDE);
        __syncwarp();                                   // lane 0's stores are visible to the warp
        st = __shfl_sync(0xFFFFFFFFu, st, 0);
        if (st == bgzfdev::ST_OK) {
            uint32_t c = bgzfdev::crc32_lane_share(out, d.out_len, lane, crc_table, crc_mats);
            for (int o = 16; o; o >>= 1) c ^= __shfl_xor_sync(0xFFFFFFFFu, c, o);
            if ((c ^ 0xFFFFFFFFu) != d.crc) st = bgzfdev::ST_CRC;
        }
        if (lane == 0) status[warp] = st;
        return;
    }
    if (lane >= lanes) return;
    const int b = (int)(warp * lanes + lane);
    if (b >= nb) return;
    const bamorch::BlockDesc d = bl[b];
    uint8_t* out = ubuf + d.out_off;
    int st = bgzfdev::inflate_block(comp + d.in_off, d.in_len, out, d.out_len, scratch + (size_t)b * bgzfdev::SCRATCH_STRIDE);
    if (st == bgzfdev::ST_OK && bgzfdev::crc32_block(out, d.out_len, crc_table) != d.crc) st = bgzfdev::ST_CRC;
    status[b] = st;
}

__global__ void bam_chain_kernel(int nb, const bamorch::BlockDesc* __restrict__ bl, const uint8_t* __restrict__ ubuf, int64_t w_end, int32_t n_ref,
                                 bamorch::BlockChain* __restrict__ out) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nb) return;
    const int64_t lo = (int64_t)bl[b].out_off, hi = lo + bl[b].out_len;
    const int64_t s = b == 0 ? 0 : bgzfdev::find_start(ubuf, lo, hi, w_end, n_ref);
    bamorch::BlockChain c;
    c.start = s; c.exit = s; c.last = bgzfdev::NO_START; c.count = 0; c.bad = 0;
    if (s != bgzfdev::NO_START) {
        const bgzfdev::Hop h = bgzfdev::hop(ubuf, s, hi, w_end);
        c.exit = h.exit; c.last = h.last; c.count = h.count; c.bad = h.bad;
    }
    out[b] = c;
}

// record offsets of the used blocks, in file order: thread per block hops once more (one load per record)
__global__ void bam_list_kernel(int nb, const bamorch::BlockChain* __restrict__ ch, const int64_t* __restrict__ base, const uint8_t* __restrict__ ubuf,
                                int64_t* __restrict__ rec_off) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nb) return;
    const uint32_t n = ch[b].count;
    int64_t p = ch[b].start;
    const int64_t k0 = base[b];
    for (uint32_t i = 0; i < n; i++) {
        rec_off[k0 + i] = p;
        p += 4 + (int64_t)bgzfdev::ld32(ubuf + p);
    }
}

// one thread per record (per pair in paired-end mode: the first mate's thread writes both rows)
__global__ void bam_parse_kernel(int64_t n_rec, const int64_t* __restrict__ rec_off, const uint8_t* __restrict__ ubuf, int mode, bgzfdev::ParseCtx pc,
                                 bgzfdev::Columns o, unsigned long long* __restrict__ first_err) {
    const int64_t step = mode == bgzfdev::MODE_PE ? 2 : 1;
    for (int64_t k = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * step; k < n_rec; k += (int64_t)gridDim.x * blockDim.x * step) {
        const int64_t p = rec_off[k], p2 = step == 2 ? rec_off[k + 1] : 0;
        const int e = bgzfdev::parse_record(ubuf, p, p2, mode, pc, o, k);
        if (e) atomicMin(first_err, ((unsigned long long)k << 8) | (unsigned long long)e);
    }
}

struct PairSets {
    bgzfdev::Columns s[2];
};

// paired-end byte range: one thread per ADJACENT pair i (records i, i + 1 of the window), written into the column set of
// the parity of its range-local index g0 + i (bgzfdev::parse_adjacent_pair); every record is parsed once as read1 and
// once as read2, in the two sets
__global__ void bam_parse_pairs_kernel(int64_t n_pairs, const int64_t* __restrict__ rec_off, const uint8_t* __restrict__ ubuf, int64_t g0,
                                       bgzfdev::ParseCtx pc, PairSets sets, unsigned long long* __restrict__ first_err) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_pairs; i += (int64_t)gridDim.x * blockDim.x) {
        const int e = bgzfdev::parse_adjacent_pair(ubuf, rec_off, i, g0, pc, sets.s);
        if (e) atomicMin(first_err, ((unsigned long long)i << 8) | (unsigned long long)e);
    }
}

struct BamGpuBackend {
    tec_ctx* ctx;
    uint8_t *d_comp = nullptr, *d_ubuf = nullptr, *d_scratch = nullptr, *d_tmp = nullptr;
    size_t comp_cap = 0, ubuf_cap = 0, tmp_cap = 0;
    int blocks_cap = 0;
    bamorch::BlockDesc* d_blocks = nullptr;
    bamorch::BlockChain* d_chain = nullptr;
    int64_t* d_base = nullptr;
    int64_t* d_rec_off = nullptr;
    int32_t* d_status = nullptr;
    uint32_t* d_crc = nullptr;             // 256-entry table, then the shift operators of bgzfdev::crc32_shift
    unsigned long long* d_err = nullptr;
    uint16_t *d_bulk_ids = nullptr, *d_sc_ids = nullptr;
    uint32_t* d_wl_slot = nullptr;
    int64_t* d_wl_off = nullptr;
    uint8_t* d_wl_bytes = nullptr;
    bool ctx_uploaded = false;
    bgzfdev::Columns col{nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    int64_t col_cap = 0, name_col_cap = 0;      // name_col_cap: rows of the MODE_PE_NAME columns (key, role)
    PairSets pairs{};                      // paired-end ranges: the two column sets (separate allocations: aligned for bulk2)
    int64_t* d_pair_off = nullptr;
    int64_t pairs_cap = 0;
    int64_t n_declined = 0;
    double ms_load = 0, ms_inflate = 0, ms_chain = 0, ms_parse = 0;

    explicit BamGpuBackend(tec_ctx* c) : ctx(c) {}
    ~BamGpuBackend() {
        cudaSetDevice(ctx->device);
        cudaStreamSynchronize(ctx->stream);
        void* blocks[] = {d_comp, d_ubuf, d_scratch, d_tmp, d_blocks, d_chain, d_base, d_status, d_crc, d_err, d_bulk_ids, d_sc_ids, d_wl_slot,
                          d_wl_off, d_wl_bytes, d_rec_off, col.start, col.end, col.chrom, col.mapq, col.flag, col.cell, col.umi, d_pair_off,
                          pairs.s[0].start, pairs.s[0].end, pairs.s[0].chrom, pairs.s[0].mapq, pairs.s[0].flag,
                          pairs.s[1].start, pairs.s[1].end, pairs.s[1].chrom, pairs.s[1].mapq, pairs.s[1].flag,
                          col.key_hi, col.key_lo, col.role};
        for (void* p : blocks) ctx->cache.put(p);            // back to the context's block cache: the next file reuses them
    }
    template <class T> cudaError_t dev_alloc(T** out, size_t bytes) {
        void* p = nullptr;
        const cudaError_t e = ctx->cache.get(&p, bytes);
        *out = (T*)p;
        return e;
    }
    template <class T> void dev_free(T*& p) {
        ctx->cache.put(p);
        p = nullptr;
    }
    static double now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
    bool nomem = false;                  // the last failure was an allocation failure (-> TEC_ERR_NOMEM)
    bool ok(cudaError_t e, const char* what) {
        if (e == cudaSuccess) return true;
        ctx->err = std::string(what) + ": " + cudaGetErrorString(e);
        nomem = e == cudaErrorMemoryAllocation;
        if (nomem) cudaGetLastError();   // not sticky: clear it, the caller may go on with the host decoder
        return false;
    }
#define BAM_CK(call) do { if (!ok((call), #call)) return 1; } while (0)

    int init() {
        if (d_crc) return 0;
        uint32_t t[256 + bgzfdev::CRC_SHIFT_MATS * 32];
        bamorch::crc32_tables(t, t + 256);
        BAM_CK(cudaSetDevice(ctx->device));
        BAM_CK(dev_alloc(&d_crc, sizeof(t)));
        BAM_CK(cudaMemcpy(d_crc, t, sizeof(t), cudaMemcpyHostToDevice));
        BAM_CK(dev_alloc(&d_err, 8));
        for (int i = 0; i < 2; i++)
            if (!ctx->bam_pinned[i]) BAM_CK(cudaHostAlloc(&ctx->bam_pinned[i], TEC_BAM_CHUNK, cudaHostAllocDefault));
        if (!ctx->bam_ev[0]) {
            for (int i = 0; i < 3; i++) BAM_CK(cudaEventCreateWithFlags(&ctx->bam_ev[i], cudaEventDisableTiming));
            BAM_CK(cudaStreamCreateWithFlags(&ctx->bam_stream2, cudaStreamNonBlocking));
        }
        return 0;
    }
    int reserve(size_t comp_bytes, size_t ubuf_bytes, int nb) {
        if (init()) return 1;
        if (comp_bytes > comp_cap) {
            BAM_CK(cudaStreamSynchronize(ctx->stream));
            dev_free(d_comp);
            comp_cap = 0;
            const size_t cap = comp_bytes + (comp_bytes >> 3) + 4096;
            BAM_CK(dev_alloc(&d_comp, cap));
            comp_cap = cap;
        }
        if (ubuf_bytes > ubuf_cap) {
            const size_t cap = ubuf_bytes + (ubuf_bytes >> 3) + 4096;
            uint8_t* q = nullptr;
            BAM_CK(dev_alloc(&q, cap));
            if (d_ubuf) {
                BAM_CK(cudaMemcpyAsync(q, d_ubuf, ubuf_cap, cudaMemcpyDeviceToDevice, ctx->stream));
                BAM_CK(cudaStreamSynchronize(ctx->stream));
                dev_free(d_ubuf);
            }
            d_ubuf = q;
            ubuf_cap = cap;
        }
        if (nb > blocks_cap) {
            BAM_CK(cudaStreamSynchronize(ctx->stream));
            dev_free(d_blocks); dev_free(d_chain); dev_free(d_base); dev_free(d_status); dev_free(d_scratch);
            blocks_cap = 0;
            const int cap = nb + (nb >> 3) + 64;
            BAM_CK(dev_alloc(&d_blocks, sizeof(bamorch::BlockDesc) * (size_t)cap));
            BAM_CK(dev_alloc(&d_chain, sizeof(bamorch::BlockChain) * (size_t)cap));
            BAM_CK(dev_alloc(&d_base, 8 * (size_t)cap));
            BAM_CK(dev_alloc(&d_status, 4 * (size_t)cap));
            BAM_CK(dev_alloc(&d_scratch, (size_t)bgzfdev::SCRATCH_STRIDE * (size_t)cap));
            blocks_cap = cap;
        }
        return 0;
    }
    const bamorch::MappedFile* cur_file = nullptr;
    size_t cur_lo = 0, cur_n = 0;
    int load(const bamorch::MappedFile& f, size_t lo, size_t n) {       // the bytes move inside inflate(), chunk by chunk
        cur_file = &f;
        cur_lo = lo;
        cur_n = n;
        return 0;
    }
    int read_chunk(uint8_t* buf, size_t off, size_t len) {
        const int nt = (int)std::max<size_t>(1, std::min<size_t>(8, len >> 22));
        std::vector<std::thread> th;
        std::vector<int> bad((size_t)nt, 0);
        const int fd = cur_file->fd;
        const size_t lo = cur_lo;
        for (int t = 0; t < nt; t++)
            th.emplace_back([&, t] {
                size_t a = len * (size_t)t / (size_t)nt, b = len * (size_t)(t + 1) / (size_t)nt;
                while (a < b) {
                    const ssize_t k = pread(fd, buf + a, b - a, (off_t)(lo + off + a));
                    if (k <= 0) { bad[(size_t)t] = 1; return; }
                    a += (size_t)k;
                }
            });
        for (auto& x : th) x.join();
        for (int x : bad)
            if (x) { ctx->err = "pread failed"; return 1; }
        return 0;
    }
    int put(int64_t at, const uint8_t* data, size_t n) {
        BAM_CK(cudaMemcpyAsync(d_ubuf + at, data, n, cudaMemcpyHostToDevice, ctx->stream));
        BAM_CK(cudaStreamSynchronize(ctx->stream));          // `data` is the caller's pageable memory
        return 0;
    }
    int carry(int64_t from, int64_t n) {
        if (from >= n) {
            BAM_CK(cudaMemcpyAsync(d_ubuf, d_ubuf + from, (size_t)n, cudaMemcpyDeviceToDevice, ctx->stream));
            return 0;
        }
        if ((size_t)n > tmp_cap) {
            BAM_CK(cudaStreamSynchronize(ctx->stream));
            dev_free(d_tmp);
            tmp_cap = 0;
            BAM_CK(dev_alloc(&d_tmp, (size_t)n + 4096));
            tmp_cap = (size_t)n + 4096;
        }
        BAM_CK(cudaMemcpyAsync(d_tmp, d_ubuf + from, (size_t)n, cudaMemcpyDeviceToDevice, ctx->stream));
        BAM_CK(cudaMemcpyAsync(d_ubuf, d_tmp, (size_t)n, cudaMemcpyDeviceToDevice, ctx->stream));
        return 0;
    }
    // page cache -> two pinned chunks (a few pread streams each: one tops out near 5 GB/s) -> HBM -> inflate
    // kernel over the blocks of the chunk.  Chunks alternate between two streams, so the host reads
    // chunk i+1 while chunk i is copied and chunk i-1 is being inflated.
    int inflate(const bamorch::BlockDesc* bl, int nb, int32_t* status) {
        const double t0 = now_ms();
        cudaStream_t st[2] = {ctx->stream, ctx->bam_stream2};
        BAM_CK(cudaMemcpyAsync(d_blocks, bl, sizeof(bamorch::BlockDesc) * (size_t)nb, cudaMemcpyHostToDevice, ctx->stream));
        BAM_CK(cudaMemsetAsync(d_status, 0xFF, 4 * (size_t)nb, ctx->stream));      // a block no kernel reports on counts as declined
        BAM_CK(cudaEventRecord(ctx->bam_ev[2], ctx->stream));
        BAM_CK(cudaStreamWaitEvent(ctx->bam_stream2, ctx->bam_ev[2], 0));       // descriptors (and the window so far) are in place
        const int lanes = ctx->opt_bam_lanes;
        int b0 = 0, i = 0;
        while (b0 < nb) {
            // blocks [b0, b1): compressed bytes [c_lo, c_hi) of the window, at most one chunk
            const size_t c_lo = b0 ? (size_t)bl[b0].in_off : 0;
            int b1 = b0;
            while (b1 < nb && (size_t)bl[b1].in_off + bl[b1].in_len + 8 - c_lo <= TEC_BAM_CHUNK) b1++;
            if (b1 == b0) { ctx->err = "BGZF block larger than the staging chunk"; return 1; }
            const size_t c_hi = std::min<size_t>(cur_n, (size_t)bl[b1 - 1].in_off + bl[b1 - 1].in_len + 8);   // through the last trailer
            uint8_t* buf = ctx->bam_pinned[i];
            BAM_CK(cudaEventSynchronize(ctx->bam_ev[i]));                       // the copy that last used this chunk is done
            if (read_chunk(buf, c_lo, c_hi - c_lo)) return 1;
            BAM_CK(cudaMemcpyAsync(d_comp + c_lo, buf, c_hi - c_lo, cudaMemcpyHostToDevice, st[i]));
            BAM_CK(cudaEventRecord(ctx->bam_ev[i], st[i]));
            const int n = b1 - b0;
            const int64_t warps = (n + lanes - 1) / lanes;
            const size_t smem = lanes == 1 ? (size_t)(BAM_TPB / 32) * bgzfdev::SCRATCH_STRIDE : 0;
            bam_inflate_kernel<<<(unsigned)((warps * 32 + BAM_TPB - 1) / BAM_TPB), BAM_TPB, smem, st[i]>>>(
                n, d_blocks + b0, d_comp, d_ubuf, d_scratch + (size_t)b0 * bgzfdev::SCRATCH_STRIDE, d_crc, d_crc + 256, d_status + b0, lanes);
            BAM_CK(cudaGetLastError());
            ctx->launches++;
            b0 = b1;
            i ^= 1;
        }
        BAM_CK(cudaEventRecord(ctx->bam_ev[2], ctx->bam_stream2));
        BAM_CK(cudaStreamWaitEvent(ctx->stream, ctx->bam_ev[2], 0));
        BAM_CK(cudaMemcpyAsync(status, d_status, 4 * (size_t)nb, cudaMemcpyDeviceToHost, ctx->stream));
        BAM_CK(cudaStreamSynchronize(ctx->stream));
        for (int k = 0; k < nb; k++) n_declined += status[k] != 0;
        ms_inflate += now_ms() - t0;
        return 0;
    }
    int chain(const bamorch::BlockDesc* bl, int nb, int64_t w_end, int32_t n_ref, bamorch::BlockChain* out) {
        const double t0 = now_ms();
        BAM_CK(cudaMemcpyAsync(d_blocks, bl, sizeof(bamorch::BlockDesc) * (size_t)nb, cudaMemcpyHostToDevice, ctx->stream));
        bam_chain_kernel<<<(nb + BAM_TPB - 1) / BAM_TPB, BAM_TPB, 0, ctx->stream>>>(nb, d_blocks, d_ubuf, w_end, n_ref, d_chain);
        BAM_CK(cudaGetLastError());
        BAM_CK(cudaMemcpyAsync(out, d_chain, sizeof(bamorch::BlockChain) * (size_t)nb, cudaMemcpyDeviceToHost, ctx->stream));
        BAM_CK(cudaStreamSynchronize(ctx->stream));
        ctx->launches++;
        ms_chain += now_ms() - t0;
        return 0;
    }
    template <class T> int up(T** dst, const void* src, size_t n) {
        dev_free(*dst);
        BAM_CK(dev_alloc(dst, n ? n : 1));
        if (n) BAM_CK(cudaMemcpy(*dst, src, n, cudaMemcpyHostToDevice));
        return 0;
    }
    int upload_maps(const bamorch::Reader& r) {
        if (!ctx_uploaded) {
            if (up(&d_bulk_ids, r.bulk_ids.data(), r.bulk_ids.size() * 2) || up(&d_sc_ids, r.sc_ids.data(), r.sc_ids.size() * 2) ||
                up(&d_wl_slot, r.wl_slot.data(), r.wl_slot.size() * 4) || up(&d_wl_off, r.wl_off.data(), r.wl_off.size() * 8) ||
                up(&d_wl_bytes, r.wl_bytes.data(), r.wl_bytes.size()))
                return 1;
            ctx_uploaded = true;
        }
        return 0;
    }
    int parse(const bamorch::BlockDesc*, int nb, const bamorch::BlockChain* ch, const int64_t* base, int64_t n, int64_t, int mode, int qual,
              const bamorch::Reader& r, int* err, int64_t* err_rec) {
        const double t0 = now_ms();
        if (upload_maps(r)) return 1;
        if (n > col_cap) {
            BAM_CK(cudaStreamSynchronize(ctx->stream));
            dev_free(col.start); dev_free(col.end); dev_free(col.chrom); dev_free(col.mapq); dev_free(col.flag); dev_free(col.cell); dev_free(col.umi);
            dev_free(d_rec_off);
            col_cap = 0;
            const size_t cap = (size_t)n + ((size_t)n >> 3) + 1024;
            BAM_CK(dev_alloc(&col.start, cap * 4)); BAM_CK(dev_alloc(&col.end, cap * 4)); BAM_CK(dev_alloc(&col.chrom, cap * 2));
            BAM_CK(dev_alloc(&col.mapq, cap)); BAM_CK(dev_alloc(&col.flag, cap)); BAM_CK(dev_alloc(&col.cell, cap * 4));
            BAM_CK(dev_alloc(&col.umi, cap * 8));
            BAM_CK(dev_alloc(&d_rec_off, cap * 8));
            col_cap = (int64_t)cap;
        }
        if (mode == bgzfdev::MODE_PE_NAME && name_col_cap < col_cap) {
            BAM_CK(cudaStreamSynchronize(ctx->stream));
            dev_free(col.key_hi); dev_free(col.key_lo); dev_free(col.role);
            name_col_cap = 0;
            BAM_CK(dev_alloc(&col.key_hi, (size_t)col_cap * 8)); BAM_CK(dev_alloc(&col.key_lo, (size_t)col_cap * 8));
            BAM_CK(dev_alloc(&col.role, (size_t)col_cap));
            name_col_cap = col_cap;
        }
        bgzfdev::ParseCtx pc;
        pc.bulk_ids = d_bulk_ids; pc.sc_ids = d_sc_ids; pc.n_ref = (int32_t)r.refs.size(); pc.n_index = r.n_index; pc.qual = qual;
        pc.wl.slot = d_wl_slot; pc.wl.off = d_wl_off; pc.wl.bytes = d_wl_bytes; pc.wl.mask = r.wl_slot.empty() ? 0 : r.wl_slot.size() - 1;
        BAM_CK(cudaMemcpyAsync(d_chain, ch, sizeof(bamorch::BlockChain) * (size_t)nb, cudaMemcpyHostToDevice, ctx->stream));
        BAM_CK(cudaMemcpyAsync(d_base, base, 8 * (size_t)nb, cudaMemcpyHostToDevice, ctx->stream));
        BAM_CK(cudaMemsetAsync(d_err, 0xFF, 8, ctx->stream));
        const bool trace = getenv("TEC_BAM_TIMING") != nullptr;
        double t1 = 0, t2 = 0;
        if (trace) { BAM_CK(cudaStreamSynchronize(ctx->stream)); t1 = now_ms(); }
        bam_list_kernel<<<(nb + BAM_TPB - 1) / BAM_TPB, BAM_TPB, 0, ctx->stream>>>(nb, d_chain, d_base, d_ubuf, d_rec_off);
        BAM_CK(cudaGetLastError());
        if (trace) { BAM_CK(cudaStreamSynchronize(ctx->stream)); t2 = now_ms(); }
        const int64_t units = mode == bgzfdev::MODE_PE ? n / 2 : n;
        const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((units + 127) / 128, (int64_t)ctx->n_sm * 64));
        bam_parse_kernel<<<grid, 128, 0, ctx->stream>>>(n, d_rec_off, d_ubuf, mode, pc, col, d_err);
        BAM_CK(cudaGetLastError());
        unsigned long long e = 0;
        BAM_CK(cudaMemcpyAsync(&e, d_err, 8, cudaMemcpyDeviceToHost, ctx->stream));
        BAM_CK(cudaStreamSynchronize(ctx->stream));
        *err = 0;
        if (e != ~0ull) {
            *err = (int)(e & 0xFF);
            *err_rec = (int64_t)(e >> 8);
        }
        ctx->launches += 2;
        if (trace) fprintf(stderr, "[tec_bam] parse: setup %.2f ms, list %.2f ms, parse %.2f ms (%lld records, %d blocks)\n", t1 - t0, t2 - t1,
                           now_ms() - t2, (long long)n, nb);
        ms_parse += now_ms() - t0;
        return 0;
    }
    int parse_pairs(const bamorch::BlockChain* ch, const int64_t* base, int nb, int64_t n, int64_t g0, int qual, const bamorch::Reader& r,
                    int* err, int64_t* err_rec) {
        const double t0 = now_ms();
        if (upload_maps(r)) return 1;
        if (n > pairs_cap) {               // each set holds at most n rows (n - 1 pairs, every other one)
            BAM_CK(cudaStreamSynchronize(ctx->stream));
            for (bgzfdev::Columns& s : pairs.s) { dev_free(s.start); dev_free(s.end); dev_free(s.chrom); dev_free(s.mapq); dev_free(s.flag); }
            dev_free(d_pair_off);
            pairs_cap = 0;
            const size_t cap = (size_t)n + ((size_t)n >> 3) + 1024;
            for (bgzfdev::Columns& s : pairs.s) {
                BAM_CK(dev_alloc(&s.start, cap * 4)); BAM_CK(dev_alloc(&s.end, cap * 4)); BAM_CK(dev_alloc(&s.chrom, cap * 2));
                BAM_CK(dev_alloc(&s.mapq, cap)); BAM_CK(dev_alloc(&s.flag, cap));
            }
            BAM_CK(dev_alloc(&d_pair_off, cap * 8));
            pairs_cap = (int64_t)cap;
        }
        bgzfdev::ParseCtx pc;
        pc.bulk_ids = d_bulk_ids; pc.sc_ids = d_sc_ids; pc.n_ref = (int32_t)r.refs.size(); pc.n_index = r.n_index; pc.qual = qual;
        pc.wl.slot = d_wl_slot; pc.wl.off = d_wl_off; pc.wl.bytes = d_wl_bytes; pc.wl.mask = r.wl_slot.empty() ? 0 : r.wl_slot.size() - 1;
        BAM_CK(cudaMemcpyAsync(d_chain, ch, sizeof(bamorch::BlockChain) * (size_t)nb, cudaMemcpyHostToDevice, ctx->stream));
        BAM_CK(cudaMemcpyAsync(d_base, base, 8 * (size_t)nb, cudaMemcpyHostToDevice, ctx->stream));
        BAM_CK(cudaMemsetAsync(d_err, 0xFF, 8, ctx->stream));
        bam_list_kernel<<<(nb + BAM_TPB - 1) / BAM_TPB, BAM_TPB, 0, ctx->stream>>>(nb, d_chain, d_base, d_ubuf, d_pair_off);
        BAM_CK(cudaGetLastError());
        const int64_t n_pairs = n - 1;
        const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((n_pairs + 127) / 128, (int64_t)ctx->n_sm * 64));
        bam_parse_pairs_kernel<<<grid, 128, 0, ctx->stream>>>(n_pairs, d_pair_off, d_ubuf, g0, pc, pairs, d_err);
        BAM_CK(cudaGetLastError());
        unsigned long long e = 0;
        BAM_CK(cudaMemcpyAsync(&e, d_err, 8, cudaMemcpyDeviceToHost, ctx->stream));
        BAM_CK(cudaStreamSynchronize(ctx->stream));
        *err = 0;
        if (e != ~0ull) {
            *err = (int)(e & 0xFF);
            *err_rec = (int64_t)(e >> 8);
        }
        ctx->launches += 2;
        ms_parse += now_ms() - t0;
        return 0;
    }
    int fetch(int64_t at, uint8_t* dst, size_t n) {
        BAM_CK(cudaMemcpyAsync(dst, d_ubuf + at, n, cudaMemcpyDeviceToHost, ctx->stream));
        BAM_CK(cudaStreamSynchronize(ctx->stream));
        return 0;
    }
    int deliver(int64_t n, int mode);
    int deliver_pairs(int64_t pairs0, int64_t pairs1);
};

struct tec_bam {
    tec_ctx* ctx;
    bamorch::Reader reader;
    BamGpuBackend be;
    std::vector<uint8_t> edge[2];          // first / last record of the last paired-end range (tec_bam_range_record)
    explicit tec_bam(tec_ctx* c) : ctx(c), be(c) {}
};
