// Context object behind the opaque tec_ctx handle.
#pragma once
#include "common.cuh"
#include "bulk.cuh"
#include "bulk2.cuh"
#include <map>

#define TEC_STAGE_RECORDS (int64_t(16) << 20)     // records per host->device staging chunk

struct DevIndex {
    int32_t* L = nullptr;
    int32_t* R = nullptr;
    int32_t* pmaxR = nullptr;
    u32* info = nullptr;
    int64_t* chrom_off = nullptr;
    u32* dir = nullptr;
    int64_t* dir_off = nullptr;
    uint8_t* chrom_valid = nullptr;
    int n_chrom = 0, n_ensg = 0, bs = 10000, shift = 9;
    int64_t n_feat = 0, n_dir = 0;
    // cell table (stab_build.h); absent when the index exceeds its limits
    u32* st_sectors = nullptr;
    uint2* st_cells = nullptr;            // per chromosome {first sector, number of cells}
    uint8_t* st_slot_type = nullptr;
    u32* st_ovf_base = nullptr;
    int st_shift = 11, st_all_counted = 1;
    bool has_stab = false;
    size_t stab_bytes = 0;
    int64_t st_primary = 0, st_overflow = 0, st_entries = 0;
    StabView stab_view() const {
        StabView v;
        v.sectors = st_sectors; v.cells = st_cells; v.slot_type = st_slot_type; v.ovf_base = st_ovf_base;
        v.shift = st_shift; v.all_counted = st_all_counted;
        return v;
    }
    // cell table, layout 2 (stab2_build.h): the default bulk path (bulk2.cuh)
    u32* s2_sectors = nullptr;
    uint2* s2_cells = nullptr;
    u32* s2_ovf_first = nullptr;
    uint8_t* s2_slot_type = nullptr;
    int s2_shift = 10, s2_ext = STAB_EXT, s2_all_counted = 1;
    bool has_stab2 = false;
    size_t stab2_bytes = 0;
    int64_t s2_primary = 0, s2_overflow = 0, s2_entries = 0, s2_edge_cells = 0, s2_twin_sectors = 0;
    std::string stab_why_not;             // why no cell table could be built (the exact search kernel is used then)
    Stab2View stab2_view() const {
        Stab2View v;
        v.sectors = s2_sectors; v.cells = s2_cells; v.ovf_first = s2_ovf_first; v.slot_type = s2_slot_type;
        v.shift = s2_shift; v.ext = s2_ext; v.all_counted = s2_all_counted;
        return v;
    }
    // single-cell cell table (sc.cuh ScTableView)
    u32* sc_sectors = nullptr;
    uint2* sc_cells = nullptr;
    u32* sc_ovf_base = nullptr;
    u32* sc_pair_key = nullptr;
    uint8_t* sc_pair_type = nullptr;
    int sc_shift = 11;
    bool has_sc_stab = false;
    size_t sc_stab_bytes = 0;
    StabView sc_stab_view() const {
        StabView v;
        v.sectors = sc_sectors; v.cells = sc_cells; v.slot_type = sc_pair_type; v.ovf_base = sc_ovf_base;
        v.shift = sc_shift; v.all_counted = 0;
        return v;
    }
    IndexView view() const {
        IndexView v;
        v.L = L; v.R = R; v.pmaxR = pmaxR; v.info = info; v.chrom_off = chrom_off;
        v.dir = dir; v.dir_off = dir_off; v.chrom_valid = chrom_valid; v.n_chrom = n_chrom; v.shift = shift; v.bs = bs; v.n_ensg = n_ensg;
        return v;
    }
};

struct StageSlot {
    void* base = nullptr;
    int32_t* start = nullptr;
    int32_t* end = nullptr;
    uint16_t* chrom = nullptr;
    uint8_t* mapq = nullptr;
    uint8_t* flag = nullptr;
    u32* cell = nullptr;
    u64* umi = nullptr;
};

struct ScState;      // sc.cuh
struct NameState;    // pair_name.cuh
struct tec_ctx;
static int name_flush(tec_ctx* ctx);     // pair_name.cuh: the rows still pending count as no-mate

// Size-keyed cache of device blocks: the single-cell finalize asks for the same sequence of
// temporaries on every call, and cudaMalloc / cudaFree (a device-wide synchronisation each) would
// otherwise sit inside the timed path.
struct DevCache {
    std::multimap<size_t, void*> free_blocks;
    std::map<void*, size_t> live;
    size_t cached_bytes = 0;
    cudaError_t get(void** out, size_t bytes) {
        bytes = (std::max<size_t>(bytes, 1) + 511) & ~size_t(511);
        auto it = free_blocks.lower_bound(bytes);
        if (it != free_blocks.end() && it->first <= bytes + (bytes >> 2) + (size_t(1) << 20)) {
            *out = it->second;
            live[*out] = it->first;
            cached_bytes -= it->first;
            free_blocks.erase(it);
            return cudaSuccess;
        }
        cudaError_t e = cudaMalloc(out, bytes);
        if (e != cudaSuccess) {
            cudaGetLastError();
            trim();
            e = cudaMalloc(out, bytes);
            if (e != cudaSuccess) cudaGetLastError();      // an allocation failure is not sticky: do not leave it for the next check
        }
        if (e == cudaSuccess) live[*out] = bytes;
        return e;
    }
    void put(void* p) {
        if (!p) return;
        auto it = live.find(p);
        if (it == live.end()) { cudaFree(p); return; }
        free_blocks.emplace(it->second, p);
        cached_bytes += it->second;
        live.erase(it);
    }
    void trim() {
        for (auto& kv : free_blocks) cudaFree(kv.second);
        free_blocks.clear();
        cached_bytes = 0;
    }
};

// log2 of the cell size of the two cell tables.  Bulk: 1 kbp cells (104 MB for the hg38-like index) measured
// 125.9e9 records/s against 121.1e9 with 2 kbp cells (65 MB): fewer overflow sectors outweigh the extra L2 misses.
#define TEC_BULK_STAB_SHIFT 10
#define TEC_BULK_STAB2_SHIFT 10
#define TEC_SC_STAB_SHIFT 11

struct tec_ctx {
    int device = 0;
    int n_sm = 148;
    int smem_optin = 227 * 1024;
    cudaStream_t stream = nullptr, copy_stream = nullptr;
    cudaEvent_t stage_ready[2] = {nullptr, nullptr}, stage_free[2] = {nullptr, nullptr};
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bool timed = false;
    int64_t launches = 0;
    std::string err;

    DevIndex idx;
    bool has_index = false;

    // bulk
    bool bulk_active = false;
    int paired = 0, qual = 20;
    u64* d_counts = nullptr;              // the bulk counter block (bulk_words)
    u64* d_bank1 = nullptr;               // paired-end byte range: the counters of the pairs of odd range-local index (same layout)
    int64_t counts_cap = 0, bank1_cap = 0;   // words allocated at d_counts / d_bank1
    bool loci = false;                    // this run tallies index rows too (opt_bulk_loci at tec_bulk_begin)
    bool bank_pending = false;            // a paired-end range count waits for tec_bulk_keep_bank
    bool name_pairing = false;            // tec_bulk_begin(ctx, 2, qual): mates paired by read name (pair_name.cuh)
    NameState* name = nullptr;
    bool name_held = false;               // tec_bam_count_range mode 4 holds rows that wait for tec_bulk_name_partition_dev
    u32* d_slow_list = nullptr;           // [0] = count, then unit indices flagged for bulk_slow_kernel
    int64_t slow_cap = 0;                 // words
    void* d_ring = nullptr;               // per-warp second deferral ring of the fast bulk kernel (QEnt)
    u32* d_ring_u = nullptr;
    int64_t ring_cap = 0;                 // entries
    u32* d_defer_list = nullptr;          // bulk2: per-warp segments of deferred unit indices
    u32* d_defer_count = nullptr;         // bulk2: entries per segment
    int64_t defer_cap = 0, defer_warps = 0, last_defer_n = 0;
    u32* d_part_count = nullptr;          // bulk2: entries bulk2_pair_kernel left per (segment, part)
    int64_t part_cap = 0, last_part_n = 0;
    std::vector<int32_t> ensg_of_slot;    // slot = rank of an ensg by number of feature rows
    // options (tec_set_option)
    int opt_bulk_algo = -1;               // -1 auto, 0 exact search kernel, 1 cell-table kernel with in-kernel rings (round 1), 2 two-pass kernels (bulk2.cuh)
    int opt_stab_shift = 0;               // log2 of the cell size; 0 = TEC_BULK_STAB_SHIFT / TEC_SC_STAB_SHIFT
    int opt_bulk_mode = 77;               // fast bulk kernel: bit 0 table sectors evict_last in L2, bit 1 prefetch the next tile's sectors,
                                          // bit 2 tally through the per-warp hit queue, bit 3 512-thread CTAs with three tiles in flight per warp,
                                          // bit 4 queue filled behind a warp prefix sum, bit 5 768-thread CTAs, bit 6 queue drained once per tile
    int opt_bulk_strand = 0;              // extension (not in the reference): strand-aware bulk counting, exact kernel only
    int opt_bulk_loci = 0;                // extension: count per index row too (read at tec_bulk_begin), exact kernel only
    int opt_second_parts = 4;             // warps of the second bulk pass (and of bulk2_pair_kernel) per segment of the deferred list
    int opt_second_mode = 2;              // second bulk pass: register set of distinct ensg, 0 stored by position, 1 shifted in; 2: units that
                                          // two sectors answer go through the straight-line bulk2_pair_kernel first
    int opt_all_hot = 1;                  // counters of every ensg in shared memory when they fit
    int opt_sc_sort = 1;                  // single cell: packed 64-bit keys + the 11-bit radix sort of csrc/radix.cuh (0: library sort, two stages)
    int opt_sc_prev_partition = 0;        // single cell: 0 prev[] by random 4-byte stores (default); 1 / 2 through one radix pass on the position
                                          // (measured SLOWER at 1 B records: 167.6 vs 156.0 ms per step, gpurun_out/r02w; 2 = also on small inputs, tests)
    int opt_sc_pack_umi = 1;              // single cell: 2-bit UMI sort keys when every UMI is fixed-length ACGT
    int opt_sc_algo = -1;                 // -1 auto, 0 exact search only, 1 cell table
    // single cell, last finalize (tec_get_info): 1 packed keys + radix.cuh, 2 library sorts on 2-bit UMI keys, 3 library sorts
    // on 3-bit UMI codes, 0 nothing sorted; and the radix passes of the packed sort
    int sc_last_sort = 0;
    int sc_last_sort_passes = 0;
    int opt_bam_lanes = 1;                // BGZF blocks decoded per warp by the inflate kernel (1..32): the streams of a warp
                                          // diverge on every symbol; measured 201 ms (1) / 206 (2) / 241 (8) / 398 (32) per 3.7 GB
    int opt_bam_window_blocks = 65536;    // BGZF blocks decoded per pass by tec_bam_count (one thread each)
    int opt_ctas_per_sm = 2;              // resident CTAs per SM of the fast bulk kernel (512 threads each)

    // host staging
    StageSlot stage[2];
    int64_t stage_cap = 0;
    bool stage_sc = false;
    int stage_next = 0;

    ScState* sc = nullptr;
    void* comm = nullptr;                 // ncclComm_t of tec_comm_init (collective.cuh); the library's own collectives run on `stream`
    int comm_rank = 0, comm_world = 1;
    uint8_t* bam_pinned[2] = {nullptr, nullptr};    // staging chunks of the device BAM decoder (bamgpu.cuh)
    cudaEvent_t bam_ev[3] = {nullptr, nullptr, nullptr};
    cudaStream_t bam_stream2 = nullptr;
    DevCache cache;

    int ensure_stage(int64_t n, bool sc_layout);
    void free_stage();
    void free_index();
    void free_sc();
    void free_name();
    void free_bam() {
        for (int i = 0; i < 2; i++) {
            if (bam_pinned[i]) cudaFreeHost(bam_pinned[i]);
            bam_pinned[i] = nullptr;
        }
        for (int i = 0; i < 3; i++) {
            if (bam_ev[i]) cudaEventDestroy(bam_ev[i]);
            bam_ev[i] = nullptr;
        }
        if (bam_stream2) cudaStreamDestroy(bam_stream2);
        bam_stream2 = nullptr;
    }
    void free_all() { free_stage(); free_index(); free_sc(); free_name(); free_bam(); cache.trim(); }
    // Words of the bulk counter block: n_ensg counters (slot order), TEC_BULK_NSTATS statistics and, in a run with
    // loci, one counter per index row (upload order).  Every copy, clear and reduction of the block takes this length.
    size_t bulk_words() const { return (size_t)idx.n_ensg + TEC_BULK_NSTATS + (loci ? (size_t)idx.n_feat : 0); }
};

inline void tec_ctx::free_stage() {
    for (int i = 0; i < 2; ++i) {
        if (stage[i].base) cudaFree(stage[i].base);
        stage[i] = StageSlot();
    }
    stage_cap = 0;
}

inline void tec_ctx::free_index() {
    DevIndex& ix = idx;
    cudaFree(ix.L); cudaFree(ix.R); cudaFree(ix.pmaxR); cudaFree(ix.info);
    cudaFree(ix.chrom_off); cudaFree(ix.dir); cudaFree(ix.dir_off); cudaFree(ix.chrom_valid);
    cudaFree(ix.st_sectors); cudaFree(ix.st_cells); cudaFree(ix.st_slot_type); cudaFree(ix.st_ovf_base);
    cudaFree(ix.s2_sectors); cudaFree(ix.s2_cells); cudaFree(ix.s2_ovf_first); cudaFree(ix.s2_slot_type);
    cudaFree(ix.sc_sectors); cudaFree(ix.sc_cells); cudaFree(ix.sc_ovf_base); cudaFree(ix.sc_pair_key); cudaFree(ix.sc_pair_type);
    ix = DevIndex();
    cudaFree(d_counts);
    d_counts = nullptr;
    cudaFree(d_bank1);
    d_bank1 = nullptr;
    counts_cap = bank1_cap = 0;
    loci = false;
    bank_pending = false;
    cudaFree(d_slow_list);
    d_slow_list = nullptr;
    cudaFree(d_ring); cudaFree(d_ring_u);
    d_ring = nullptr; d_ring_u = nullptr; ring_cap = 0;
    cudaFree(d_defer_list); cudaFree(d_defer_count); cudaFree(d_part_count);
    d_defer_list = nullptr; d_defer_count = nullptr; defer_cap = 0; defer_warps = 0; last_defer_n = 0;
    d_part_count = nullptr; part_cap = 0; last_part_n = 0;
    slow_cap = 0;
    has_index = false;
    bulk_active = false;
}

// two staging slots, each one allocation carved into the SoA columns (256-byte aligned)
inline int tec_ctx::ensure_stage(int64_t n, bool sc_layout) {
    tec_ctx* ctx = this;
    if (n <= stage_cap && (stage_sc || !sc_layout)) return TEC_OK;
    TEC_CUDA(cudaStreamSynchronize(stream));
    TEC_CUDA(cudaStreamSynchronize(copy_stream));
    free_stage();
    const int64_t cap = std::max<int64_t>(n, 1 << 16);
    auto al = [](size_t b) { return (b + 255) & ~size_t(255); };
    const size_t o_start = 0, o_end = o_start + al((size_t)cap * 4), o_chrom = o_end + al((size_t)cap * 4),
                 o_mapq = o_chrom + al((size_t)cap * 2), o_flag = o_mapq + al((size_t)cap),
                 o_cell = o_flag + al((size_t)cap), o_umi = o_cell + (sc_layout ? al((size_t)cap * 4) : 0),
                 total = o_umi + (sc_layout ? al((size_t)cap * 8) : 0);
    for (int i = 0; i < 2; ++i) {
        TEC_CUDA(cudaMalloc(&stage[i].base, total));
        char* b = (char*)stage[i].base;
        stage[i].start = (int32_t*)(b + o_start);
        stage[i].end = (int32_t*)(b + o_end);
        stage[i].chrom = (uint16_t*)(b + o_chrom);
        stage[i].mapq = (uint8_t*)(b + o_mapq);
        stage[i].flag = (uint8_t*)(b + o_flag);
        stage[i].cell = sc_layout ? (u32*)(b + o_cell) : nullptr;
        stage[i].umi = sc_layout ? (u64*)(b + o_umi) : nullptr;
    }
    stage_cap = cap;
    stage_sc = sc_layout;
    // mark both slots free
    for (int i = 0; i < 2; ++i) TEC_CUDA(cudaEventRecord(stage_free[i], stream));
    return TEC_OK;
}
