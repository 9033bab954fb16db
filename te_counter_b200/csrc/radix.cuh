// Stable LSD radix sort of (key, u32 value) pairs with digits of up to 11 bits, written for sm_100a.
//
// Used by the single-cell path (sc.cuh): the (cell, UMI) key groups of te_count.py:440-473 are found by
// sorting the survivors by a packed key, value = position in the file.  A library sort moves the pairs once
// per 8 bits of key; here a pass takes 11 bits, so the 41 key bits of the 10x configuration (17 bits of cell,
// 24 of UMI) need four passes instead of six.
//
// One pass = a count, a prefix sum and a scatter; no CTA ever waits for another one (nothing can hang):
//   rdx_hist_kernel     the input is cut into chunks of `chunk_tiles` tiles of RDX_TILE items (one tile by default: tools/radix_test sweeps, profiles/);
//                       CTA c counts the digits of chunk c in shared memory: counts[digit][chunk]
//   rdx_scan_*          exclusive prefix sum over (digit major, chunk minor): where each chunk's run of each digit
//                       starts (three kernels: block sums, their scan, block scans)
//   rdx_scatter_kernel  CTA c moves chunk c, tile by tile.  CTAs start in the order of their numbers, so at any moment
//                       the few hundred chunks in flight are neighbours in the input and, for every digit, write to
//                       neighbouring addresses: the partially written 32-byte sectors of the 2 x 2048 write fronts are
//                       completed in L2 by the neighbour CTAs before they are evicted.  (The first version gave every
//                       CTA 1/296 of the input: 1.2 M independent write fronts, more than L2 holds, and 2.6 x the
//                       algorithmic DRAM write traffic, profiles/r02_sc_launches_1b.md.)
//                       Inside a tile (6144 pairs, 24 per thread, two CTAs per SM) the stable rank of an item comes from
//                       match.any: the lanes of a warp that hold the same digit in one round find each other with one
//                       instruction, the lowest one advances the warp's own 16-bit counter of that digit; a scan over
//                       (digit, warp) turns the counters into tile positions.  The tile is then laid out in shared
//                       memory in sorted order (over the counters, which are dead by then) and leaves the SM as runs of
//                       consecutive addresses, 32 consecutive tile positions per store instruction.
// Bytes per pass and pair: key read twice (count, scatter), value read once, both written once; the counts matrix adds
// 4 x 4 bytes per (digit, chunk) = 22 % at one tile per chunk.
#pragma once
#include "common.cuh"

#define RDX_THREADS 256
#define RDX_WARPS (RDX_THREADS / 32)
#define RDX_ITEMS 24
#define RDX_TILE (RDX_THREADS * RDX_ITEMS)          // 6144
#define RDX_WARP_ITEMS (32 * RDX_ITEMS)             // 768: a warp's items are tile positions [w * 768, w * 768 + 768)
#define RDX_MAX_BITS 11
#define RDX_MAX_BINS (1 << RDX_MAX_BITS)
#define RDX_BINS_PER_THREAD (RDX_MAX_BINS / RDX_THREADS)     // 8
#define RDX_SCAN_BLOCK 8192                         // elements of the counts matrix per CTA of the prefix sum

template <class K> __device__ __forceinline__ u32 rdx_digit(K key, int shift, u32 mask) { return (u32)(key >> shift) & mask; }

template <class K>
__global__ void __launch_bounds__(512)
rdx_hist_kernel(const K* __restrict__ keys, int64_t n, int shift, int bits, int64_t chunk_items, u32* __restrict__ counts) {
    __shared__ u32 hist[RDX_MAX_BINS];
    const u32 nb = 1u << bits, mask = nb - 1u;
    for (u32 i = threadIdx.x; i < nb; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    const int64_t lo = (int64_t)blockIdx.x * chunk_items;
    const int64_t hi = min(n, lo + chunk_items);
    for (int64_t i = lo + threadIdx.x; i < hi; i += blockDim.x) atomicAdd(&hist[rdx_digit(keys[i], shift, mask)], 1u);
    __syncthreads();
    for (u32 i = threadIdx.x; i < nb; i += blockDim.x) counts[(size_t)i * gridDim.x + blockIdx.x] = hist[i];
}

// ---- exclusive prefix sum of m counters in place: block sums, scan of the block sums by one CTA, block scans
__device__ __forceinline__ u32 rdx_block_excl_scan_1024(u32 v, u32* warp_tot /* shared [32] */, u32* total) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    u32 incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const u32 t = __shfl_up_sync(0xFFFFFFFFu, incl, d);
        if (lane >= d) incl += t;
    }
    if (lane == 31) warp_tot[w] = incl;
    __syncthreads();
    if (w == 0) {
        const u32 x = warp_tot[lane];
        u32 y = x;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const u32 t = __shfl_up_sync(0xFFFFFFFFu, y, d);
            if (lane >= d) y += t;
        }
        warp_tot[lane] = y - x;
        if (lane == 31 && total) *total = y;
    }
    __syncthreads();
    return warp_tot[w] + incl - v;
}

__global__ void __launch_bounds__(1024)
rdx_scan_sums_kernel(const u32* __restrict__ v, int64_t m, u32* __restrict__ sums) {
    __shared__ u32 warp_tot[32];
    __shared__ u32 total;
    const int64_t a = (int64_t)blockIdx.x * RDX_SCAN_BLOCK + (int64_t)threadIdx.x * 8;
    u32 s = 0;
    if (a + 8 <= m) {
        const uint4 x = *reinterpret_cast<const uint4*>(v + a), y = *reinterpret_cast<const uint4*>(v + a + 4);
        s = x.x + x.y + x.z + x.w + y.x + y.y + y.z + y.w;
    } else {
        for (int64_t i = a; i < m; ++i) s += v[i];
    }
    rdx_block_excl_scan_1024(s, warp_tot, &total);
    if (threadIdx.x == 0) sums[blockIdx.x] = total;
}

// exclusive prefix sum of m counters by one CTA of 1024 threads (the block sums: a few thousand)
__global__ void __launch_bounds__(1024)
rdx_scan_kernel(u32* __restrict__ v, int64_t m) {
    __shared__ u32 warp_tot[32];
    const int64_t per = (m + 1023) / 1024;
    const int64_t a = min(m, (int64_t)threadIdx.x * per), b = min(m, a + per);
    u32 sum = 0;
    for (int64_t i = a; i < b; ++i) sum += v[i];
    u32 run = rdx_block_excl_scan_1024(sum, warp_tot, nullptr);
    for (int64_t i = a; i < b; ++i) { const u32 c = v[i]; v[i] = run; run += c; }
}

__global__ void __launch_bounds__(1024)
rdx_scan_apply_kernel(u32* __restrict__ v, int64_t m, const u32* __restrict__ sums) {
    __shared__ u32 warp_tot[32];
    const int64_t a = (int64_t)blockIdx.x * RDX_SCAN_BLOCK + (int64_t)threadIdx.x * 8;
    u32 e[8];
    const bool full = a + 8 <= m;
    if (full) {
        const uint4 x = *reinterpret_cast<const uint4*>(v + a), y = *reinterpret_cast<const uint4*>(v + a + 4);
        e[0] = x.x; e[1] = x.y; e[2] = x.z; e[3] = x.w; e[4] = y.x; e[5] = y.y; e[6] = y.z; e[7] = y.w;
    } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) e[i] = a + i < m ? v[a + i] : 0u;
    }
    u32 s = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += e[i];
    u32 run = rdx_block_excl_scan_1024(s, warp_tot, nullptr) + sums[blockIdx.x];
#pragma unroll
    for (int i = 0; i < 8; ++i) { const u32 c = e[i]; e[i] = run; run += c; }
    if (full) {
        *reinterpret_cast<uint4*>(v + a) = make_uint4(e[0], e[1], e[2], e[3]);
        *reinterpret_cast<uint4*>(v + a + 4) = make_uint4(e[4], e[5], e[6], e[7]);
    } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) if (a + i < m) v[a + i] = e[i];
    }
}

// ---- scatter
template <class K> struct RdxSmem {
    // the warps' digit counters while the tile is ranked, the tile in sorted order afterwards
    union {
        unsigned short wcnt[RDX_WARPS][RDX_MAX_BINS];                 // 32 KB
        struct { K keys[RDX_TILE]; u32 vals[RDX_TILE]; } tile;        // 72 KB (64-bit keys)
    } u;
    u32 goff[RDX_MAX_BINS];                         // where the chunk's next item of each digit goes
    u32 delta[RDX_MAX_BINS];                        // per tile: goff[d] - (tile position of the digit's first item)
    u32 warp_tot[RDX_WARPS];
};

template <class K, bool HAS_VALUES>
__global__ void __launch_bounds__(RDX_THREADS, 2)
rdx_scatter_kernel(const K* __restrict__ keys_in, const u32* __restrict__ vals_in, K* __restrict__ keys_out, u32* __restrict__ vals_out,
                   int64_t n, int shift, int bits, int64_t chunk_tiles, const u32* __restrict__ starts) {
    extern __shared__ __align__(16) unsigned char rdx_smem_raw[];
    RdxSmem<K>& sm = *reinterpret_cast<RdxSmem<K>*>(rdx_smem_raw);
    const u32 nb = 1u << bits, mask = nb - 1u;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const u32 lt = (1u << lane) - 1u;
    const int64_t n_tiles = (n + RDX_TILE - 1) / RDX_TILE;
    const int64_t t0 = (int64_t)blockIdx.x * chunk_tiles, t1 = min(n_tiles, t0 + chunk_tiles);
    const u32 p0 = (u32)w * RDX_WARP_ITEMS + (u32)lane;
    unsigned short* const myc = sm.u.wcnt[w];
    K key[RDX_ITEMS];
    u32 val[RDX_ITEMS];
    // the items of a tile, as loaded: item r of a thread is tile position p0 + 32 r
    auto load_tile = [&](int64_t tile) {
        const int64_t g0 = tile * RDX_TILE;
        const u32 nv = (u32)min((int64_t)RDX_TILE, n - g0);
#pragma unroll
        for (int r = 0; r < RDX_ITEMS; ++r) {
            const u32 p = p0 + (u32)r * 32u;
            key[r] = p < nv ? keys_in[g0 + p] : (K)0;
            if (HAS_VALUES) val[r] = p < nv ? vals_in[g0 + p] : 0u;
        }
    };
    // the first tile and the chunk's write positions are requested together (one exposed round trip per chunk; the
    // next tile's items are requested while the current one is written out)
    if (t0 < t1) load_tile(t0);
    {
        u32 g[RDX_BINS_PER_THREAD];
#pragma unroll
        for (int i = 0; i < RDX_BINS_PER_THREAD; ++i) {
            const u32 d = threadIdx.x + (u32)i * RDX_THREADS;
            g[i] = d < nb ? starts[(size_t)d * gridDim.x + blockIdx.x] : 0u;
        }
#pragma unroll
        for (int i = 0; i < RDX_BINS_PER_THREAD; ++i) sm.goff[threadIdx.x + (u32)i * RDX_THREADS] = g[i];
    }
    for (int64_t tile = t0; tile < t1; ++tile) {
        const int64_t g0 = tile * RDX_TILE;
        const u32 n_valid = (u32)min((int64_t)RDX_TILE, n - g0);       // < RDX_TILE only in the last tile of the input
        // ---- counters to zero (the previous tile's sorted copy lies there; its readers are past the barrier below)
        {
            uint4* z = reinterpret_cast<uint4*>(&sm.u.wcnt[0][0]);
#pragma unroll
            for (int i = 0; i < (int)(sizeof(sm.u.wcnt) / 16 / RDX_THREADS); ++i) z[threadIdx.x + i * RDX_THREADS] = make_uint4(0u, 0u, 0u, 0u);
        }
        u32 rk[RDX_ITEMS / 2];                                         // two 16-bit ranks / tile positions per word
        __syncthreads();
        // ---- rank inside the warp: round r holds tile positions p0 + 32 r, so (round, lane) is the tile order
#pragma unroll
        for (int r = 0; r < RDX_ITEMS; ++r) {
            const bool valid = p0 + (u32)r * 32u < n_valid;
            const u32 d = rdx_digit(key[r], shift, mask);
            const u32 peers = __match_any_sync(0xFFFFFFFFu, valid ? d : 0xFFFFFFFFu);
            const u32 below = __popc(peers & lt);
            const u32 cnt = myc[d];
            const u32 rank = cnt + below;
            if (r & 1) rk[r >> 1] |= rank << 16; else rk[r >> 1] = rank;
            __syncwarp();
            if (below == 0 && valid) myc[d] = (unsigned short)(cnt + __popc(peers));
            __syncwarp();
        }
        __syncthreads();
        // ---- per digit: exclusive sum over the warps, digit totals -> tile position of every (digit, warp) run.
        // A thread owns 8 consecutive digits (16 bytes of every warp's row); 16-bit lanes never carry (sums <= 6144).
        {
            const u32 b0 = threadIdx.x * RDX_BINS_PER_THREAD;
            uint4 tot = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
            for (int x = 0; x < RDX_WARPS; ++x) {
                const uint4 c = *reinterpret_cast<const uint4*>(&sm.u.wcnt[x][b0]);
                tot.x += c.x; tot.y += c.y; tot.z += c.z; tot.w += c.w;
            }
            u32 t[RDX_BINS_PER_THREAD] = {tot.x & 0xFFFFu, tot.x >> 16, tot.y & 0xFFFFu, tot.y >> 16,
                                          tot.z & 0xFFFFu, tot.z >> 16, tot.w & 0xFFFFu, tot.w >> 16};
            u32 s = 0;
#pragma unroll
            for (int i = 0; i < RDX_BINS_PER_THREAD; ++i) s += t[i];
            // block-wide exclusive sum of the threads' totals
            u32 incl = s;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const u32 y = __shfl_up_sync(0xFFFFFFFFu, incl, d);
                if (lane >= d) incl += y;
            }
            if (lane == 31) sm.warp_tot[w] = incl;
            __syncthreads();
            u32 base = incl - s;
#pragma unroll
            for (int x = 0; x < RDX_WARPS; ++x) base += x < w ? sm.warp_tot[x] : 0u;
            u32 st[RDX_BINS_PER_THREAD];                                // tile position of the digit's first item
#pragma unroll
            for (int i = 0; i < RDX_BINS_PER_THREAD; ++i) { st[i] = base; base += t[i]; }
            uint4 run = make_uint4(st[0] | st[1] << 16, st[2] | st[3] << 16, st[4] | st[5] << 16, st[6] | st[7] << 16);
#pragma unroll
            for (int x = 0; x < RDX_WARPS; ++x) {
                uint4* q = reinterpret_cast<uint4*>(&sm.u.wcnt[x][b0]);
                const uint4 c = *q;
                *q = run;
                run.x += c.x; run.y += c.y; run.z += c.z; run.w += c.w;
            }
            // where the digit's run goes, and the chunk's write positions moved past this tile
            uint4* go = reinterpret_cast<uint4*>(&sm.goff[b0]);
            uint4* de = reinterpret_cast<uint4*>(&sm.delta[b0]);
            const uint4 g0v = go[0], g1v = go[1];
            de[0] = make_uint4(g0v.x - st[0], g0v.y - st[1], g0v.z - st[2], g0v.w - st[3]);
            de[1] = make_uint4(g1v.x - st[4], g1v.y - st[5], g1v.z - st[6], g1v.w - st[7]);
            go[0] = make_uint4(g0v.x + t[0], g0v.y + t[1], g0v.z + t[2], g0v.w + t[3]);
            go[1] = make_uint4(g1v.x + t[4], g1v.y + t[5], g1v.z + t[6], g1v.w + t[7]);
        }
        __syncthreads();
        // ---- tile position of every item
#pragma unroll
        for (int r = 0; r < RDX_ITEMS; ++r) {
            const u32 d = rdx_digit(key[r], shift, mask);
            const u32 add = myc[d];
            rk[r >> 1] += (r & 1) ? add << 16 : add;
        }
        __syncthreads();                                               // the counters are dead: the sorted tile goes over them
#pragma unroll
        for (int r = 0; r < RDX_ITEMS; ++r) {
            if (p0 + (u32)r * 32u < n_valid) {
                const u32 pos = (r & 1) ? rk[r >> 1] >> 16 : rk[r >> 1] & 0xFFFFu;
                sm.u.tile.keys[pos] = key[r];
                if (HAS_VALUES) sm.u.tile.vals[pos] = val[r];
            }
        }
        if (tile + 1 < t1) load_tile(tile + 1);                        // the registers are free: the next tile is on its way
        __syncthreads();
        // ---- out: 32 consecutive tile positions per store instruction
#pragma unroll
        for (int r = 0; r < RDX_ITEMS; ++r) {
            const u32 p = threadIdx.x + (u32)r * RDX_THREADS;
            if (p < n_valid) {
                const K k = sm.u.tile.keys[p];
                const u32 dst = sm.delta[rdx_digit(k, shift, mask)] + p;
                keys_out[dst] = k;
                if (HAS_VALUES) vals_out[dst] = sm.u.tile.vals[p];
            }
        }
        __syncthreads();
    }
}

// ---- host side -----------------------------------------------------------------------------------------------------
static int g_rdx_max_bits = RDX_MAX_BITS;          // widest digit of a pass (experiments: tools/radix_test)
static int g_rdx_chunk_tiles = 1;                  // tiles per chunk (a chunk = one CTA of the count and of the scatter)

struct RdxPlan {
    int n_chunks = 0;
    int64_t chunk_tiles = 0;
    int64_t n_scan_blocks = 0;
    size_t counts_bytes = 0;                        // scratch: u32 [2048][n_chunks], then the block sums of the prefix sum
};

static inline RdxPlan rdx_plan(int64_t n, int n_sm) {
    (void)n_sm;
    RdxPlan p;
    const int64_t n_tiles = std::max<int64_t>(1, (n + RDX_TILE - 1) / RDX_TILE);
    p.chunk_tiles = std::max(1, g_rdx_chunk_tiles);
    p.n_chunks = (int)((n_tiles + p.chunk_tiles - 1) / p.chunk_tiles);
    const int64_t m = (int64_t)RDX_MAX_BINS * p.n_chunks;
    p.n_scan_blocks = (m + RDX_SCAN_BLOCK - 1) / RDX_SCAN_BLOCK;
    p.counts_bytes = (size_t)(m + 8 + p.n_scan_blocks) * 4;
    return p;
}

// one stable pass on key bits [shift, shift + bits), bits <= 11; scratch: plan.counts_bytes
template <class K, bool HAS_VALUES>
static cudaError_t rdx_pass(const K* keys_in, const u32* vals_in, K* keys_out, u32* vals_out, int64_t n, int shift, int bits,
                            const RdxPlan& plan, u32* scratch, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    const int64_t m = ((int64_t)1 << bits) * plan.n_chunks;
    const int64_t nblk = (m + RDX_SCAN_BLOCK - 1) / RDX_SCAN_BLOCK;
    u32* sums = scratch + (((int64_t)RDX_MAX_BINS * plan.n_chunks + 7) & ~(int64_t)7);
    rdx_hist_kernel<K><<<plan.n_chunks, 512, 0, st>>>(keys_in, n, shift, bits, plan.chunk_tiles * RDX_TILE, scratch);
    rdx_scan_sums_kernel<<<(unsigned)nblk, 1024, 0, st>>>(scratch, m, sums);
    rdx_scan_kernel<<<1, 1024, 0, st>>>(sums, nblk);
    rdx_scan_apply_kernel<<<(unsigned)nblk, 1024, 0, st>>>(scratch, m, sums);
    auto kfn = rdx_scatter_kernel<K, HAS_VALUES>;
    cudaError_t e = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(RdxSmem<K>));
    if (e != cudaSuccess) return e;
    kfn<<<plan.n_chunks, RDX_THREADS, sizeof(RdxSmem<K>), st>>>(keys_in, vals_in, keys_out, vals_out, n, shift, bits, plan.chunk_tiles, scratch);
    return cudaGetLastError();
}
#define RDX_LAUNCHES_PER_PASS 5

// digit widths of a sort over `total` key bits (at most 64): ceil(total / max_bits) passes whose widths differ by at most
// one, wider passes first; returns the number of passes
static inline int rdx_digit_widths(int total, int widths[64]) {
    total = std::min(64, std::max(0, total));
    const int max_bits = std::min(RDX_MAX_BITS, std::max(1, g_rdx_max_bits));
    const int passes = (total + max_bits - 1) / max_bits;
    for (int i = 0, done = 0; i < passes; ++i) done += widths[i] = (total - done + (passes - i) - 1) / (passes - i);
    return passes;
}

// stable sort on key bits [bit_lo, bit_hi) in ceil((bit_hi - bit_lo) / 11) passes of equal width, ping-pong between
// (keys_a, vals_a) and (keys_b, vals_b); *in_b says where the result is.  n < 2^32 - 2^13.
template <class K, bool HAS_VALUES>
static cudaError_t rdx_sort(K* keys_a, u32* vals_a, K* keys_b, u32* vals_b, int64_t n, int bit_lo, int bit_hi, int n_sm,
                            u32* scratch, cudaStream_t st, bool* in_b, int* n_passes = nullptr) {
    int widths[64];
    const int passes = rdx_digit_widths(bit_hi - bit_lo, widths);
    const RdxPlan plan = rdx_plan(n, n_sm);
    bool flip = false;
    int done = 0;
    for (int i = 0; i < passes; ++i) {
        const int bits = widths[i];
        cudaError_t e = flip ? rdx_pass<K, HAS_VALUES>(keys_b, vals_b, keys_a, vals_a, n, bit_lo + done, bits, plan, scratch, st)
                             : rdx_pass<K, HAS_VALUES>(keys_a, vals_a, keys_b, vals_b, n, bit_lo + done, bits, plan, scratch, st);
        if (e != cudaSuccess) return e;
        done += bits;
        flip = !flip;
    }
    *in_b = flip;
    if (n_passes) *n_passes = passes;
    return cudaSuccess;
}
