// C entry points over te_counter_b200/csrc/radix.cuh for tests/test_gpu_radix.py: rdx_sort and rdx_pass on device
// pointers the caller owns (torch tensors), with this library's own copies of the digit width and chunk size.
// Every call allocates its scratch, runs on the legacy default stream and waits for the result.
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -shared -Xcompiler -fPIC -I te_counter_b200/csrc tests/radix_harness.cu
#include "radix.cuh"

namespace {
template <class K, bool V>
int sort_one(void* ka, void* va, void* kb, void* vb, int64_t n, int lo, int hi, int* in_b, int* passes) {
    u32* scratch = nullptr;
    cudaError_t e = cudaMalloc(&scratch, rdx_plan(n, 148).counts_bytes);
    if (e != cudaSuccess) return (int)e;
    bool b = false;
    e = rdx_sort<K, V>((K*)ka, (u32*)va, (K*)kb, (u32*)vb, n, lo, hi, 148, scratch, 0, &b, passes);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    cudaFree(scratch);
    *in_b = b ? 1 : 0;
    return (int)e;
}
}  // namespace

extern "C" {

void rh_set(int max_bits, int chunk_tiles) {
    g_rdx_max_bits = max_bits;
    g_rdx_chunk_tiles = chunk_tiles;
}

// key_bytes 4 or 8; has_values 0: the value pointers are not read (the keys-only sort of the triples)
int rh_sort(int key_bytes, int has_values, void* ka, void* va, void* kb, void* vb, int64_t n, int lo, int hi, int* in_b, int* passes) {
    if (key_bytes == 8)
        return has_values ? sort_one<u64, true>(ka, va, kb, vb, n, lo, hi, in_b, passes) : sort_one<u64, false>(ka, va, kb, vb, n, lo, hi, in_b, passes);
    return has_values ? sort_one<u32, true>(ka, va, kb, vb, n, lo, hi, in_b, passes) : sort_one<u32, false>(ka, va, kb, vb, n, lo, hi, in_b, passes);
}

// digit widths rdx_sort uses for `total` key bits at the current max_bits; returns the number of passes
int rh_digit_bits(int total, int* bits /* [64] */) { return rdx_digit_widths(total, bits); }

// one stable pass of u32 keys with values on bits [shift, shift + bits) (the prev[] partition of sc.cuh)
int rh_pass_u32(const void* kin, const void* vin, void* kout, void* vout, int64_t n, int shift, int bits) {
    const RdxPlan plan = rdx_plan(n, 148);
    u32* scratch = nullptr;
    cudaError_t e = cudaMalloc(&scratch, plan.counts_bytes);
    if (e != cudaSuccess) return (int)e;
    e = rdx_pass<u32, true>((const u32*)kin, (const u32*)vin, (u32*)kout, (u32*)vout, n, shift, bits, plan, scratch, 0);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    cudaFree(scratch);
    return (int)e;
}

}  // extern "C"
