"""csrc/radix.cuh (rdx_sort, rdx_pass) against numpy's stable argsort of the digit field, through the C entry points
of tests/radix_harness.cu: whole keys (bits outside [lo, hi) included), values, the buffer the result lands in and
the number of passes must all be exact.  Sizes around a warp's items, a tile and 1024 block sums of the single-CTA
prefix sum; bit ranges up to bit 63 and widths that split into unequal digits; digit widths of 1 to 11 bits; 1 to
64 tiles per chunk; key distributions that stress the ranking (all equal, all-ones digits, descending, keys that only
differ outside the sorted field)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from te_counter_b200 import build

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TILE = 6144


@pytest.fixture(scope="module")
def rh(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("radix") / "libradixharness.so")
    subprocess.run([build.NVCC, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-shared",
                    "-Xcompiler", "-fPIC", "-I", os.path.join(ROOT, "te_counter_b200", "csrc"), "-o", out,
                    os.path.join(ROOT, "tests", "radix_harness.cu")], check=True)
    lib = ctypes.CDLL(out)
    vp, i64, c_int = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int
    lib.rh_set.argtypes = [c_int, c_int]
    lib.rh_sort.argtypes = [c_int, c_int, vp, vp, vp, vp, i64, c_int, c_int, ctypes.POINTER(c_int), ctypes.POINTER(c_int)]
    lib.rh_pass_u32.argtypes = [vp, vp, vp, vp, i64, c_int, c_int]
    lib.rh_digit_bits.argtypes = [c_int, ctypes.POINTER(c_int)]
    yield lib
    lib.rh_set(11, 1)


def _mix64(x):
    x = x ^ (x >> np.uint64(33))
    x = x * np.uint64(0xff51afd7ed558ccd)
    x = x ^ (x >> np.uint64(33))
    x = x * np.uint64(0xc4ceb9fe1a85ec53)
    return x ^ (x >> np.uint64(33))


def make_keys(dist, n, bits, lo, hi, seed):
    """`bits`-bit keys (numpy uint64) of one distribution; lo, hi: the sorted field."""
    rng = np.random.default_rng(seed)
    full = np.uint64((1 << bits) - 1)
    field = np.uint64(((1 << (hi - lo)) - 1) << lo) if hi > lo else np.uint64(0)
    u = rng.integers(0, 1 << 63, n, dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, n, dtype=np.uint64)
    if dist == "uniform":
        k = u
    elif dist == "equal":
        k = np.full(n, u[0] if n else 0, np.uint64)
    elif dist == "two":
        k = np.where(rng.integers(0, 2, n) == 1, u[0] if n else 0, u[1] if n > 1 else 0).astype(np.uint64)
    elif dist == "ones":                                  # every digit 0x7FF; the other bits vary
        k = u | field
    elif dist == "descending":                            # whole keys descending: every item moves
        k = np.sort(u & full)[::-1]
    elif dist == "outside":                               # the field is constant: the result is the input order
        k = (u & ~field) | (u[0] & field if n else np.uint64(0))
    elif dist == "skew":                                  # tools/radix_test.cu: skewed high part (cells), uniform low 24 bits (UMIs)
        x = _mix64(np.arange(n, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15) + np.uint64(seed))
        m = _mix64(x) % np.uint64(1000)
        k = (x & np.uint64(0xFFFFFF)) | ((m * m // np.uint64(10)) << np.uint64(24))
    else:
        raise ValueError(dist)
    return k & full


def digit(k, lo, hi):
    if hi <= lo:
        return np.zeros(len(k), np.uint8)
    d = (k >> np.uint64(lo)) & np.uint64((1 << (hi - lo)) - 1)
    return d.astype(np.uint16) if hi - lo <= 16 else d               # numpy sorts 16-bit keys by radix


def _dev(a, torch):
    if a.dtype == np.uint64:
        return torch.from_numpy(a.view(np.int64)).cuda()
    return torch.from_numpy(a.view(np.int32)).cuda()


def _host(t, dtype):
    return t.cpu().numpy().view(dtype)


def check_sort(rh, key_bits, n, lo, hi, dist, max_bits=11, chunk=1, values=True, seed=1):
    import torch
    rh.rh_set(max_bits, chunk)
    kt = np.uint64 if key_bits == 64 else np.uint32
    k = make_keys(dist, n, key_bits, lo, hi, seed + n + 131 * lo + hi).astype(kt)
    v = np.random.default_rng(seed).permutation(n).astype(np.uint32)
    ka, kb = _dev(k, torch), torch.full((n,), -1, dtype=torch.int64 if key_bits == 64 else torch.int32, device="cuda")
    va, vb = (_dev(v, torch), torch.full((n,), -1, dtype=torch.int32, device="cuda")) if values else (None, None)
    in_b, passes = ctypes.c_int(-1), ctypes.c_int(-1)
    ptr = lambda t: t.data_ptr() if t is not None else None
    torch.cuda.synchronize()
    rc = rh.rh_sort(key_bits // 8, 1 if values else 0, ptr(ka), ptr(va), ptr(kb), ptr(vb), n, lo, hi, ctypes.byref(in_b), ctypes.byref(passes))
    assert rc == 0, rc
    mb = min(11, max(1, max_bits))
    assert passes.value == (max(0, hi - lo) + mb - 1) // mb
    assert in_b.value == passes.value % 2
    order = np.argsort(digit(k.astype(np.uint64), lo, hi), kind="stable")
    got_k = _host(kb if in_b.value else ka, kt)
    what = (key_bits, n, lo, hi, dist, max_bits, chunk, values)
    assert np.array_equal(got_k, k[order]), what
    if values:
        assert np.array_equal(_host(vb if in_b.value else va, np.uint32), v[order]), what
    if dist == "outside":
        assert np.array_equal(order, np.arange(n))


SIZES = [0, 1, 2, 31, 32, 33, 767, 768, 769, 6143, 6144, 6145, 2 * TILE, 5 * TILE + 1, 1_000_003]


@pytest.mark.parametrize("n", SIZES)
def test_sizes(rh, n):
    check_sort(rh, 64, n, 18, 59, "skew")
    check_sort(rh, 64, n, 0, 64, "uniform", chunk=3, values=False)
    check_sort(rh, 32, n, 0, 32, "uniform", chunk=2)


U64_RANGES = [(0, 1), (0, 11), (0, 12), (0, 23), (3, 44), (18, 59), (21, 64), (32, 64), (53, 64), (63, 64), (0, 64), (40, 40)]


@pytest.mark.parametrize("lo,hi", U64_RANGES)
def test_u64_bit_ranges(rh, lo, hi):
    n = 5 * TILE + 1
    check_sort(rh, 64, n, lo, hi, "uniform")
    if hi - lo < 64:
        check_sort(rh, 64, n, lo, hi, "outside", values=False)
    check_sort(rh, 64, 769, lo, hi, "descending", chunk=2)


@pytest.mark.parametrize("lo,hi", [(0, 32), (21, 32), (31, 32)])
def test_u32_bit_ranges(rh, lo, hi):
    for dist in ("uniform", "outside", "descending", "two"):
        check_sort(rh, 32, 2 * TILE + 33, lo, hi, dist, values=dist != "two")


@pytest.mark.parametrize("max_bits", [1, 7, 10, 11])
@pytest.mark.parametrize("chunk", [1, 2, 3, 64])
def test_digit_width_and_chunk_settings(rh, max_bits, chunk):
    """max_bits 7 and 10 split 43 and 64 bits into digits of unequal width; 64 tiles per chunk puts the whole input
    into one CTA's chunk."""
    n = 2 * TILE + 7 if max_bits == 1 else 5 * TILE + 1
    check_sort(rh, 64, n, 21, 64, "uniform", max_bits, chunk)
    check_sort(rh, 64, n, 0, 64, "skew", max_bits, chunk, values=False)
    if max_bits >= 7:
        check_sort(rh, 64, 200_003, 0, 64, "ones", max_bits, chunk)


@pytest.mark.parametrize("max_bits", [1, 7, 10, 11, 12, 0])
def test_digit_split(rh, max_bits):
    """ceil(total / max_bits) passes whose widths differ by at most one, wider ones first, none over 11 bits."""
    rh.rh_set(max_bits, 1)
    mb = min(11, max(1, max_bits))
    bits = (ctypes.c_int * 64)()
    for total in range(0, 65):
        p = rh.rh_digit_bits(total, bits)
        w = list(bits[:p])
        assert p == (total + mb - 1) // mb and sum(w) == total
        assert all(1 <= x <= mb for x in w) and w == sorted(w, reverse=True) and (not w or w[0] - w[-1] <= 1), (total, w)


@pytest.mark.parametrize("dist", ["uniform", "equal", "two", "ones", "descending", "outside", "skew"])
def test_key_distributions(rh, dist):
    for lo, hi in ((0, 64), (3, 44), (53, 64)):
        if dist == "outside" and hi - lo == 64:
            continue
        check_sort(rh, 64, 2 * TILE + 5, lo, hi, dist, values=lo != 3)
    check_sort(rh, 64, 1_000_003, 21, 64, dist, chunk=2)


@pytest.mark.parametrize("block_sums", [1023, 1024, 1025])
def test_prefix_sum_around_1024_block_sums(rh, block_sums):
    """At 11-bit digits and one tile per chunk the counts matrix has 2048 x n_chunks entries, 8192 per block sum:
    4 chunks per block sum.  rdx_scan_kernel scans the block sums with one CTA of 1024 threads."""
    n = (4 * block_sums - 1) * TILE + 1                   # 4 * block_sums chunks, the last one holding one item
    check_sort(rh, 32, n, 0, 11, "uniform")
    check_sort(rh, 64, n, 53, 64, "uniform", values=False)


def test_rdx_pass_u32(rh):
    """One pass on the top bits of a 21-bit position with values (the prev[] placement of the single-cell sort)."""
    import torch
    rh.rh_set(11, 1)
    for n in (1, 6145, 1_000_003):
        rng = np.random.default_rng(n)
        k = rng.permutation(np.arange(n, dtype=np.uint32) * np.uint32(2) % np.uint32(1 << 21)).astype(np.uint32)
        v = rng.integers(0, 1 << 32, n, dtype=np.uint32)
        ki, vi = _dev(k, torch), _dev(v, torch)
        ko, vo = torch.full_like(ki, -1), torch.full_like(vi, -1)
        for shift, bits in ((10, 11), (0, 1), (20, 1), (31, 1)):
            assert rh.rh_pass_u32(ki.data_ptr(), vi.data_ptr(), ko.data_ptr(), vo.data_ptr(), n, shift, bits) == 0
            order = np.argsort(digit(k.astype(np.uint64), shift, shift + bits), kind="stable")
            assert np.array_equal(_host(ko, np.uint32), k[order]) and np.array_equal(_host(vo, np.uint32), v[order]), (n, shift, bits)
