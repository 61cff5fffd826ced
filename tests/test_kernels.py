"""Kernel-level tests: the look-back scan, the segmented radix sort, K5 selection, find_pairs and
K6 verification, each run alone through tests/kernels/kernel_harness.cu and compared with a plain
NumPy reference at the sizes, alignments and key widths where such kernels go wrong.  Every device
buffer of the harness sits between guard words; every call asserts that they are intact.

End to end: the radix sort's ballot ranking (the fallback for devices where shared-memory atomics
do not rank in lane order) against the oracle, and both branches of the selection retry."""
import ctypes as C
import importlib.util
import os

import numpy as np
import pytest

from conftest import PRM, ROOT
from test_gpu_parity import COUNTERS, assert_parity

gpu = pytest.mark.gpu

u8p = np.ctypeslib.ndpointer(dtype=np.uint8, flags="C_CONTIGUOUS")
u32p = np.ctypeslib.ndpointer(dtype=np.uint32, flags="C_CONTIGUOUS")
i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
u64p = np.ctypeslib.ndpointer(dtype=np.uint64, flags="C_CONTIGUOUS")
intp = C.POINTER(C.c_int)
ullp = C.POINTER(C.c_ulonglong)

WRAPPERS = ["kh_scan_temp_new", "kh_scan_temp_free", "kh_scan_temp_epoch", "kh_scan", "kh_sort_u32",
            "kh_sort_u64", "kh_select", "kh_find_pairs", "kh_verify"]

LB_TILE = 16384  # k_scan_lookback's tile (scan.cuh kLbTile); one k_scan_tiles block takes 4096
RS_TILE = 8192   # radix sort tile (radix_sort.cuh kRsTile); a warp's chunk is 512


def _build():
    spec = importlib.util.spec_from_file_location(
        "gds_build", os.path.join(ROOT, "genome-downsampler_b200", "build.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    return b.build_kernel_harness()  # rebuilds when a source is newer than the .so


class Harness:
    def __init__(self, path):
        L = C.CDLL(path)
        L.kh_scan_temp_new.restype = C.c_void_p
        L.kh_scan_temp_free.argtypes = [C.c_void_p]
        L.kh_scan_temp_free.restype = None
        L.kh_scan_temp_epoch.argtypes = [C.c_void_p]
        L.kh_scan_temp_epoch.restype = C.c_uint32
        L.kh_scan.argtypes = [C.c_void_p, u32p, u32p, C.c_int, C.c_uint64, C.c_uint32, C.c_uint32,
                              C.c_int, C.c_longlong, intp]
        L.kh_sort_u32.argtypes = [u32p, u64p, C.c_uint32, C.c_int, C.c_int, u32p, u32p, intp, intp]
        L.kh_sort_u64.argtypes = [u64p, u64p, C.c_uint32, C.c_int, C.c_int, u64p, u32p, intp, intp]
        L.kh_select.argtypes = [u32p, u32p, C.c_uint32, u32p, C.c_uint64, C.c_uint64, u32p, ullp, intp]
        L.kh_find_pairs.argtypes = [u32p, C.c_uint64, intp]
        L.kh_verify.argtypes = [u32p, u32p, u32p, C.c_uint64, u64p, u32p, C.c_uint32, i32p, u32p,
                                C.c_uint32, ullp, intp]
        for name in WRAPPERS[3:]:
            getattr(L, name).restype = C.c_int
        self.L = L

    @staticmethod
    def _check(rc, intact, what):
        if rc != 0:
            raise RuntimeError("%s: CUDA error %d" % (what, rc))
        assert intact.value == 1, "%s wrote outside its buffers (a guard word changed)" % what

    def scan(self, tmp, arrays, in_off=0, out_off=0, in_place=False, epoch=-1):
        a = np.ascontiguousarray(np.stack(arrays), np.uint32)
        out = np.zeros_like(a)
        ok = C.c_int(0)
        rc = self.L.kh_scan(tmp, a.reshape(-1), out.reshape(-1), len(arrays), a.shape[1], in_off,
                            out_off, int(in_place), epoch, C.byref(ok))
        self._check(rc, ok, "exclusive_scan_u32_multi")
        return out

    def sort(self, keys, group_sizes, bits, atomic):
        u64 = keys.dtype == np.uint64
        keys = np.ascontiguousarray(keys)
        ko = np.zeros_like(keys)
        vo = np.zeros(len(keys), np.uint32)
        gs = np.ascontiguousarray(group_sizes, np.uint64)
        passes, ok = C.c_int(0), C.c_int(0)
        fn = self.L.kh_sort_u64 if u64 else self.L.kh_sort_u32
        rc = fn(keys, gs, len(gs), bits, int(atomic), ko, vo, C.byref(passes), C.byref(ok))
        self._check(rc, ok, "radix_sort_pairs")
        return ko, vo, passes.value

    def select(self, b_first, flow, sorted_idx, n):
        n_words = (n + 31) // 32
        bm = np.zeros(max(n_words, 1), np.uint32)
        kept, ok = C.c_ulonglong(0), C.c_int(0)
        rc = self.L.kh_select(np.ascontiguousarray(b_first, np.uint32),
                              np.ascontiguousarray(flow, np.uint32), len(flow),
                              np.ascontiguousarray(sorted_idx, np.uint32), len(sorted_idx), n_words,
                              bm, C.byref(kept), C.byref(ok))
        self._check(rc, ok, "k_select")
        return bm[:n_words], kept.value

    def find_pairs(self, bitmap):
        bm = np.array(bitmap, np.uint32)
        ok = C.c_int(0)
        rc = self.L.kh_find_pairs(bm if len(bm) else np.zeros(1, np.uint32), len(bm), C.byref(ok))
        self._check(rc, ok, "k_find_pairs")
        return bm

    def verify(self, bitmap, s, e, read_off, ref_lens, diff_in, excl_in, M):
        viol, ok = C.c_ulonglong(0), C.c_int(0)
        rc = self.L.kh_verify(np.ascontiguousarray(bitmap, np.uint32), s, e, len(s),
                              np.ascontiguousarray(read_off, np.uint64),
                              np.ascontiguousarray(ref_lens, np.uint32), len(ref_lens), diff_in,
                              excl_in, M, C.byref(viol), C.byref(ok))
        self._check(rc, ok, "K6 verification")
        return viol.value


@pytest.fixture(scope="module")
def kh():
    return Harness(_build())


@pytest.fixture
def scan_temp(kh):
    t = kh.L.kh_scan_temp_new()
    yield t
    kh.L.kh_scan_temp_free(t)


def test_harness_builds_and_exports_every_wrapper():
    # no GPU needed: nvcc cross-compiles the production headers into the harness
    L = C.CDLL(_build())
    for name in WRAPPERS:
        assert hasattr(L, name), name


# ------------------------------------------------------------------------------------ scan
def excl_scan_ref(x):
    """exclusive prefix sum mod 2^32 (64-bit cumsum, reduced)"""
    x = np.asarray(x).view(np.uint32).astype(np.uint64)
    c = np.cumsum(x, dtype=np.uint64) & np.uint64(0xffffffff)
    return np.concatenate([np.zeros(1, np.uint64), c[:-1]])[:len(x)].astype(np.uint32)


def scan_inputs(rng, n, n_arr):
    """different contents per array: wrapping u32 values, int32 differences, small counts"""
    kinds = [lambda: rng.integers(0, 1 << 32, size=n, dtype=np.uint64).astype(np.uint32),
             lambda: rng.integers(-(1 << 20), 1 << 20, size=n).astype(np.int32).view(np.uint32),
             lambda: rng.integers(0, 9, size=n).astype(np.uint32)]
    return [kinds[k % 3]() for k in range(n_arr)]


SCAN_SIZES = [0, 1, 4095, 4096, 4097, LB_TILE - 1, LB_TILE, LB_TILE + 1, 3 * LB_TILE - 1,
              3 * LB_TILE + 1, 64 * LB_TILE - 1, 64 * LB_TILE + 1]


@gpu
@pytest.mark.parametrize("n", SCAN_SIZES)
@pytest.mark.parametrize("n_arr", [1, 2, 3])
def test_scan_sizes_and_arrays(kh, scan_temp, n, n_arr):
    rng = np.random.default_rng(n * 3 + n_arr)
    arrs = scan_inputs(rng, n, n_arr)
    out = kh.scan(scan_temp, arrs)
    for k in range(n_arr):
        assert np.array_equal(out[k], excl_scan_ref(arrs[k])), "array %d" % k


@gpu
@pytest.mark.parametrize("n,n_arr", [(40_000_003, 1), (3_000_017, 3)])
def test_scan_thousands_of_tiles(kh, scan_temp, n, n_arr):
    rng = np.random.default_rng(n)
    arrs = scan_inputs(rng, n, n_arr)
    out = kh.scan(scan_temp, arrs)
    for k in range(n_arr):
        assert np.array_equal(out[k], excl_scan_ref(arrs[k])), "array %d" % k


@gpu
@pytest.mark.parametrize("in_off,out_off", [(1, 0), (0, 1), (2, 0), (0, 3), (3, 3), (1, 2)])
@pytest.mark.parametrize("n", [4097, 5 * LB_TILE + 7, 40 * LB_TILE])
def test_scan_misaligned_arrays(kh, scan_temp, in_off, out_off, n):
    # pointers off 16-byte alignment take the scalar load/store path for whole tiles
    rng = np.random.default_rng(n + 10 * in_off + out_off)
    for n_arr in (1, 3):
        arrs = scan_inputs(rng, n, n_arr)
        out = kh.scan(scan_temp, arrs, in_off=in_off, out_off=out_off)
        for k in range(n_arr):
            assert np.array_equal(out[k], excl_scan_ref(arrs[k])), (n_arr, k)


@gpu
@pytest.mark.parametrize("off", [0, 1, 3])
@pytest.mark.parametrize("n", [4096, LB_TILE + 1, 100_003])
def test_scan_in_place(kh, scan_temp, off, n):
    rng = np.random.default_rng(n + off)
    for n_arr in (1, 2, 3):
        arrs = scan_inputs(rng, n, n_arr)
        out = kh.scan(scan_temp, arrs, in_off=off, out_off=off, in_place=True)
        for k in range(n_arr):
            assert np.array_equal(out[k], excl_scan_ref(arrs[k])), (n_arr, k)


@gpu
def test_scan_status_words_across_calls_and_epoch_reset(kh, scan_temp):
    # one ScanTemp: the status words of earlier, larger launches stay behind (stale epochs), and the
    # epoch wraps after 2^30 - 1 launches (the status array is cleared and the count restarts)
    rng = np.random.default_rng(99)
    for n, n_arr in ((60 * LB_TILE + 5, 2), (3 * LB_TILE + 1, 3), (40 * LB_TILE - 3, 1),
                     (20 * LB_TILE, 3), (LB_TILE + 1, 1)):
        arrs = scan_inputs(rng, n, n_arr)
        out = kh.scan(scan_temp, arrs)
        for k in range(n_arr):
            assert np.array_equal(out[k], excl_scan_ref(arrs[k])), (n, k)
    epochs = []
    for i in range(5):
        n, n_arr = (30 * LB_TILE + 11 * i, 1 + i % 3)
        arrs = scan_inputs(rng, n, n_arr)
        out = kh.scan(scan_temp, arrs, epoch=(1 << 30) - 3 if i == 0 else -1)
        epochs.append(kh.L.kh_scan_temp_epoch(scan_temp))
        for k in range(n_arr):
            assert np.array_equal(out[k], excl_scan_ref(arrs[k])), (i, k)
    assert epochs == [(1 << 30) - 2, (1 << 30) - 1, 1, 2, 3]


# ------------------------------------------------------------------------------ radix sort
def sort_ref(keys, group_sizes, bits):
    """stable order by (group, key mod 2^bits, index)"""
    n = len(keys)
    group = np.repeat(np.arange(len(group_sizes)), np.asarray(group_sizes, np.int64))
    k = np.asarray(keys, np.uint64)
    if bits < 64:
        k = k & np.uint64((1 << bits) - 1)
    order = np.lexsort((np.arange(n), k, group))
    return keys[order], order.astype(np.uint32)


KEY_SHAPES = ["uniform", "equal", "seven", "sorted", "reversed", "top_digit"]


def make_keys(rng, n, bits, dtype, shape):
    """keys below 2^bits (the sort's contract)"""
    hi = 1 << bits

    def uni(size):
        return rng.integers(0, hi, size=size, dtype=np.uint64)

    if shape == "uniform":
        k = uni(n)
    elif shape == "equal":
        k = np.full(n, uni(1)[0], np.uint64)
    elif shape == "seven":
        k = rng.choice(uni(7), size=n)
    elif shape == "sorted":
        k = np.sort(uni(n))
    elif shape == "reversed":
        k = np.sort(uni(n))[::-1].copy()
    else:  # only the last pass's digit varies
        shift = 8 * (max(1, (bits + 7) // 8) - 1)
        low = uni(1)[0] & np.uint64((1 << shift) - 1)
        k = (rng.integers(0, hi >> shift, size=n, dtype=np.uint64) << np.uint64(shift)) | low
    return k.astype(dtype)


KEY_WIDTHS = [(np.uint32, b) for b in (0, 1, 5, 8, 9, 15, 16, 17, 24, 32)] + \
             [(np.uint64, b) for b in (33, 40, 52)]
RANKS = [pytest.param(True, id="atomic"), pytest.param(False, id="ballot")]


def check_sort(kh, keys, group_sizes, bits, atomic):
    ko, vo, passes = kh.sort(keys, group_sizes, bits, atomic)
    rk, rv = sort_ref(keys, group_sizes, bits)
    assert passes == max(1, (bits + 7) // 8)
    assert np.array_equal(vo, rv), "values (source indices) differ"
    assert np.array_equal(ko, rk), "keys differ"


@gpu
@pytest.mark.parametrize("atomic", RANKS)
@pytest.mark.parametrize("dtype,bits", KEY_WIDTHS, ids=lambda x: str(getattr(x, "__name__", x)))
@pytest.mark.parametrize("n", [511, 512, 513, RS_TILE - 1, RS_TILE, RS_TILE + 1])
def test_radix_sort_one_group(kh, atomic, dtype, bits, n):
    rng = np.random.default_rng(bits * 100_003 + n)
    for shape in KEY_SHAPES:
        check_sort(kh, make_keys(rng, n, bits, dtype, shape), [n], bits, atomic)


@gpu
@pytest.mark.parametrize("atomic", RANKS)
@pytest.mark.parametrize("dtype,bits,n", [(np.uint32, 24, 3_000_000), (np.uint32, 32, 2_999_999),
                                          (np.uint64, 40, 2_000_001)],
                         ids=lambda x: str(getattr(x, "__name__", x)))
def test_radix_sort_millions(kh, atomic, dtype, bits, n):
    rng = np.random.default_rng(n)
    for shape in ("uniform", "seven"):
        check_sort(kh, make_keys(rng, n, bits, dtype, shape), [n], bits, atomic)


SEGMENT_MAPS = [[0, 1, 8191, 8192, 8193, 0],
                [8193, 0, 0, 1, 8192, 8191, 20_000],
                [1, 1, 1, 0, 8192],
                [0, 0],  # no items at all
                [5000] * 3 + [0] + [RS_TILE * 3 + 17]]


@gpu
@pytest.mark.parametrize("atomic", RANKS)
@pytest.mark.parametrize("dtype,bits", [(np.uint32, 1), (np.uint32, 9), (np.uint32, 17),
                                        (np.uint32, 32), (np.uint64, 40)],
                         ids=lambda x: str(getattr(x, "__name__", x)))
@pytest.mark.parametrize("groups", range(len(SEGMENT_MAPS)))
def test_radix_sort_segmented(kh, atomic, dtype, bits, groups):
    sizes = SEGMENT_MAPS[groups]
    n = sum(sizes)
    rng = np.random.default_rng(1000 * groups + bits)
    for shape in ("uniform", "seven", "reversed"):
        check_sort(kh, make_keys(rng, n, bits, dtype, shape), sizes, bits, atomic)


# ---------------------------------------------------------------------------- K5, find_pairs
def make_bundles(rng, n, sizes, share=0.05):
    """Bundles over reads 0..n-1: each read in one bundle, a `share` of them in a second one too (a
    read cut at a segment boundary).  Returns b_first, mult, sorted_idx."""
    perm = rng.permutation(n).astype(np.uint32)
    slices, pos = [], 0
    for sz in sizes:
        slices.append(list(perm[pos:pos + sz]))
        pos += sz
    assert pos == n
    for r in rng.choice(n, size=int(share * n), replace=False):
        slices[int(rng.integers(0, len(slices)))].append(np.uint32(r))
    mult = np.array([len(x) for x in slices], np.uint32)
    b_first = np.concatenate([[0], np.cumsum(mult)[:-1]]).astype(np.uint32)
    return b_first, mult, np.concatenate([np.array(x, np.uint32) for x in slices])


def select_ref(b_first, flow, sorted_idx, n):
    mask = np.zeros(n, bool)
    for f0, f in zip(b_first, flow):
        mask[sorted_idx[f0:f0 + f]] = True
    return np.packbits(mask, bitorder="little").view(np.uint8), int(mask.sum())


def check_select(kh, b_first, flow, sorted_idx, n):
    bm, kept = kh.select(b_first, flow, sorted_idx, n)
    ref, nref = select_ref(b_first, flow, sorted_idx, n)
    nw = (n + 31) // 32
    want = np.zeros(nw * 4, np.uint8)
    want[:len(ref)] = ref
    assert np.array_equal(bm, want.view(np.uint32)), "kept bitmap differs"
    assert kept == nref, "n_kept must count every read once"


@gpu
@pytest.mark.parametrize("n", [45, 10_007, 200_003])
def test_select_flows_and_shared_reads(kh, n):
    rng = np.random.default_rng(n)
    # bundle sizes: mostly small, some at the 64-read boundary of the warp-wide branch, some large
    sizes = []
    left = n
    while left:
        sz = int(rng.choice([1, 2, 5, 9, 64, 65, 66, 300, 777], p=[.2, .2, .2, .15, .06, .06, .05, .05, .03]))
        sz = min(sz, left)
        sizes.append(sz)
        left -= sz
    b_first, mult, sidx = make_bundles(rng, n, sizes)
    B = len(mult)
    # flows: 0, 1, 64, 65, everything, or a random share
    pick = rng.integers(0, 6, size=B)
    flow = np.where(pick == 0, 0, np.where(pick == 1, 1, np.where(pick == 2, 64, np.where(
        pick == 3, 65, np.where(pick == 4, mult, rng.integers(0, mult + 1))))))
    flow = np.minimum(flow, mult).astype(np.uint32)
    if n > 1000:
        assert (flow > 64).sum() > 10 and (flow == 64).any() and (flow == 0).any()
    check_select(kh, b_first, flow, sidx, n)
    # every read of every bundle chosen: each read counted once although many appear twice
    check_select(kh, b_first, mult, sidx, n)
    # one warp of 32 bundles, all wide, every one of them sharing reads with the others
    k = np.arange(32 * 100, dtype=np.uint32) % 500
    check_select(kh, np.arange(32, dtype=np.uint32) * 100, np.full(32, 100, np.uint32), k, 500)


@gpu
@pytest.mark.parametrize("n_words", [0, 1, 255, 256, 257, 100_001])
def test_find_pairs(kh, n_words):
    rng = np.random.default_rng(n_words)
    x = rng.integers(0, 1 << 32, size=n_words, dtype=np.uint64).astype(np.uint32)
    x[::7] = 0
    x[1::7] = 0xffffffff
    x[2::7] &= 0x55555555
    x[3::7] &= 0xaaaaaaaa
    got = kh.find_pairs(x)
    any_ = (x & 0x55555555) | ((x >> 1) & 0x55555555)
    assert np.array_equal(got, (any_ | (any_ << 1)).astype(np.uint32))


# ------------------------------------------------------------------------------------- K6
def node_diff(s, e, read_off, ref_lens, mask=None):
    """int64 difference array over the batch's nodes (sample k owns ref_len[k] + 1 nodes); a
    zero-length read (end == start - 1, 32-bit) adds and removes at the same node"""
    base = np.concatenate([[0], np.cumsum(np.asarray(ref_lens, np.int64) + 1)])
    k = np.repeat(np.arange(len(ref_lens)), np.diff(np.asarray(read_off, np.int64)))
    if mask is not None:
        s, e, k = s[mask], e[mask], k[mask]
    d = np.zeros(base[-1] + 1, np.int64)
    np.add.at(d, base[k] + s.astype(np.int64), 1)
    np.add.at(d, base[k] + (e + np.uint32(1)).astype(np.int64), -1)
    return d


def violations_ref(s, e, read_off, ref_lens, mask, M):
    n_nodes = int(np.sum(np.asarray(ref_lens, np.int64) + 1))
    cin = np.cumsum(node_diff(s, e, read_off, ref_lens))[:n_nodes]
    cout = np.cumsum(node_diff(s, e, read_off, ref_lens, mask))[:n_nodes]
    return int(np.count_nonzero(np.minimum(cout, M) != np.minimum(cin, M)))


@pytest.fixture(scope="module")
def k6_input(O):
    # three samples, one of them tiny, with zero-length reads (one at start 0: end wraps to 2^32-1);
    # n is not a multiple of 32
    rng = np.random.default_rng(61)
    ref_lens = [40_000, 7, 90_000]
    ss, ee, off = [], [], [0]
    for k, (L, pairs) in enumerate(zip(ref_lens, (60_000, 11, 130_001))):
        if L > 150:
            s, e, _, _ = O.gen_reads(610 + k, pairs, L, 150)
            s, e = s.copy(), e.copy()
        else:
            s = rng.integers(0, L, size=2 * pairs).astype(np.uint32)
            e = np.minimum(s + rng.integers(0, 3, size=len(s)), L - 1).astype(np.uint32)
        z = rng.choice(len(s), size=max(1, len(s) // 50), replace=False)
        e[z] = s[z] - np.uint32(1)
        s[z[0]] = 0
        e[z[0]] = np.uint32(0xffffffff)
        ss.append(s); ee.append(e); off.append(off[-1] + len(s))
    s = np.concatenate(ss); e = np.concatenate(ee)
    s, e, off = s[:-3].copy(), e[:-3].copy(), off[:-1] + [off[-1] - 3]
    assert len(s) % 32 != 0
    off = np.array(off, np.uint64)
    d = node_diff(s, e, off, ref_lens)
    diff_in = d.astype(np.int32)
    excl_in = excl_scan_ref(diff_in)
    return s, e, off, ref_lens, diff_in, excl_in


def pack(mask):
    nw = (len(mask) + 31) // 32
    b = np.zeros(nw * 4, np.uint8)
    p = np.packbits(mask, bitorder="little")
    b[:len(p)] = p
    return b.view(np.uint32).copy()


@gpu
@pytest.mark.parametrize("M", [1, 30, 10_000])
def test_verification_counts_violations(kh, O, k6_input, M):
    s, e, off, ref_lens, diff_in, excl_in = k6_input
    n = len(s)
    rng = np.random.default_rng(M)
    bm, _ = O.sync_solve(s, e, ref_lens, off, M, params=PRM)
    valid = O.bitmap_to_mask(bm, n).astype(bool)

    def check(mask, bitmap=None, expect_zero=False):
        want = violations_ref(s, e, off, ref_lens, mask, M)
        got = kh.verify(pack(mask) if bitmap is None else bitmap, s, e, off, ref_lens, diff_in,
                        excl_in, M)
        assert got == want
        assert (want == 0) == expect_zero
        return got

    check(valid, expect_zero=True)
    kept = np.flatnonzero(valid & (e >= s))
    # drop one kept read that some position needs
    for i in rng.permutation(kept)[:200]:
        m = valid.copy()
        m[i] = False
        if violations_ref(s, e, off, ref_lens, m, M):
            check(m)
            break
    else:
        assert M == 10_000 and len(kept) == np.count_nonzero(e >= s)  # then every read is needed
    # drop many
    m = valid.copy()
    m[rng.choice(kept, size=len(kept) // 10, replace=False)] = False
    check(m)
    # add reads: more than M never changes min(cov, M) where the answer was valid
    m = valid.copy()
    m[rng.choice(n, size=n // 3, replace=False)] = True
    check(m, expect_zero=True)
    # stray bits past n in the last word are not reads
    b = pack(valid)
    b[-1] |= np.uint32(0xffffffff) << np.uint32(n % 32)
    check(valid, bitmap=b, expect_zero=True)
    # nothing kept
    check(np.zeros(n, bool), expect_zero=not np.any(e >= s))


# -------------------------------------------------------------- ballot ranking end to end
@pytest.fixture(scope="module")
def ballot_solver(pkg):
    # gds_create reads GDS_RANK once: this context sorts with the ballot ranking throughout
    old = os.environ.get("GDS_RANK")
    os.environ["GDS_RANK"] = "ballot"
    try:
        s = pkg.Solver(0)
    finally:
        if old is None:
            del os.environ["GDS_RANK"]
        else:
            os.environ["GDS_RANK"] = old
    yield s
    s.close()


def assert_ballot_matches(O, solver, ballot_solver, s, e, Ls, off, M, prm, len_hint=None):
    kw = dict(read_off=off, params=prm, verify=True, want_vectors=True, len_hint=len_hint)
    rb = ballot_solver.solve(s, e, Ls, M, **kw)
    ra = solver.solve(s, e, Ls, M, **kw)
    assert rb.sort_passes > 0 or len(s) == 0, "not on the radix-sort path"
    for key in COUNTERS + ("key_bits", "sort_passes", "n_arc_items", "verify_violations"):
        assert rb[key] == ra[key], key
    assert np.array_equal(rb.kept_bitmap, ra.kept_bitmap)
    assert_parity(O, rb, s, e, Ls, off, M, prm[:5])
    return rb


@gpu
def test_ballot_rank_ragged_batches(solver, ballot_solver, O):
    rng = np.random.default_rng(71)
    for it in range(36):
        ns = int(rng.integers(1, 6))
        Ls = rng.integers(1, 400, size=ns).astype(np.uint32)
        ss, ee, off = [], [], [0]
        for L in Ls:
            n = 2 * int(rng.integers(0, 300))
            mode = int(rng.integers(0, 3))
            if mode == 0:
                s = rng.integers(0, L, size=n); ln = rng.integers(1, max(2, L // 2 + 1), size=n)
            elif mode == 1:
                s = rng.integers(0, max(1, L // 3), size=n); ln = rng.integers(1, 6, size=n)
            else:
                s = rng.integers(0, L, size=n); ln = np.full(n, rng.integers(1, 30))
            e = np.minimum(s + ln - 1, L - 1)
            ss.append(s); ee.append(e); off.append(off[-1] + n)
        s = np.concatenate(ss).astype(np.uint32); e = np.concatenate(ee).astype(np.uint32)
        M = int(rng.integers(1, 12))
        seg = int(rng.integers(1, 120)) if it % 3 == 0 else 0  # short segments every third case
        prm = (int(rng.integers(1, 100)), int(rng.integers(0, 300)), int(rng.integers(0, 5)), 0, seg, 1)
        assert_ballot_matches(O, solver, ballot_solver, s, e, Ls, np.array(off, np.uint64), M, prm)


@gpu
def test_ballot_rank_64bit_keys(solver, ballot_solver, O):
    rng = np.random.default_rng(5)
    L, n = 2_000_000, 40_000
    s = rng.integers(0, L - 1_000_001, size=n).astype(np.uint32)
    e = (s + rng.integers(1, 1_000_000, size=n) - 1).astype(np.uint32)
    r = assert_ballot_matches(O, solver, ballot_solver, s, e, [L], np.array([0, n], np.uint64), 7,
                              PRM + (0, 1))
    assert r.key_bits > 32


@gpu
def test_ballot_rank_zero_length_reads(solver, ballot_solver, O):
    rng = np.random.default_rng(29)
    s, e, _, _ = O.gen_reads(77, 40_000, 9_000, 150)
    s, e = s.copy(), e.copy()
    idx = rng.choice(len(s), size=600, replace=False)
    e[idx] = s[idx] - np.uint32(1)
    s[idx[0]] = 0
    e[idx[0]] = np.uint32(0xffffffff)
    off = np.array([0, len(s)], np.uint64)
    for prm in (PRM + (0, 1), (64, 150, 1, 0, 2048, 1)):
        r = assert_ballot_matches(O, solver, ballot_solver, s, e, [9_000], off, 30, prm)
        assert not O.bitmap_to_mask(r.kept_bitmap, len(s))[idx].any()


@gpu
def test_ballot_rank_several_read_lengths(solver, ballot_solver, O):
    # more than one read length: the in-CSR order comes from a second sort, of the bundles
    rng = np.random.default_rng(11)
    parts = []
    for k, L in enumerate((9_200, 30_000)):
        s = rng.integers(0, L - 200, size=200_000 + 2 * k).astype(np.uint32)
        parts.append((s, (s + rng.integers(120, 180, size=len(s))).astype(np.uint32)))
    s = np.concatenate([p[0] for p in parts]); e = np.concatenate([p[1] for p in parts])
    off = np.array([0, len(parts[0][0]), len(s)], np.uint64)
    assert_ballot_matches(O, solver, ballot_solver, s, e, [9_200, 30_000], off, 200, PRM + (0, 1))


# ------------------------------------------------------------------ selection retry
def _retry_then_unhinted(pkg, O, s, e, L, M, prm, len_hint):
    """The call on a fresh context (empty candidate buffer), profiled; then the same call again, and
    once more without the length hints (k_validate finds the bounds, then the same selection).  All
    must match the oracle."""
    fresh = pkg.Solver(0)
    try:
        fresh.kernel_profile_reset()
        r = fresh.solve(s, e, L, M, params=prm, verify=True, want_vectors=True, len_hint=len_hint,
                        profile=True)
        prof = {k["name"]: k["launches"] for k in fresh.kernel_profile()}
        again = fresh.solve(s, e, L, M, params=prm, verify=True, len_hint=len_hint)
        unhinted = fresh.solve(s, e, L, M, params=prm, verify=True, want_vectors=True)
    finally:
        fresh.close()
    off = np.array([0, len(s)], np.uint64)
    assert_parity(O, r, s, e, [L], off, M, prm[:5])
    assert_parity(O, unhinted, s, e, [L], off, M, prm[:5])
    for key in COUNTERS:
        assert r[key] == unhinted[key] == again[key], key
    assert np.array_equal(r.kept_bitmap, unhinted.kept_bitmap)
    assert np.array_equal(r.kept_bitmap, again.kept_bitmap)
    return r, again, unhinted, prof


@gpu
def test_selection_retry_grows_the_candidate_buffer(pkg, O):
    # config 4's density (10 reads per start, one length, M = 500: coverage 1500) on a segmented
    # reference: the global histogram path.  Most reads sit in partial bundles, more than the N/8
    # candidate slots a fresh context starts with: the first selection overflows and is repeated.
    L, M = 200_000, 500
    s, e, _, _ = O.gen_reads(4040, 1_000_000, L, 150)
    r, again, unhinted, prof = _retry_then_unhinted(pkg, O, s, e, L, M, (64, 150, 1, 0, 8192, 0),
                                                    (150, 150))
    assert r.bundle_path == 2 and unhinted.bundle_path == 2
    assert r.partial_candidates > r.n_filtered // 8
    assert prof["direct_classify"] == 2, prof  # the selection ran twice
    # the buffer has grown: the same call on the same context selects once
    assert again.kernel_launches < r.kernel_launches


@gpu
def test_selection_ranks_a_partial_bundle_beyond_2048_reads(pkg, O):
    # 5000 identical reads, M = 17: one partial bundle of 5000 candidates on the shared-memory
    # histogram path, ranked by one warp's bisection.  Its candidates overflow the N/8 slots of a
    # fresh context, so the selection runs twice.
    s = np.full(5000, 10, np.uint32)
    e = np.full(5000, 60, np.uint32)
    r, again, unhinted, prof = _retry_then_unhinted(pkg, O, s, e, 100, 17, PRM + (0, 0), (51, 51))
    assert r.bundle_path == 1 and r.n_bundles == 1
    assert r.partial_bundles == 1 and r.partial_candidates == 5000
    assert prof.get("direct_classify") == 2 and prof.get("direct_partial") == 2, prof
    assert "direct_walk" not in prof and "direct_quota" not in prof, prof
    assert pkg.Solver.bitmap_to_indices(r.kept_bitmap, 5000).tolist() == list(range(17))
