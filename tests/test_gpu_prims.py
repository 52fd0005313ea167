"""The device-wide primitives of csrc/rt_prims.cuh called directly through their self-test entries, against numpy, bit for
bit: the exclusive scan (adaptive pixel list, 4-wide BVH compaction, JPEG bit offsets) at every tile and recursion boundary
up to the 8K pixel count, in place and out of place, and the stable LSD radix sort (LBVH Morton order) at every pass count,
with stability, odd pass counts and key bits above the sorted ones.  Every call also reports whether a guard byte around
any output, ping-pong or scratch buffer changed, which checks the scratch sizing helpers the library's callers use."""
import ctypes as C

import numpy as np
import pytest

import raytracing_renderer_cuda_b200 as rt
from raytracing_renderer_cuda_b200 import capi

pytestmark = pytest.mark.gpu

TILE = 2048  # prims::kTile: one CTA scans / sorts one tile; the tile totals are scanned recursively above TILE tiles
SCAN_SIZES = (1, 2, 31, 32, 33, 255, 256, 257, 2047, 2048, 2049, 4095, 4096, 4097, TILE * TILE - 1, TILE * TILE, TILE * TILE + 1,
              2 * TILE * TILE + 3)
PIXELS_8K = 7680 * 4320  # the adaptive pass's pixel list at 8K: the only caller that reaches the second recursion level
SORT_SIZES = (1, 2, 255, 2047, 2048, 2049, 4097, TILE * 9 + 1, 1_000_003, TILE * TILE + 1)  # TILE*9+1: 10 tiles, so the
# digit-major histogram table (256 x tiles) the sort scans is itself more than one tile


@pytest.fixture(scope="module")
def ctx():
    return rt.Context(0)


def _exclusive(a: np.ndarray) -> np.ndarray:
    """exclusive prefix sum in a's own unsigned dtype (numpy's cumsum wraps around like the kernel's integer adds)"""
    out = np.zeros_like(a)
    np.cumsum(a[:-1], dtype=a.dtype, out=out[1:])
    return out


def _scan_inputs(n: int, dtype, rng):
    yield "flags", rng.integers(0, 2, n, dtype=np.uint8).astype(dtype)  # the adaptive pass's keep flags
    if dtype == np.uint32:
        yield "wrapping", rng.integers(0, 2**32, n, dtype=np.uint64).astype(np.uint32) | np.uint32(1 << 31)
    else:
        yield "past 2^32", rng.integers(0, 2**36, n, dtype=np.uint64)  # JPEG bit offsets of a large frame
        yield "wrapping", rng.integers(0, 2**64, n, dtype=np.uint64, endpoint=False) | np.uint64(1 << 63)
    yield "zeros", np.zeros(n, dtype)
    yield "ones", np.ones(n, dtype)


def _check_scan(ctx, n, dtype, seed):
    rng = np.random.default_rng(seed)
    for name, a in _scan_inputs(n, dtype, rng):
        want = _exclusive(a)
        if name == "wrapping" and n > 1:
            assert np.sum(a, dtype=np.float64) > float(np.iinfo(dtype).max)  # the total really wraps
        for in_place in (False, True):
            got, overrun = rt.capi.selftest_exclusive_sum(ctx, a, in_place=in_place)
            assert not overrun, (n, name, in_place)
            assert got.dtype == dtype and np.array_equal(got, want), (n, name, in_place, int(np.argmax(got != want)))


@pytest.mark.parametrize("n", SCAN_SIZES + (PIXELS_8K,))
def test_exclusive_sum_u32(ctx, n):
    _check_scan(ctx, n, np.uint32, seed=n)


@pytest.mark.parametrize("n", SCAN_SIZES)
def test_exclusive_sum_u64(ctx, n):
    _check_scan(ctx, n, np.uint64, seed=n + 1)


def test_exclusive_sum_of_nothing_writes_nothing(ctx):
    lib = ctx.lib
    for eb, dtype in ((4, np.uint32), (8, np.uint64)):
        src = np.arange(5, dtype=dtype)
        out = np.full(5, 7, dtype)
        overrun = C.c_int32(-1)
        for in_place in (0, 1):
            assert lib.rt_selftest_exclusive_sum(ctx._h, src.ctypes.data, out.ctypes.data, 0, eb, in_place, C.byref(overrun)) == capi.RT_OK
            assert overrun.value == 0 and np.array_equal(out, np.full(5, 7, dtype))
        assert lib.rt_selftest_exclusive_sum(ctx._h, None, None, 0, eb, 0, C.byref(overrun)) == capi.RT_OK


def _interleave3(x, y, z) -> np.ndarray:
    """63-bit Morton code of three 21-bit coordinates (bit 3i + 2 of x, 3i + 1 of y, 3i of z)"""
    code = np.zeros(x.size, np.uint64)
    for b in range(21):
        for c, s in ((x, 2), (y, 1), (z, 0)):
            code |= ((c >> np.uint64(b)) & np.uint64(1)) << np.uint64(3 * b + s)
    return code


def _sort_keys(n: int, rng) -> dict:
    """name -> 64-bit keys"""
    cell = rng.integers(0, 24, (3, n), dtype=np.uint64) * np.uint64(87_381)  # 24 positions per axis: many equal codes
    return {"random": rng.integers(0, 2**64, n, dtype=np.uint64, endpoint=False), "morton": _interleave3(*cell),
            "equal": np.full(n, 0xDEADBEEF_01234567, np.uint64), "reversed": np.arange(n, dtype=np.uint64)[::-1] * np.uint64(0x1_0000_0001)}


def _keys_above(n: int, passes: int, rng) -> np.ndarray:
    """keys equal in the sorted bits [0, 8 * passes) and different above them"""
    high = rng.integers(0, 2 ** (64 - 8 * passes), n, dtype=np.uint64, endpoint=False)
    return (high << np.uint64(8 * passes)) | np.uint64(0xA5A5A5A5_A5A5A5A5 & ((1 << (8 * passes)) - 1))


def _stable_order(keys: np.ndarray, passes: int) -> np.ndarray:
    masked = keys & np.uint64((1 << (8 * passes)) - 1) if passes < 8 else keys
    if passes <= 2:
        masked = masked.astype(np.uint8 if passes == 1 else np.uint16)  # (numpy's stable sort of small integers is a radix sort)
    return np.argsort(masked, kind="stable")


@pytest.mark.parametrize("n", SORT_SIZES)
def test_sort_pairs(ctx, n):
    rng = np.random.default_rng(n)
    idx = np.arange(n, dtype=np.uint32)
    keys_of = _sort_keys(n, rng)
    for passes in range(1, 9):
        cases = [(name, keys, name == "equal") for name, keys in keys_of.items()]
        if passes < 8:  # must come out in index order, with their full keys
            cases.append(("above", _keys_above(n, passes, rng), True))
        for name, keys, identity in cases:
            order = idx if identity else _stable_order(keys, passes)
            k, v, in_alt, overrun = rt.capi.selftest_sort_pairs(ctx, keys, idx, passes)
            case = (n, passes, name)
            assert not overrun, case
            assert in_alt == (passes % 2 == 1), case
            assert np.array_equal(v, order), (case, int(np.argmax(v != order)))
            assert np.array_equal(k, keys[order]), case


def test_selftest_arguments_are_checked_before_any_device_work(ctx):
    """A dummy context handle is never dereferenced: an invalid-argument status shows that nothing reached the device."""
    lib = ctx.lib
    dummy = C.c_void_p(1)
    a = np.arange(8, dtype=np.uint32)
    out = np.full(8, 7, np.uint32)
    ov = C.c_int32(-1)
    for h in (ctx._h, dummy):
        for eb in (0, 2, 3, 16, -4):
            assert lib.rt_selftest_exclusive_sum(h, a.ctypes.data, out.ctypes.data, 8, eb, 0, C.byref(ov)) == capi.RT_ERR_INVALID_ARG
        assert lib.rt_selftest_exclusive_sum(h, None, out.ctypes.data, 8, 4, 0, C.byref(ov)) == capi.RT_ERR_INVALID_ARG
        assert lib.rt_selftest_exclusive_sum(h, a.ctypes.data, None, 8, 4, 0, C.byref(ov)) == capi.RT_ERR_INVALID_ARG
        assert lib.rt_selftest_exclusive_sum(h, a.ctypes.data, out.ctypes.data, 8, 4, 0, None) == capi.RT_ERR_INVALID_ARG
    assert lib.rt_selftest_exclusive_sum(None, a.ctypes.data, out.ctypes.data, 8, 4, 0, C.byref(ov)) == capi.RT_ERR_INVALID_ARG
    assert np.array_equal(out, np.full(8, 7, np.uint32)) and ov.value == -1

    keys, vals = np.arange(8, dtype=np.uint64)[::-1].copy(), np.arange(8, dtype=np.uint32)
    ko, vo = np.full(8, 7, np.uint64), np.full(8, 7, np.uint32)
    alt = C.c_int32(-1)
    K, V, KO, VO = keys.ctypes.data, vals.ctypes.data, ko.ctypes.data, vo.ctypes.data
    for h in (ctx._h, dummy):
        for passes in (0, 9, -1):
            assert lib.rt_selftest_sort_pairs(h, K, V, 8, passes, KO, VO, C.byref(alt), C.byref(ov)) == capi.RT_ERR_INVALID_ARG
        for bad in ((None, V, KO, VO), (K, None, KO, VO), (K, V, None, VO), (K, V, KO, None)):
            assert lib.rt_selftest_sort_pairs(h, *bad[:2], 8, 8, *bad[2:], C.byref(alt), C.byref(ov)) == capi.RT_ERR_INVALID_ARG
        assert lib.rt_selftest_sort_pairs(h, K, V, 8, 8, KO, VO, None, C.byref(ov)) == capi.RT_ERR_INVALID_ARG
        assert lib.rt_selftest_sort_pairs(h, K, V, 8, 8, KO, VO, C.byref(alt), None) == capi.RT_ERR_INVALID_ARG
        assert lib.rt_selftest_sort_pairs(h, K, V, 2**32, 8, KO, VO, C.byref(alt), C.byref(ov)) == capi.RT_ERR_INVALID_ARG
    assert np.array_equal(ko, np.full(8, 7, np.uint64)) and np.array_equal(vo, np.full(8, 7, np.uint32))
    assert alt.value == -1 and ov.value == -1
    # n = 0 is valid: nothing is launched or written
    assert lib.rt_selftest_sort_pairs(ctx._h, K, V, 0, 3, KO, VO, C.byref(alt), C.byref(ov)) == capi.RT_OK
    assert alt.value == 0 and ov.value == 0 and np.array_equal(ko, np.full(8, 7, np.uint64))
    assert lib.rt_selftest_sort_pairs(ctx._h, None, None, 0, 3, None, None, C.byref(alt), C.byref(ov)) == capi.RT_OK
