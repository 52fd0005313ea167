"""Adaptive sampling without a device: the numpy float32 restatement of the per-pixel error e, the windowed error ebar and
the selection step (include/rt_api.h, csrc/rt_adaptive.cu), its unit cases, the ABI of rt_adaptive_params and the
argument checks that reject a call before any device work."""
import ctypes as C

import numpy as np
import pytest

import raytracing_renderer_cuda_b200 as rt
from raytracing_renderer_cuda_b200 import capi

F32 = np.float32


def error_map(planes: np.ndarray) -> np.ndarray:
    """e of every pixel of a two-plane accumulator [2, H, W, 4] in float32, one IEEE operation per step as on the device:
    (|g(A_r/A_w) - g(B_r/B_w)| + |g(A_g/A_w) - g(B_g/B_w)| + |g(A_b/A_w) - g(B_b/B_w)|) / 6, g(x) = sqrt(saturate(x)),
    +inf where either plane has no samples."""
    a, b = np.asarray(planes[0], F32), np.asarray(planes[1], F32)
    ok = (a[..., 3] > 0) & (b[..., 3] > 0)
    with np.errstate(divide="ignore", invalid="ignore"):
        ga = np.sqrt(np.clip(a[..., :3] / a[..., 3:4], F32(0), F32(1)))
        gb = np.sqrt(np.clip(b[..., :3] / b[..., 3:4], F32(0), F32(1)))
    d = np.abs(ga - gb)
    e = ((d[..., 0] + d[..., 1]) + d[..., 2]) / F32(6)
    return np.where(ok, e, F32(np.inf)).astype(F32)


def window(e: np.ndarray) -> np.ndarray:
    """ebar: the 3x3 neighbourhood of every pixel, coordinates clamped to the frame, summed in row-major order, / 9."""
    h, w = e.shape
    ys, xs = np.arange(h), np.arange(w)
    s = np.zeros_like(e, dtype=F32)
    for dy in (-1, 0, 1):
        yy = np.clip(ys + dy, 0, h - 1)
        for dx in (-1, 0, 1):
            xx = np.clip(xs + dx, 0, w - 1)
            s = (s + e[yy][:, xx]).astype(F32)
    return (s / F32(9)).astype(F32)


def select(planes: np.ndarray, current: np.ndarray, tau: float, max_spp: int) -> np.ndarray:
    """The next pixel list: the entries of `current` (flat pixel indices) with ebar >= tau and count < max_spp, in list order."""
    eb = window(error_map(planes)).ravel()
    count = (planes[0, ..., 3] + planes[1, ..., 3]).ravel()
    keep = (eb[current] >= F32(tau)) & (count[current] < max_spp)
    return current[keep]


def _planes(h, w, counts, seed=0, noise=0.1):
    """Two planes whose halves hold counts / 2 samples of a value around 0.5 each."""
    rng = np.random.default_rng(seed)
    half = (np.asarray(counts, F32) / 2).reshape(h, w)
    p = np.zeros((2, h, w, 4), F32)
    for k in range(2):
        p[k, ..., :3] = (0.5 + noise * rng.standard_normal((h, w, 3))).astype(F32) * half[..., None]
        p[k, ..., 3] = half
    return p


def test_error_of_identical_planes_is_zero_and_empty_planes_are_inf():
    p = _planes(4, 5, np.full(20, 8))
    p[1] = p[0]
    assert (error_map(p) == 0).all()
    p[1, 2, 3] = 0.0  # pixel (row 2, column 3): plane B has no samples
    e = error_map(p)
    assert np.isinf(e[2, 3]) and np.isfinite(np.delete(e.ravel(), 2 * 5 + 3)).all()
    eb = window(e)
    # an infinite error keeps its whole 3x3 neighbourhood above any threshold
    assert np.isinf(eb[1:4, 2:5]).all() and np.isfinite(eb[:, :2]).all() and np.isfinite(eb[0]).all()
    cur = np.arange(20, dtype=np.uint32)
    nxt = select(p, cur, 1e30, 1 << 20)
    assert sorted(nxt.tolist()) == [r * 5 + c for r in (1, 2, 3) for c in (2, 3, 4)]


def test_error_is_half_the_mean_display_difference():
    p = np.zeros((2, 1, 1, 4), F32)
    p[0, 0, 0] = (0.25 * 4, 0.25 * 4, 0.0, 4)  # A: mean (0.25, 0.25, 0), display (0.5, 0.5, 0)
    p[1, 0, 0] = (1.0 * 4, 0.0, 2.0 * 4, 4)    # B: mean (1, 0, 2), display (1, 0, 1): saturated before the square root
    assert error_map(p)[0, 0] == F32((0.5 + 0.5 + 1.0) / 6)


def test_window_clamps_at_the_border():
    e = np.arange(12, dtype=F32).reshape(3, 4)
    eb = window(e)
    # corner (0, 0): rows {0, 0, 1} x columns {0, 0, 1}
    want = (e[0, 0] * 4 + e[0, 1] * 2 + e[1, 0] * 2 + e[1, 1]) / 9
    assert abs(float(eb[0, 0]) - want) < 1e-6
    assert abs(float(eb[1, 1]) - e[0:3, 0:3].mean()) < 1e-6
    # a one-pixel frame is its own neighbourhood
    one = window(np.array([[F32(0.3)]]))[0, 0]
    s = F32(0)
    for _ in range(9):
        s = F32(s + F32(0.3))
    assert one == F32(s / F32(9))


def test_selection_keeps_list_order_and_never_grows():
    h, w = 16, 24
    rng = np.random.default_rng(3)
    counts = np.full(h * w, 16)
    cur = np.arange(h * w, dtype=np.uint32)
    for it in range(6):
        p = _planes(h, w, counts, seed=it, noise=float(rng.uniform(0.0, 0.2)))
        nxt = select(p, cur, 0.01, 256)
        assert set(nxt.tolist()) <= set(cur.tolist())
        assert np.all(np.diff(nxt.astype(np.int64)) > 0)  # pixel order, as the first list
        counts[nxt] += 16
        cur = nxt


def test_max_spp_caps_the_list():
    h, w = 8, 8
    counts = np.full(h * w, 32)
    counts[:10] = 64
    p = _planes(h, w, counts, noise=0.3)
    cur = np.arange(h * w, dtype=np.uint32)
    assert select(p, cur, 0.0, 64).tolist() == list(range(10, 64))
    assert select(p, cur, 0.0, 32).size == 0


def test_threshold_zero_keeps_every_pixel_and_inf_none():
    p = _planes(5, 7, np.full(35, 4))
    cur = np.arange(35, dtype=np.uint32)
    assert np.array_equal(select(p, cur, 0.0, 1 << 20), cur)
    assert select(p, cur, np.finfo(np.float32).max, 1 << 20).size == 0


def test_adaptive_params_abi_and_defaults():
    lib = capi.load_library()
    assert lib.rt_abi_sizeof(b"rt_adaptive_params") == C.sizeof(capi.rt_adaptive_params) == 16
    capi.check_layout(lib)
    a = rt.default_adaptive_params()
    assert (a.min_spp, a.step_spp, a.max_spp) == (32, 32, 256) and a.threshold == F32(1 / 255)
    assert rt.default_adaptive_params(max_spp=64).max_spp == 64


BAD = [dict(min_spp=0), dict(min_spp=3), dict(min_spp=-2), dict(step_spp=0), dict(step_spp=5), dict(max_spp=8),
       dict(max_spp=40), dict(max_spp=(1 << 24) + 16), dict(threshold=float("nan")), dict(threshold=-1e-3),
       dict(threshold=float("inf"))]


@pytest.mark.parametrize("kw", BAD)
def test_bad_adaptive_params_are_rejected_before_any_device_work(kw):
    """The parameter checks run before the context or the scene is read: the dummy handles below are never dereferenced,
    so an invalid-argument status shows that nothing reached the device."""
    lib = capi.load_library()
    p = rt.default_params(width=16, height=8)
    a = rt.default_adaptive_params(**kw)
    out = np.empty((8, 16, 3), np.float32)
    dummy = C.c_void_p(1)
    assert lib.rt_render_adaptive(dummy, dummy, C.byref(p), C.byref(a), out.ctypes.data, None, None) == capi.RT_ERR_INVALID_ARG
    assert lib.rt_render_adaptive_device(dummy, dummy, C.byref(p), C.byref(a), dummy, None, None, None) == capi.RT_ERR_INVALID_ARG


def test_null_and_bad_frame_arguments_are_rejected():
    lib = capi.load_library()
    dummy = C.c_void_p(1)
    p = rt.default_params(width=16, height=8)
    a = rt.default_adaptive_params()
    out = np.empty((8, 16, 3), np.float32)
    calls = [
        lambda: lib.rt_render_adaptive(None, dummy, C.byref(p), C.byref(a), out.ctypes.data, None, None),
        lambda: lib.rt_render_adaptive(dummy, None, C.byref(p), C.byref(a), out.ctypes.data, None, None),
        lambda: lib.rt_render_adaptive(dummy, dummy, None, C.byref(a), out.ctypes.data, None, None),
        lambda: lib.rt_render_adaptive(dummy, dummy, C.byref(p), None, out.ctypes.data, None, None),
        lambda: lib.rt_render_adaptive(dummy, dummy, C.byref(p), C.byref(a), None, None, None),
        lambda: lib.rt_render_adaptive(dummy, dummy, C.byref(rt.default_params(width=0)), C.byref(a), out.ctypes.data, None, None),
        lambda: lib.rt_render_adaptive(dummy, dummy, C.byref(rt.default_params(sample_offset=(1 << 31) - 100)), C.byref(a),
                                       out.ctypes.data, None, None),
        lambda: lib.rt_render_adaptive_device(None, dummy, C.byref(p), C.byref(a), dummy, None, None, None),
        lambda: lib.rt_render_adaptive_device(dummy, None, C.byref(p), C.byref(a), dummy, None, None, None),
        lambda: lib.rt_render_adaptive_device(dummy, dummy, None, C.byref(a), dummy, None, None, None),
        lambda: lib.rt_render_adaptive_device(dummy, dummy, C.byref(p), None, dummy, None, None, None),
        lambda: lib.rt_render_adaptive_device(dummy, dummy, C.byref(p), C.byref(a), None, None, None, None),
        lambda: lib.rt_adaptive_error_device(None, dummy, 16, 8, dummy),
        lambda: lib.rt_adaptive_error_device(dummy, None, 16, 8, dummy),
        lambda: lib.rt_adaptive_error_device(dummy, dummy, 16, 8, None),
        lambda: lib.rt_adaptive_error_device(dummy, dummy, 0, 8, dummy),
        lambda: lib.rt_adaptive_error_device(dummy, dummy, 16, -1, dummy),
        lambda: lib.rt_adaptive_error_device(dummy, dummy, 1 << 16, 1 << 15, dummy),
    ]
    for k, call in enumerate(calls):
        assert call() == capi.RT_ERR_INVALID_ARG, k
