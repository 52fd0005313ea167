"""The framebuffer passes bit for bit: rt_tonemap_device (k_tonemap, four pixels per thread or one) and the peer form of
rt_reduce_tonemap_peers (k_reduce_tonemap) run on one device with N accumulators on that device as the members.

References: the oracle's pixel finalisation (main.cu:124-127) for the float image, a numpy float32 restatement of the
writer's conversion (Y flip, int(255.999f * c) & 255) for the bytes, and the float32 sum a0 + a1 + ... in rank order for
the summed accumulator.  The accumulators hold random sums plus pixels with count 0, NaN and infinities, negative values and
-0.0, denormals, means next to 1 and means whose 255.999 c lands next to an integer.  Every output buffer sits inside a
larger buffer of sentinel bytes, at byte offsets that force the one-pixel form of a width that allows four: the bytes
written must be those of the references and nothing outside the image (or outside the band of rows) may change.

Out of scope here: the NVLS multicast form (tests/test_gpu_multi.py) and misaligned accumulator or out_sum pointers, which
the entries do not check and the kernels' 16-byte accesses cannot take."""
import ctypes as C

import numpy as np
import pytest

import raytracing_renderer_cuda_b200 as rt
from raytracing_renderer_cuda_b200 import capi

pytestmark = pytest.mark.gpu

F32 = np.float32
SENTINEL = 0x5C  # as a float 2.5e17: never a finalised value
PAD = 256        # sentinel bytes before and after every output (keeps the allocation's alignment)
SIZES = ((1, 1), (3, 1), (4, 1), (5, 2), (63, 17), (64, 17), (65, 17), (66, 17), (67, 17), (1200, 600))  # (width, height)
# (byte offset of out_rgb, of out_rgb8); None = that output is not requested.  Offsets 4 / 8 and 1..3 take away the
# alignment of the 16-byte (rgb) and 4-byte (rgb8) stores, so the launcher must pick the one-pixel form.
OUTPUTS = ((0, 0), (4, 0), (8, 0), (0, 1), (0, 2), (0, 3), (8, 3), (0, None), (4, None), (8, None), (None, 0), (None, 1), (None, 2),
           (None, 3))
G_FORMS = (None, "4", "1")  # RT_REDUCE_G: unset (the launcher's choice), four pixels per thread, one


def _torch():
    import torch

    return torch


@pytest.fixture(scope="module")
def ctx():
    return rt.Context(0)


# ------------------------------------------------------------------------------------------------------ inputs ----
def _q8_edge_pixels(oracle) -> np.ndarray:
    """(m, m, m, 1) pixels whose finalised value c = sqrt_rz(m) puts 255.999f * c at an integer or one ulp either side"""
    cands = []
    for k in range(1, 256):
        c0 = F32(k / 255.999)
        for d in range(-3, 4):
            c = F32(c0 + d * np.spacing(c0))
            if c > 1:
                continue
            c2 = float(c) * float(c)
            m = F32(c2)
            if float(m) < c2:
                m = np.nextafter(m, F32(2))  # the smallest float >= c^2: its truncated root is c
            cands.append((m, c))
    px = np.array([[m, m, m, 1] for m, _ in cands], F32)
    c = np.array([c for _, c in cands], F32)
    got = oracle.tonemap(px[None])[0, :, 0]
    keep = got == c
    assert keep.mean() > 0.9
    px, c = px[keep], c[keep]
    p = F32(255.999) * c
    k = np.rint(p)
    ulps = np.rint((p - k) / np.spacing(k.astype(F32)))
    near = np.abs(ulps) <= 1
    assert set(ulps[near].astype(int).tolist()) == {-1, 0, 1}
    return px[near]


def _special_pixels(oracle) -> np.ndarray:
    nan, inf = np.nan, np.inf
    sub, sub_min = 1e-40, 1.4e-45  # denormals
    one_m, one_p = float(np.nextafter(F32(1), F32(0))), float(np.nextafter(F32(1), F32(2)))
    rows = [
        # count 0 (and -0.0), with zero and with non-zero sums
        (0, 0, 0, 0), (1, 2, 3, 0), (-1, 0.5, 1e30, 0), (0, 0, 0, -0.0), (0.25, 0, 0, -0.0),
        # NaN and infinities in the sums and in the count
        (nan, 0.5, 0.5, 1), (0.5, nan, 0.5, 2), (0.5, 0.5, nan, 3), (inf, -inf, 0.5, 1), (-inf, inf, inf, 4),
        (0.5, 0.5, 0.5, nan), (0.5, 0.5, 0.5, inf), (0.5, 0.5, 0.5, -inf), (inf, nan, -inf, inf), (nan, nan, nan, nan),
        (inf, inf, inf, 0), (nan, 1, 1, 0),
        # negative values and -0.0
        (-1, -2, -3, 4), (-0.0, -0.0, -0.0, 1), (-0.0, 0.25, -0.0, 2), (0.5, 0.25, 1.0, -1), (-0.5, -0.25, -1.0, -2),
        (0.3, -0.0, 0.7, -0.0), (-1e-30, 1e-30, -0.0, 1e-30),
        # denormals in the sums and in the count
        (sub, sub_min, 1e-39, 1), (0.5, 0.25, 0.125, sub), (sub, sub, sub, sub), (sub_min, sub_min, sub_min, 3),
        (1e-38, 1.17e-38, sub, 0.5), (-sub, sub, -sub_min, 1), (sub, 0, 0, 1e38),
        # means at 1 - ulp, 1, 1 + ulp, and sums whose mean is 1 only up to rz(1 / count)
        (one_m, 1, one_p, 1), (2 * one_m, 2, 2 * one_p, 2), (3, 3, 3, 3), (7, 7, 7, 7), (1e20, 1e20, 1e20, 1e20),
        (3 * one_p, 5 * one_p, 7 * one_p, 1), (1e-20, 1e-19, 1e-18, 1e-20),
    ]
    return np.concatenate([np.array(rows, F32), _q8_edge_pixels(oracle)])


def _accum(w: int, h: int, seed: int, specials: np.ndarray) -> np.ndarray:
    """[h, w, 4] float32: random sums of 1..64 samples (means up to 1.3, so some saturate) with special pixels at random
    places"""
    rng = np.random.default_rng(seed)
    cnt = rng.integers(1, 65, (h, w)).astype(F32)
    acc = np.empty((h, w, 4), F32)
    acc[..., :3] = rng.random((h, w, 3), dtype=F32) * cnt[..., None] * F32(1.3)
    acc[..., 3] = cnt
    flat = acc.reshape(-1, 4)
    k = min(len(specials), flat.shape[0])
    flat[rng.choice(flat.shape[0], k, replace=False)] = specials[rng.permutation(len(specials))[:k]]
    return acc


@pytest.fixture(scope="module")
def specials(oracle):
    return _special_pixels(oracle)


# -------------------------------------------------------------------------------------------------- references ----
def _ref_rgb8(rgb: np.ndarray) -> np.ndarray:
    """the writer's conversion (main.cu:476-487): row r of the picture is row H - 1 - r of the frame, int(255.999f*c) & 255"""
    return np.ascontiguousarray(((F32(255.999) * rgb).astype(np.int32) & 255).astype(np.uint8)[::-1])


def _rank_order_sum(members) -> np.ndarray:
    s = members[0].copy()
    with np.errstate(invalid="ignore"):  # (inf + -inf of the special pixels)
        for a in members[1:]:
            s = s + a
    return s


def _same_floats(got: np.ndarray, want: np.ndarray) -> bool:
    """bit for bit, except that any NaN matches any NaN (the payload of a NaN produced by an add is not specified)"""
    g, w = got.reshape(-1).view(np.uint32), want.reshape(-1).view(np.uint32)
    both_nan = np.isnan(got.reshape(-1)) & np.isnan(want.reshape(-1))
    return bool(np.all((g == w) | both_nan))


# ------------------------------------------------------------------------------------------- sentinel buffers ----
class Sentinel:
    """`nbytes` of device memory at byte offset `off` inside a buffer of sentinel bytes"""

    def __init__(self, nbytes: int, off: int = 0):
        torch = _torch()
        self.lo, self.hi = PAD + off, PAD + off + nbytes
        self.buf = torch.full((self.hi + PAD,), SENTINEL, dtype=torch.uint8, device="cuda")
        self.ptr = self.buf.data_ptr() + self.lo

    def host(self) -> np.ndarray:
        return self.buf.cpu().numpy()

    def payload(self, dtype=np.uint8) -> np.ndarray:
        return np.frombuffer(self.host()[self.lo:self.hi].tobytes(), dtype)

    def outside_untouched(self) -> bool:
        b = self.host()
        return bool((b[:self.lo] == SENTINEL).all() and (b[self.hi:] == SENTINEL).all())


def _outputs(w, h, rgb_off, rgb8_off, with_sum=False):
    rgb = Sentinel(w * h * 12, rgb_off) if rgb_off is not None else None
    rgb8 = Sentinel(w * h * 3, rgb8_off) if rgb8_off is not None else None
    tot = Sentinel(w * h * 16) if with_sum else None
    _torch().cuda.synchronize()
    return rgb, rgb8, tot


def _ptr(s):
    return s.ptr if s is not None else 0


def _check_image(rgb, rgb8, want_rgb, want_rgb8, what):
    if rgb is not None:
        assert rgb.outside_untouched(), ("rgb written outside the image", what)
        assert np.array_equal(rgb.payload(np.uint32), want_rgb.reshape(-1).view(np.uint32)), ("rgb", what)
    if rgb8 is not None:
        assert rgb8.outside_untouched(), ("rgb8 written outside the image", what)
        assert np.array_equal(rgb8.payload(), want_rgb8.reshape(-1)), ("rgb8", what)


def _device(a: np.ndarray):
    return _torch().from_numpy(np.ascontiguousarray(a)).cuda()


# -------------------------------------------------------------------------------------------- rt_tonemap_device ----
def _tonemap_all_outputs(ctx, acc_dev, w, h, want_rgb, want_rgb8, outputs):
    for rgb_off, rgb8_off in outputs:
        rgb, rgb8, _ = _outputs(w, h, rgb_off, rgb8_off)
        rt.tonemap_device(ctx, acc_dev.data_ptr(), w, h, _ptr(rgb), _ptr(rgb8))
        ctx.synchronize()
        _check_image(rgb, rgb8, want_rgb, want_rgb8, (w, h, rgb_off, rgb8_off))


@pytest.mark.parametrize("w,h", SIZES)
def test_tonemap_every_output_form_bit_exact(ctx, oracle, specials, w, h):
    acc = _accum(w, h, seed=w * 1000 + h, specials=specials)
    want = oracle.tonemap(acc)
    assert np.all((want >= 0) & (want <= 1))
    _tonemap_all_outputs(ctx, _device(acc), w, h, want, _ref_rgb8(want), OUTPUTS)


def test_tonemap_8k_bit_exact(ctx, oracle, specials):
    w, h = 7680, 4320
    acc = _accum(w, h, seed=8, specials=specials)
    want = oracle.tonemap(acc)
    _tonemap_all_outputs(ctx, _device(acc), w, h, want, _ref_rgb8(want), ((0, 0), (4, 1)))


def test_special_pixels_finalise_as_the_oracle(ctx, oracle, specials):
    """Every special pixel once, in both kernel forms (a width of 4 and a width of 1), and what the oracle makes of them."""
    px = specials
    want = oracle.tonemap(px[None])[0]
    # count 0: 1 / 0 = inf, so zero sums (0 * inf = NaN) finalise to +0 and positive sums to 1
    assert np.array_equal(want[:2].view(np.uint32), np.array([[0] * 3, [0x3F800000] * 3], np.uint32))
    for w in (4, 1):
        n = len(px) - len(px) % 4
        h = n // w
        acc = px[:n].reshape(h, w, 4)
        wr = want[:n].reshape(h, w, 3)
        _tonemap_all_outputs(ctx, _device(acc), w, h, wr, _ref_rgb8(wr), ((0, 0), (4, 2)))


# --------------------------------------------------------------------------------- rt_reduce_tonemap_peers ----
def _set_g(monkeypatch, g):
    if g is None:
        monkeypatch.delenv("RT_REDUCE_G", raising=False)
    else:
        monkeypatch.setenv("RT_REDUCE_G", g)  # read by the launcher on every call


def _members(w, h, n, seed, specials):
    host = [_accum(w, h, seed + 7919 * m, specials) for m in range(n)]
    return host, [_device(a) for a in host]


def _reduce(ctx, devs, w, h, r0, r1, rgb, rgb8, tot):
    rt.reduce_tonemap_peers(ctx, [d.data_ptr() for d in devs], 0, w, h, r0, r1, _ptr(rgb), _ptr(rgb8), _ptr(tot))
    ctx.synchronize()


@pytest.mark.parametrize("n_members", (1, 2, 3, 4, 8, 16))
@pytest.mark.parametrize("w,h", ((67, 19), (128, 21)))
def test_reduce_tonemap_peers_on_one_device(ctx, oracle, specials, monkeypatch, n_members, w, h):
    host, devs = _members(w, h, n_members, seed=n_members * 100 + w, specials=specials)
    want_sum = _rank_order_sum(host)
    want_rgb = oracle.tonemap(want_sum)
    want_rgb8 = _ref_rgb8(want_rgb)
    for g in G_FORMS:
        _set_g(monkeypatch, g)
        for rgb_off, rgb8_off, with_sum in ((0, 0, True), (4, 1, True), (None, 0, False), (8, None, False), (None, None, True)):
            what = (n_members, w, h, g, rgb_off, rgb8_off, with_sum)
            rgb, rgb8, tot = _outputs(w, h, rgb_off, rgb8_off, with_sum)
            _reduce(ctx, devs, w, h, 0, h, rgb, rgb8, tot)
            _check_image(rgb, rgb8, want_rgb, want_rgb8, what)
            if tot is not None:
                assert tot.outside_untouched(), ("out_sum written outside the frame", what)
                assert _same_floats(tot.payload(F32), want_sum), ("out_sum", what)
            if n_members == 1 and rgb is not None and rgb8 is not None:  # one member: the same bytes as rt_tonemap_device
                rgb_t, rgb8_t, _ = _outputs(w, h, rgb_off, rgb8_off)
                rt.tonemap_device(ctx, devs[0].data_ptr(), w, h, rgb_t.ptr, rgb8_t.ptr)
                ctx.synchronize()
                assert np.array_equal(rgb_t.host(), rgb.host()) and np.array_equal(rgb8_t.host(), rgb8.host()), what


def _band_expectation(full: dict, w: int, h: int, r0: int, r1: int) -> dict:
    """the sentinel buffers after a band [r0, r1): the full-frame bytes in the band's rows (rgb8: the flipped rows), sentinel
    everywhere else"""
    out = {}
    for name, b in full.items():
        e = np.full_like(b, SENTINEL)
        if name == "rgb8":
            lo, hi = (h - r1) * w * 3, (h - r0) * w * 3
        else:
            per = 12 if name == "rgb" else 16
            lo, hi = r0 * w * per, r1 * w * per
        e[PAD + lo:PAD + hi] = b[PAD + lo:PAD + hi]
        out[name] = e
    return out


@pytest.mark.parametrize("w,h", ((67, 19), (128, 21)))
def test_reduce_tonemap_row_bands(ctx, oracle, specials, monkeypatch, w, h):
    host, devs = _members(w, h, 3, seed=w + h, specials=specials)
    want_sum = _rank_order_sum(host)
    want_rgb = oracle.tonemap(want_sum)
    for g in G_FORMS:
        _set_g(monkeypatch, g)

        def run(bands):
            rgb, rgb8, tot = _outputs(w, h, 0, 0, True)
            for r0, r1 in bands:
                _reduce(ctx, devs, w, h, r0, r1, rgb, rgb8, tot)
            return {"rgb": rgb.host(), "rgb8": rgb8.host(), "sum": tot.host()}

        full = run([(0, h)])
        assert np.array_equal(full["rgb"][PAD:-PAD].view(np.uint32), want_rgb.reshape(-1).view(np.uint32)), g
        assert np.array_equal(full["rgb8"][PAD:-PAD], _ref_rgb8(want_rgb).reshape(-1)), g
        assert _same_floats(full["sum"][PAD:-PAD].view(F32), want_sum), g
        singles = [(0, 0), (h, h), (0, 1), (h - 1, h), (2, 5)]
        for world in range(2, 9):
            shards = [rt.shard_rows(h, r, world) for r in range(world)]
            union = run(shards)
            for name in full:
                assert np.array_equal(union[name], full[name]), (g, world, name)
            singles += shards
        for r0, r1 in singles:
            got, want = run([(r0, r1)]), _band_expectation(full, w, h, r0, r1)
            for name in full:
                assert np.array_equal(got[name], want[name]), (g, (r0, r1), name)


def test_reduce_tonemap_8k_two_members(ctx, oracle, specials):
    """the peer form at the full frame size of the multi-GPU configuration"""
    w, h = 7680, 4320
    host, devs = _members(w, h, 2, seed=2, specials=specials)
    want_sum = _rank_order_sum(host)
    want_rgb = oracle.tonemap(want_sum)
    rgb, rgb8, tot = _outputs(w, h, 0, 0, True)
    _reduce(ctx, devs, w, h, 0, h, rgb, rgb8, tot)
    _check_image(rgb, rgb8, want_rgb, _ref_rgb8(want_rgb), "8k")
    assert tot.outside_untouched() and _same_floats(tot.payload(F32), want_sum)


def test_reduce_tonemap_bad_arguments_write_nothing(ctx, specials):
    w, h = 16, 8
    _, devs = _members(w, h, 17, seed=5, specials=specials)
    ptrs = [d.data_ptr() for d in devs]
    rgb, rgb8, tot = _outputs(w, h, 0, 0, True)
    lib = ctx.lib

    def call(members, n, r0=0, r1=h, outs=(rgb.ptr, rgb8.ptr, tot.ptr), width=w, height=h, table=True):
        arr = (C.c_void_p * max(len(members), 1))(*[C.c_void_p(p) for p in members]) if table else None
        return lib.rt_reduce_tonemap_peers(ctx._h, arr, n, None, width, height, r0, r1, *[C.c_void_p(p or None) for p in outs])

    assert call(ptrs[:1], 0) == capi.RT_ERR_INVALID_ARG
    assert call(ptrs, 17) == capi.RT_ERR_INVALID_ARG
    assert call([ptrs[0], 0, ptrs[2]], 3) == capi.RT_ERR_INVALID_ARG  # a NULL member
    assert call(ptrs[:2], 2, table=False) == capi.RT_ERR_INVALID_ARG   # neither a member table nor a multicast address
    assert call(ptrs[:2], 2, r0=5, r1=4) == capi.RT_ERR_INVALID_ARG
    assert call(ptrs[:2], 2, r0=0, r1=h + 1) == capi.RT_ERR_INVALID_ARG
    assert call(ptrs[:2], 2, r0=-1, r1=h) == capi.RT_ERR_INVALID_ARG
    assert call(ptrs[:2], 2, outs=(0, 0, 0)) == capi.RT_ERR_INVALID_ARG
    assert call(ptrs[:2], 2, width=0) == capi.RT_ERR_INVALID_ARG
    assert call(ptrs[:2], 2, height=-1, r1=0) == capi.RT_ERR_INVALID_ARG
    ctx.synchronize()
    for s in (rgb, rgb8, tot):
        assert (s.host() == SENTINEL).all()
    assert call(ptrs[:16], 16) == capi.RT_OK  # (the same call with 16 members is valid)
    ctx.synchronize()
