"""Denoiser (include/rt_api.h: rt_render_features_device, rt_denoise_device, rt_render_denoised) without a GPU: the ABI of
rt_denoise_params, the CPU restatement of the feature pass (tests/feature_oracle.cpp, built here against the unchanged
oracle) and the numpy restatement of the edge-avoiding à-trous filter.  The restatements are what
tests/test_gpu_denoise.py holds the device kernels against; the quality test below lets the default sigmas be checked
on a CPU."""
import ctypes as C
import json
import subprocess

import numpy as np
import pytest

import raytracing_renderer_cuda_b200 as rt
from raytracing_renderer_cuda_b200 import capi
from tests.conftest import ROOT

H_B3 = np.array([1.0, 4.0, 6.0, 4.0, 1.0]) / 16.0
Z_EPS = 1e-4  # RT_ATROUS_EPS (csrc/rt_denoise.cu)


def atrous_reference(accum: np.ndarray, features: np.ndarray, d) -> np.ndarray:
    """The filter of rt_denoise_device in float64: accum [H, W, 4] float32, features [2, H, W, 4].  Returns the float4
    buffer the pixel finalisation reads: (c, 1) where the pixel has samples, the accumulator's own value where it has none."""
    acc = np.asarray(accum, np.float32)
    h, w = acc.shape[:2]
    valid = acc[..., 3] > 0
    with np.errstate(divide="ignore", invalid="ignore"):
        inv = np.float32(1.0) / acc[..., 3]  # the level-0 mean colour: saturate(sum * rn(1 / count)) in float32
        col = np.clip(acc[..., :3] * inv[..., None], 0.0, 1.0).astype(np.float64)
    col[~valid] = 0.0
    f0 = np.asarray(features[0], np.float64)
    f1 = np.asarray(features[1], np.float64)
    nrm, z = f0[..., :3], f0[..., 3]
    for level in range(d.iterations):
        step = 1 << level
        k_c = 1.0 / (np.float32(d.sigma_color) / step) ** 2
        k_n, k_z, k_a = 1.0 / np.float32(d.sigma_normal) ** 2, 1.0 / np.float32(d.sigma_depth), 1.0 / np.float32(d.sigma_albedo) ** 2
        num = np.zeros((h, w, 3))
        den = np.zeros((h, w))
        for dy in range(-2, 3):
            yy = np.arange(h) + dy * step
            iny = (yy >= 0) & (yy < h)
            yy = np.clip(yy, 0, h - 1)
            for dx in range(-2, 3):
                xx = np.arange(w) + dx * step
                inx = (xx >= 0) & (xx < w)
                xx = np.clip(xx, 0, w - 1)
                ok = iny[:, None] & inx[None, :] & valid[yy][:, xx]
                cq, nq, zq, aq = col[yy][:, xx], nrm[yy][:, xx], z[yy][:, xx], f1[yy][:, xx]
                e = (((col - cq) ** 2).sum(-1) * k_c + ((nrm - nq) ** 2).sum(-1) * k_n
                     + np.abs(z - zq) / np.maximum(np.maximum(z, zq), Z_EPS) * k_z + ((f1 - aq) ** 2).sum(-1) * k_a)
                wt = np.where(ok, H_B3[dy + 2] * H_B3[dx + 2] * np.exp(-e), 0.0)
                den += wt
                num += wt[..., None] * cq
        col = np.where(valid[..., None], num / np.where(valid, den, 1.0)[..., None], col)
    out = acc.copy()
    out[valid, :3] = col[valid]
    out[valid, 3] = 1.0
    return out


def finalise(buf: np.ndarray) -> np.ndarray:
    """Pixel finalisation (main.cu:124-127) in ordinary float arithmetic: enough for PSNR comparisons."""
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.sqrt(np.nan_to_num(np.clip(buf[..., :3] / buf[..., 3:4], 0.0, 1.0)))


class FeatureOracle:
    """tests/feature_oracle.cpp: orc_features(scene, params, feature_spp, nthreads, out)."""

    def __init__(self, path):
        L = self.L = C.CDLL(str(path))
        L.orc_scene_create.restype = C.c_void_p
        L.orc_scene_create.argtypes = [C.POINTER(capi.rt_scene_desc)]
        L.orc_scene_destroy.argtypes = [C.c_void_p]
        L.orc_features.argtypes = [C.c_void_p, C.POINTER(capi.rt_render_params), C.c_int, C.c_int, C.c_void_p]
        L.orc_render.argtypes = [C.c_void_p, C.POINTER(capi.rt_render_params), C.c_int, C.c_int, C.c_int, C.c_void_p,
                                 C.POINTER(C.c_ulonglong)]

    def features(self, desc, params, feature_spp: int, nthreads: int = 8) -> np.ndarray:
        out = np.zeros((2, params.height, params.width, 4), np.float32)
        h = self.L.orc_scene_create(desc._ptr)
        try:
            self.L.orc_features(h, C.byref(params), feature_spp, nthreads, out.ctypes.data)
        finally:
            self.L.orc_scene_destroy(h)
        return out


def build_feature_oracle(directory) -> FeatureOracle:
    so = directory / "libfeature_oracle.so"
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-pthread", "-w",
                           str(ROOT / "tests" / "feature_oracle.cpp"), "-o", str(so)])
    return FeatureOracle(so)


@pytest.fixture(scope="module")
def feature_oracle(tmp_path_factory):
    return build_feature_oracle(tmp_path_factory.mktemp("feature_oracle"))


def test_denoise_params_abi_and_defaults():
    lib = rt.load_library()
    assert lib.rt_abi_sizeof(b"rt_denoise_params") == C.sizeof(capi.rt_denoise_params) == 24
    d = rt.default_denoise_params()
    # the values include/rt_api.h documents for rt_default_denoise_params
    assert (d.iterations, d.feature_spp) == (3, 4)
    assert np.float32(d.sigma_color) == np.float32(0.5) and d.sigma_normal == 1.0
    assert np.float32(d.sigma_depth) == np.float32(0.3) and d.sigma_albedo == 1.0
    assert rt.default_denoise_params(iterations=2).iterations == 2


TWO_SPHERES = {
    "camera": {"lookfrom": [0, 0, 5], "lookat": [0, 0, 0], "up": [0, 1, 0], "vfov": 30, "aspect": 2, "aperture": 0,
               "focus_dist": 5, "time0": 0, "time1": 0},
    "textures": {"a": {"type": "constant", "color": [0.75, 0.25, 0.5]}, "b": {"type": "constant", "color": [0.125, 0.875, 0.5]}},
    "materials": {"ma": {"type": "lambertian", "texture": "a"}, "mb": {"type": "lambertian", "texture": "b"}},
    "objects": [{"type": "sphere", "center": [-1.2, 0, 0], "radius": 0.6, "material": "ma"},
                {"type": "sphere", "center": [1.2, 0, 0], "radius": 0.6, "material": "mb"}],
}


@pytest.mark.parametrize("k", [1, 4])
def test_oracle_features_of_constant_spheres_before_the_sky(feature_oracle, k):
    desc = rt.SceneDesc.from_json(json.dumps(TWO_SPHERES))
    p = rt.default_params(width=96, height=48, world=(0.75, 0.5, 0.25))  # binary fractions: sums of K copies are exact
    f = feature_oracle.features(desc, p, k)
    n, z, alb, frac = f[0, ..., :3], f[0, ..., 3], f[1, ..., :3], f[1, ..., 3]
    full, sky = frac == 1.0, frac == 0.0
    assert full.mean() > 0.1 and sky.mean() > 0.3
    assert ((frac > 0) & (frac < 1)).any() == (k > 1)  # silhouettes
    length = np.linalg.norm(n[full], axis=1)
    if k == 1:
        assert np.abs(length - 1.0).max() < 1e-5
    else:  # mean of K unit normals of one pixel's footprint
        assert length.max() < 1.0 + 1e-5 and length.min() > 0.99
    a, b = np.array([0.75, 0.25, 0.5], np.float32), np.array([0.125, 0.875, 0.5], np.float32)
    is_a, is_b = (alb[full] == a).all(axis=1), (alb[full] == b).all(axis=1)
    assert (is_a | is_b).all() and is_a.any() and is_b.any()  # the texture constant, exactly
    assert (z[full] > 4.0).all() and (z[full] < 5.3).all()  # |lookfrom - surface| along the ray: 4.4 .. ~5.2
    assert (alb[sky] == np.array([0.75, 0.5, 0.25], np.float32)).all()  # the world colour
    assert (f[0][sky] == 0.0).all()


def _c1_frames(oracle, feature_oracle, earth, w=160, h=80):
    desc = rt.SceneDesc.builtin("earth_emitter", earth)
    o = oracle.scene(desc)
    frames = {spp: o.render(rt.default_params(width=w, height=h, spp=spp), sampler=1)[0] for spp in (4, 16)}
    # independent samples for the converged frame
    ref = o.render(rt.default_params(width=w, height=h, spp=1024, sample_offset=1 << 20), sampler=1)[0]
    feats = feature_oracle.features(desc, rt.default_params(width=w, height=h), rt.default_denoise_params().feature_spp)
    return frames, ref, feats


def test_filter_with_default_sigmas_on_c1(oracle, feature_oracle, earth):
    """Measured at 160x80 against 1024 spp: raw 4 spp 25.3 dB, denoised 4 spp 29.1 dB, raw 16 spp 31.4 dB.  The filter
    does NOT reach the quality of four times the samples (2.3 dB short, profiles/r03_denoise.md); what is asserted is the
    gain over the frame it filters and that the gap to 16 spp stays where it was measured."""
    frames, ref, feats = _c1_frames(oracle, feature_oracle, earth)
    d = rt.default_denoise_params()
    want = finalise(ref)
    raw16 = rt.psnr(finalise(frames[16]), want)
    den4 = rt.psnr(finalise(atrous_reference(frames[4], feats, d)), want)
    raw4 = rt.psnr(finalise(frames[4]), want)
    assert den4 >= raw4 + 3.0, (den4, raw4)
    assert den4 >= raw16 - 3.0, (den4, raw16)


def test_filter_returns_a_constant_image_unchanged():
    rng = np.random.default_rng(3)
    h, w = 40, 56
    acc = np.zeros((h, w, 4), np.float32)
    acc[..., :3] = np.float32(0.375) * 8
    acc[..., 3] = 8
    feats = rng.random((2, h, w, 4)).astype(np.float32)  # arbitrary guides: the weights are normalised
    out = atrous_reference(acc, feats, rt.default_denoise_params())
    assert np.abs(out[..., :3] - 0.375).max() < 1e-12 and (out[..., 3] == 1).all()


def test_filter_keeps_empty_pixels_and_ignores_them_as_neighbours():
    rng = np.random.default_rng(4)
    h, w = 24, 32
    acc = np.concatenate([rng.random((h, w, 3)) * 4, np.full((h, w, 1), 4.0)], -1).astype(np.float32)
    acc[5, 7] = (1e9, 0, 0, 0)  # no samples: must neither be filtered nor leak into its neighbours
    feats = rng.random((2, h, w, 4)).astype(np.float32)
    out = atrous_reference(acc, feats, rt.default_denoise_params(iterations=3))
    assert (out[5, 7] == acc[5, 7]).all()
    assert out[..., :3][out[..., 3] == 1].max() <= 1.0 + 1e-12
