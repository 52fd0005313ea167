"""Denoiser on the B200: the feature pass against its CPU restatement (tests/feature_oracle.cpp), the à-trous filter
against the numpy restatement (tests/test_denoise.py), the quality of denoised low-sample frames against the reference
kernel's 4096-spp frames, determinism, argument checks and the C++ app's --denoise."""
import ctypes as C
import subprocess

import numpy as np
import pytest

import raytracing_renderer_cuda_b200 as rt
from raytracing_renderer_cuda_b200 import capi
from tests.conftest import ROOT, SCENES, record_parity
from tests.test_denoise import atrous_reference, build_feature_oracle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    return rt.Context(0)


@pytest.fixture(scope="module")
def feature_oracle(tmp_path_factory):
    return build_feature_oracle(tmp_path_factory.mktemp("feature_oracle"))


@pytest.fixture(scope="module")
def gpu_golden():
    return np.load(ROOT / "tests" / "golden" / "ref_gpu_golden.npz")


def _dev(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _features(ctx, scene, p, k):
    import torch

    f = torch.zeros((2, p.height, p.width, 4), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    scene.render_features_device(p, k, f.data_ptr())
    ctx.synchronize()
    return f


def _denoise(ctx, acc_dev, feat_dev, w, h, d, rgb8=False):
    import torch

    rgb = torch.empty((h, w, 3), dtype=torch.float32, device="cuda")
    q = torch.empty((h, w, 3), dtype=torch.uint8, device="cuda") if rgb8 else None
    torch.cuda.synchronize()
    rt.denoise_device(ctx, acc_dev.data_ptr(), feat_dev.data_ptr(), w, h, d, rgb.data_ptr(), q.data_ptr() if rgb8 else 0)
    ctx.synchronize()
    return rgb.cpu().numpy(), (q.cpu().numpy() if rgb8 else None)


def test_zero_iterations_is_the_tonemap_bit_for_bit(ctx, scene_descs):
    import torch

    sc = rt.Scene(ctx, scene_descs["earth_emitter"])
    for w, h in ((64, 32), (67, 31)):  # the 4-pixel vector path and the scalar one
        acc, _ = sc.render_accum(rt.default_params(width=w, height=h, spp=4))
        acc[0, 0, :3] = 1e9
        acc[0, 1] = 0.0  # no samples
        dev = _dev(acc)
        feat = torch.zeros((2, h, w, 4), dtype=torch.float32, device="cuda")
        rgb = torch.empty((h, w, 3), dtype=torch.float32, device="cuda")
        rgb8 = torch.empty((h, w, 3), dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        rt.tonemap_device(ctx, dev.data_ptr(), w, h, rgb.data_ptr(), rgb8.data_ptr())
        ctx.synchronize()
        got, got8 = _denoise(ctx, dev, feat, w, h, rt.default_denoise_params(iterations=0), rgb8=True)
        assert got.tobytes() == rgb.cpu().numpy().tobytes() and got8.tobytes() == rgb8.cpu().numpy().tobytes()


@pytest.mark.parametrize("name,size", [("earth_emitter", (96, 48)), ("book1_final", (64, 36)), ("perlin_motion", (80, 40))])
@pytest.mark.parametrize("k", [1, 8])
def test_features_match_oracle(ctx, feature_oracle, scene_descs, name, size, k):
    """Same Philox camera rays, closest hit, hit surface and shading step as the oracle.  Hit fractions are exact.  The
    other values carry the SFU approximations of the product: the lens sample's sincos moves a ray by an ulp, which moves
    its hit point by ulps (more at grazing hits, and near a silhouette a sample may land on another object), and the
    marble and checker textures use `__sinf` (a checker near its zero crossing may pick the other child).  Measured on a
    B200: C1 0.02 % of the pixels beyond 1e-4 relative in normal or distance, C2 10-15 %, C3 3-11 %, medians <= 4e-6; the
    cause of the wider C2/C3 spread has not been isolated (profiles/r03_denoise.md).  Albedo beyond 2e-3: <= 0.1 %."""
    w, h = size
    d = scene_descs[name]
    p = rt.default_params(width=w, height=h, sample_offset=3)
    got = _features(ctx, rt.Scene(ctx, d), p, k).cpu().numpy()
    want = feature_oracle.features(d, p, k)
    assert np.array_equal(got[1, ..., 3], want[1, ..., 3])  # hit fractions
    geo = (np.abs(got[0] - want[0]) / np.maximum(np.abs(want[0]), 1.0)).max(axis=2)
    alb = np.abs(got[1, ..., :3] - want[1, ..., :3]).max(axis=2)
    record_parity("denoise_features_vs_oracle", scene=name, k=k, geo_exact=float((geo == 0).mean()), geo_frac_gt_1e4=float((geo > 1e-4).mean()),
                  geo_median=float(np.median(geo)), albedo_exact=float((alb == 0).mean()), albedo_frac_gt_2e3=float((alb > 2e-3).mean()),
                  albedo_median=float(np.median(alb)))
    assert (geo > 1e-4).mean() < 0.2 and np.median(geo) < 1e-5
    assert (alb > 2e-3).mean() < 3e-3 and np.median(alb) < 1e-5


@pytest.mark.parametrize("size", [(96, 64), (257, 131)])
@pytest.mark.parametrize("levels", [1, 2, 3, 4, 5])
def test_filter_matches_numpy_restatement(ctx, size, levels):
    """Random accumulators (with pixels that have no samples) and random features.  The device evaluates each weight with
    one __expf (max error 2 + 1.17|x| ulp, i.e. < 3e-6 relative for the exponents that carry weight) in float32 and
    divides the depth term with __fdividef; the restatement is float64.  A level's output is a normalised average of colours
    in [0, 1], so its error is a few 1e-6, and the colour term of the next level (1 / sigma_c 2^-i up to 16 here) amplifies
    it by at most ~20 per level: 1e-4 over five levels, checked on the linear values (the square of the finalised output)."""
    w, h = size
    rng = np.random.default_rng(levels * 1000 + w)
    acc = np.empty((h, w, 4), np.float32)
    acc[..., 3] = rng.integers(1, 9, (h, w))
    acc[..., :3] = rng.random((h, w, 3)) * acc[..., 3:4] * 1.3  # some means above 1: saturated
    empty = rng.random((h, w)) < 0.05
    acc[empty] = 0.0
    feats = rng.random((2, h, w, 4)).astype(np.float32)
    feats[0, ..., 3] *= 10.0  # distances
    d = rt.default_denoise_params(iterations=levels)
    got, _ = _denoise(ctx, _dev(acc), _dev(feats), w, h, d)
    want = atrous_reference(acc, feats, d)
    assert (got[empty] == 0.0).all()
    lin = got.astype(np.float64) ** 2
    err = np.abs(lin - want[..., :3])[~empty]
    assert err.max() < 1e-4 and np.median(err) < 1e-6, (float(err.max()), float(np.median(err)))


def _texture_mask(feat):
    a = feat[1, ..., :3]
    g = np.zeros(a.shape[:2])
    g[:, :-1] += np.abs(a[:, 1:] - a[:, :-1]).sum(-1)
    g[:-1, :] += np.abs(a[1:] - a[:-1]).sum(-1)
    return g > 0.1


# margin of PSNR(denoised 4 spp) over PSNR(raw 16 spp).  Measured on a B200: C1 +0.23 dB; C2 -1.26 dB, C3 -2.37 dB: on
# those two the denoised 4-spp frame does NOT reach the raw 16-spp frame at these sizes (profiles/r03_denoise.md)
@pytest.mark.parametrize("name,size,margin", [("earth_emitter", (400, 200), 0.0), ("book1_final", (320, 180), -1.5),
                                              ("perlin_motion", (300, 150), -2.6)])
def test_denoised_quality_against_reference_kernel(ctx, gpu_golden, scene_descs, name, size, margin):
    """Against the reference kernel's 4096-spp frame: the denoised 4-spp frame against the raw 16-spp frame (see the
    margins above), and on textured pixels (large local albedo gradient) at least as close as the raw 4-spp frame."""
    w, h = size
    ref = gpu_golden[f"{name}_fb_{w}x{h}x4096"]
    sc = rt.Scene(ctx, scene_descs[name])
    raw4, _ = sc.render(rt.default_params(width=w, height=h, spp=4))
    raw16, _ = sc.render(rt.default_params(width=w, height=h, spp=16))
    den4, _ = sc.render_denoised(rt.default_params(width=w, height=h, spp=4))
    feats = _features(ctx, sc, rt.default_params(width=w, height=h), rt.default_denoise_params().feature_spp).cpu().numpy()
    m = _texture_mask(feats)  # frames and features share the layout (row 0 = bottom)
    p4, p16, pd = rt.psnr(raw4, ref), rt.psnr(raw16, ref), rt.psnr(den4, ref)
    t4, td = rt.psnr(raw4[m], ref[m]), rt.psnr(den4[m], ref[m])
    record_parity("denoise_quality_vs_reference_kernel", scene=name, size=f"{w}x{h}", psnr_raw4=p4, psnr_raw16=p16, psnr_denoised4=pd,
                  texture_fraction=float(m.mean()), texture_psnr_raw4=t4, texture_psnr_denoised4=td)
    assert pd > p4 + 2.0, (pd, p4)
    assert pd >= p16 + margin, (pd, p16, p4)
    assert td >= t4, (td, t4)


def test_denoised_render_is_deterministic_and_composed_of_the_device_entries(ctx, scene_descs):
    """One sample per pixel: the render's accumulator is then free of the order of float atomics, so every stage after it
    must reproduce its bits."""
    import torch

    sc = rt.Scene(ctx, scene_descs["book1_final"])
    w, h = 160, 90
    p = rt.default_params(width=w, height=h, spp=1)
    before, _ = sc.render(p)
    a, st = sc.render_denoised(p)
    b, _ = sc.render_denoised(p)
    after, _ = sc.render(p)
    assert a.tobytes() == b.tobytes() and before.tobytes() == after.tobytes()
    assert st.paths == w * h and st.ms_tonemap > 0.0
    acc = torch.zeros((h, w, 4), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    sc.render_accum_device(p, acc.data_ptr())
    feat = _features(ctx, sc, p, rt.default_denoise_params().feature_spp)
    c, _ = _denoise(ctx, acc, feat, w, h, rt.default_denoise_params())
    assert c.tobytes() == a.tobytes()


def test_invalid_arguments_are_rejected(ctx, scene_descs):
    import torch

    lib = ctx.lib
    sc = rt.Scene(ctx, scene_descs["earth_emitter"])
    p = rt.default_params(width=32, height=16, spp=1)
    buf = torch.zeros((2, 16, 32, 4), dtype=torch.float32, device="cuda")
    out = np.empty((16, 32, 3), np.float32)
    ptr = C.c_void_p(buf.data_ptr())
    ok = rt.default_denoise_params()
    bad = [dict(iterations=-1), dict(iterations=9), dict(feature_spp=0), dict(sigma_color=0.0), dict(sigma_normal=-1.0),
           dict(sigma_depth=float("inf")), dict(sigma_albedo=float("nan"))]
    for kw in bad:
        d = rt.default_denoise_params(**kw)
        assert lib.rt_denoise_device(ctx._h, ptr, ptr, 32, 16, C.byref(d), ptr, None) == capi.RT_ERR_INVALID_ARG, kw
        assert lib.rt_render_denoised(ctx._h, sc._h, C.byref(p), C.byref(d), out.ctypes.data, None) == capi.RT_ERR_INVALID_ARG, kw
    calls = [
        lambda: lib.rt_denoise_device(None, ptr, ptr, 32, 16, C.byref(ok), ptr, None),
        lambda: lib.rt_denoise_device(ctx._h, None, ptr, 32, 16, C.byref(ok), ptr, None),
        lambda: lib.rt_denoise_device(ctx._h, ptr, None, 32, 16, C.byref(ok), ptr, None),
        lambda: lib.rt_denoise_device(ctx._h, ptr, ptr, 0, 16, C.byref(ok), ptr, None),
        lambda: lib.rt_denoise_device(ctx._h, ptr, ptr, 32, -1, C.byref(ok), ptr, None),
        lambda: lib.rt_denoise_device(ctx._h, ptr, ptr, 32, 16, None, ptr, None),
        lambda: lib.rt_denoise_device(ctx._h, ptr, ptr, 32, 16, C.byref(ok), None, None),
        lambda: lib.rt_render_features_device(None, sc._h, C.byref(p), 4, ptr),
        lambda: lib.rt_render_features_device(ctx._h, None, C.byref(p), 4, ptr),
        lambda: lib.rt_render_features_device(ctx._h, sc._h, None, 4, ptr),
        lambda: lib.rt_render_features_device(ctx._h, sc._h, C.byref(p), 0, ptr),
        lambda: lib.rt_render_features_device(ctx._h, sc._h, C.byref(p), 4, None),
        lambda: lib.rt_render_features_device(ctx._h, sc._h, C.byref(rt.default_params(width=0)), 4, ptr),
        lambda: lib.rt_render_denoised(None, sc._h, C.byref(p), C.byref(ok), out.ctypes.data, None),
        lambda: lib.rt_render_denoised(ctx._h, None, C.byref(p), C.byref(ok), out.ctypes.data, None),
        lambda: lib.rt_render_denoised(ctx._h, sc._h, None, C.byref(ok), out.ctypes.data, None),
        lambda: lib.rt_render_denoised(ctx._h, sc._h, C.byref(p), None, out.ctypes.data, None),
        lambda: lib.rt_render_denoised(ctx._h, sc._h, C.byref(p), C.byref(ok), None, None),
        lambda: lib.rt_render_denoised(ctx._h, sc._h, C.byref(rt.default_params(height=-4)), C.byref(ok), out.ctypes.data, None),
    ]
    for k, call in enumerate(calls):
        assert call() == capi.RT_ERR_INVALID_ARG, k


def test_app_denoise_matches_the_binding(ctx, tmp_path):
    exe = ROOT / "apps" / "render_scene"
    out = tmp_path / "f.ppm"
    subprocess.check_call([str(exe), "--scene", "earth_emitter", "--width", "300", "--height", "150", "--spp", "4", "--denoise",
                           "--out", str(out), "--earth", str(ROOT / "assets" / "earth_stb.ppm")], cwd=tmp_path)
    raw = out.read_bytes()
    got = np.frombuffer(raw[raw.index(b"255\n") + 4:], np.uint8).reshape(150, 300, 3)
    from raytracing_renderer_cuda_b200.assets import load_earth

    img, _ = rt.Scene(ctx, rt.SceneDesc.builtin("earth_emitter", load_earth())).render_denoised(
        rt.default_params(width=300, height=150, spp=4))
    assert np.array_equal(got, rt.quantize_rgb8(img))
    r = subprocess.run([str(exe), "--scene", "earth_emitter", "--width", "64", "--height", "32", "--spp", "4", "--denoise", "--gpus", "2",
                        "--out", str(tmp_path / "g.ppm")], capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode != 0 and "--denoise" in (r.stdout + r.stderr)
