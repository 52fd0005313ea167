"""Adaptive sampling on the B200: the error map against the numpy restatement (tests/test_adaptive.py), the threshold-0
and huge-threshold limits against uniform frames, every pixel of an adaptive frame against the uniform frame of its own
sample count (on every kernel granularity, the megakernel, emitter sampling and a ragged size), the two pipelines'
count maps, the quality against the reference kernel's 4096-spp frames, the denoiser on an adaptive accumulator,
argument checks and the C++ app's --adaptive."""
import ctypes as C
import subprocess

import numpy as np
import pytest

import raytracing_renderer_cuda_b200 as rt
from raytracing_renderer_cuda_b200 import capi
from tests.conftest import ROOT, record_parity
from tests.test_adaptive import error_map, window
from tests.test_denoise import atrous_reference

pytestmark = pytest.mark.gpu

HUGE = float(np.finfo(np.float32).max)


@pytest.fixture(scope="module")
def ctx():
    return rt.Context(0)


def _torch():
    import torch

    return torch


def _adaptive_device(ctx, sc, p, a):
    """(accumulator [H, W, 4], windowed error [H, W], passes, stats) of rt_render_adaptive_device."""
    torch = _torch()
    acc = torch.full((p.height, p.width, 4), -1.0, dtype=torch.float32, device="cuda")  # written, not added to
    err = torch.empty((p.height, p.width), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    passes, st = sc.render_adaptive_device(p, a, acc.data_ptr(), err.data_ptr(), want_stats=True)
    ctx.synchronize()
    return acc.cpu().numpy(), err.cpu().numpy(), passes, st


def _error_device(ctx, planes):
    torch = _torch()
    _, h, w, _ = planes.shape
    dev = torch.from_numpy(np.ascontiguousarray(planes)).cuda()
    out = torch.empty((h, w), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    rt.adaptive_error_device(ctx, dev.data_ptr(), w, h, out.data_ptr())
    ctx.synchronize()
    return out.cpu().numpy()


def _assert_ulp(got, want, ulps=1):
    inf = np.isinf(want)
    assert np.array_equal(np.isinf(got), inf)
    g, w = got[~inf].astype(np.float32), want[~inf].astype(np.float32)
    dist = np.abs(g.view(np.int32).astype(np.int64) - w.view(np.int32).astype(np.int64))
    assert dist.max(initial=0) <= ulps, int(dist.max())


def test_error_map_of_rendered_planes_is_exact(ctx, scene_descs):
    sc = rt.Scene(ctx, scene_descs["earth_emitter"])
    w, h = 96, 48
    a, _ = sc.render_accum(rt.default_params(width=w, height=h, spp=6))
    b, _ = sc.render_accum(rt.default_params(width=w, height=h, spp=6, sample_offset=6))
    planes = np.stack([a, b])
    _assert_ulp(_error_device(ctx, planes), window(error_map(planes)))


@pytest.mark.parametrize("size", [(64, 32), (67, 31), (1, 1), (1, 9)])
def test_error_map_of_random_planes_with_empty_pixels_is_exact(ctx, size):
    w, h = size
    rng = np.random.default_rng(w * 100 + h)
    planes = np.empty((2, h, w, 4), np.float32)
    planes[..., 3] = rng.integers(1, 9, (2, h, w))
    planes[..., :3] = (rng.random((2, h, w, 3)) * 1.3 * planes[..., 3:4]).astype(np.float32)  # some means above 1
    planes[0][rng.random((h, w)) < 0.05] = 0.0
    planes[1][rng.random((h, w)) < 0.05] = 0.0
    _assert_ulp(_error_device(ctx, planes), window(error_map(planes)))


def test_threshold_zero_is_the_uniform_frame(ctx, scene_descs):
    sc = rt.Scene(ctx, scene_descs["earth_emitter"])
    w, h = 120, 60
    a = rt.default_adaptive_params(min_spp=4, step_spp=4, max_spp=12, threshold=0.0)
    got, spp, st, passes = sc.render_adaptive(rt.default_params(width=w, height=h), a)
    want, st_u = sc.render(rt.default_params(width=w, height=h, spp=12))
    assert passes == 3 and (spp == 12).all()
    assert st.paths == st_u.paths and st.rays == st_u.rays
    assert np.abs(got - want).max() < 2e-6
    # a threshold nothing reaches: one pass, the min_spp frame
    a.threshold = HUGE
    got, spp, st, passes = sc.render_adaptive(rt.default_params(width=w, height=h), a)
    want, st_u = sc.render(rt.default_params(width=w, height=h, spp=4))
    assert passes == 1 and (spp == 4).all() and st.paths == st_u.paths and st.rays == st_u.rays
    assert np.abs(got - want).max() < 2e-6
    acc, _, passes_d, st_d = _adaptive_device(ctx, sc, rt.default_params(width=w, height=h), a)
    assert passes_d == 1 and st_d.paths == st.paths and (acc[..., 3] == 4).all()


CASES = {  # name: (scene, size, extra render params)
    "c1_list_cta": ("earth_emitter", (96, 48), {}),
    "c2_bvh_warp": ("book1_final", (80, 45), {}),
    "c3_bvh_warp": ("perlin_motion", (80, 40), {}),
    "spheres5000_pt": ("random_spheres", (64, 36), {}),
    "c1_megakernel": ("earth_emitter", (96, 48), {"pipeline": capi.RT_PIPE_MEGAKERNEL}),
    "c1_emitter_sampling": ("earth_emitter", (96, 48), {"flags": capi.RT_RENDER_EMITTER_SAMPLING}),
    "c2_emitter_sampling": ("book1_final", (80, 45), {"flags": capi.RT_RENDER_EMITTER_SAMPLING}),
    "c1_ragged": ("earth_emitter", (67, 31), {}),
}


def _scene(ctx, scene_descs, name):
    d = rt.SceneDesc.builtin("random_spheres", n=5000) if name == "random_spheres" else scene_descs[name]
    return rt.Scene(ctx, d)


def _mid():
    return rt.default_adaptive_params(min_spp=4, step_spp=4, max_spp=20, threshold=0.02)


@pytest.mark.parametrize("case", list(CASES))
def test_every_pixel_is_the_uniform_pixel_of_its_count(ctx, scene_descs, monkeypatch, case):
    name, (w, h), extra = CASES[case]
    sc = _scene(ctx, scene_descs, name)
    if name == "random_spheres":
        assert sc.info().n_spheres >= 4096  # the persistent-lane kernel
    a = _mid()
    p = rt.default_params(width=w, height=h, **extra)
    img, spp, st, passes = sc.render_adaptive(p, a)
    levels = np.unique(spp)
    assert ((levels - a.min_spp) % a.step_spp == 0).all() and levels.min() >= a.min_spp and levels.max() <= a.max_spp
    assert st.paths == int(spp.sum())
    assert len(levels) >= 2, levels  # the threshold splits the frame
    for c in levels:
        want, _ = sc.render(rt.default_params(width=w, height=h, spp=int(c), **extra))
        m = spp == c
        assert np.abs(img[m] - want[m]).max() < 2e-6, int(c)
    record_parity("adaptive_levels", case=case, size=f"{w}x{h}", passes=passes, mean_spp=float(spp.mean()),
                  levels=[int(c) for c in levels], frac_min=float((spp == a.min_spp).mean()))
    # The device entry gives the same counts.  (Two runs add a pixel's samples in a different order, so an error within
    # a few ulps of the threshold may decide differently: counts are compared on 99.9 % of the pixels.)
    acc, _, passes_d, st_d = _adaptive_device(ctx, sc, p, a)
    assert abs(passes_d - passes) <= 1 and (acc[..., 3].astype(np.int32) == spp).mean() >= 0.999
    if extra.get("pipeline") != capi.RT_PIPE_MEGAKERNEL and name != "random_spheres":
        # at these sizes nearly every pass ends in k_wf_tail (the persistent-lane kernel has no tail): switched off, the
        # same paths take more step launches
        monkeypatch.setenv("RT_WF_TAIL_PATHS", "0")
        img0, spp0, st0, _ = sc.render_adaptive(p, a)
        same = spp0 == spp
        assert same.mean() >= 0.999
        if same.all():
            assert st0.paths == st.paths and st0.rays == st.rays
        assert np.abs(img0[same] - img[same]).max() < 2e-6
        assert st.iterations < st0.iterations, (st.iterations, st0.iterations)


def test_pipelines_agree_on_the_count_map(ctx, scene_descs):
    sc = rt.Scene(ctx, scene_descs["earth_emitter"])
    w, h = 160, 80
    a = _mid()
    maps = {}
    for pipe in (capi.RT_PIPE_WAVEFRONT, capi.RT_PIPE_MEGAKERNEL):
        img, spp, st, _ = sc.render_adaptive(rt.default_params(width=w, height=h, pipeline=pipe), a)
        for c in np.unique(spp):  # each pixel still is the uniform pixel of its count
            want, _ = sc.render(rt.default_params(width=w, height=h, spp=int(c), pipeline=pipe))
            assert np.abs(img[spp == c] - want[spp == c]).max() < 2e-6
        maps[pipe] = spp
    agree = float((maps[capi.RT_PIPE_WAVEFRONT] == maps[capi.RT_PIPE_MEGAKERNEL]).mean())
    record_parity("adaptive_pipelines_agree", size=f"{w}x{h}", agree=agree)
    assert agree >= 0.999


# margin of PSNR(adaptive) over PSNR(uniform at the adaptive frame's mean spp, rounded up to even), against the reference
# kernel's 4096-spp frames, default adaptive parameters: about half of what a B200 measured (C1 +1.25 dB, C2 +0.94 dB,
# C3 +1.02 dB at mean 168 / 168 / 196 spp; profiles/r04_adaptive.md)
@pytest.mark.parametrize("name,size,margin", [("earth_emitter", (400, 200), 0.6), ("book1_final", (320, 180), 0.4),
                                              ("perlin_motion", (300, 150), 0.5)])
def test_adaptive_quality_against_reference_kernel(ctx, scene_descs, name, size, margin):
    gold = np.load(ROOT / "tests" / "golden" / "ref_gpu_golden.npz")
    w, h = size
    ref = gold[f"{name}_fb_{w}x{h}x4096"]
    sc = rt.Scene(ctx, scene_descs[name])
    a = rt.default_adaptive_params()
    img, spp, st, passes = sc.render_adaptive(rt.default_params(width=w, height=h), a)
    mean = float(spp.mean())
    s_uni = int(np.ceil(mean / 2) * 2)
    uni, _ = sc.render(rt.default_params(width=w, height=h, spp=s_uni))
    pa, pu = rt.psnr(img, ref), rt.psnr(uni, ref)
    record_parity("adaptive_quality_vs_reference_kernel", scene=name, size=f"{w}x{h}", mean_spp=mean, uniform_spp=s_uni,
                  passes=passes, frac_min=float((spp == a.min_spp).mean()), psnr_adaptive=pa, psnr_uniform=pu, margin=pa - pu)
    assert pa >= pu + margin, (pa, pu)


def test_denoiser_on_an_adaptive_accumulator(ctx, scene_descs):
    torch = _torch()
    sc = rt.Scene(ctx, scene_descs["earth_emitter"])
    w, h = 96, 48
    p = rt.default_params(width=w, height=h)
    acc, _, _, _ = _adaptive_device(ctx, sc, p, _mid())
    assert len(np.unique(acc[..., 3])) >= 2
    d = rt.default_denoise_params()
    feat = torch.zeros((2, h, w, 4), dtype=torch.float32, device="cuda")
    acc_dev = torch.from_numpy(acc).cuda()
    rgb = torch.empty((h, w, 3), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    sc.render_features_device(p, d.feature_spp, feat.data_ptr())
    rt.denoise_device(ctx, acc_dev.data_ptr(), feat.data_ptr(), w, h, d, rgb.data_ptr())
    ctx.synchronize()
    want = atrous_reference(acc, feat.cpu().numpy(), d)
    err = np.abs(rgb.cpu().numpy().astype(np.float64) ** 2 - want[..., :3])
    assert err.max() < 1e-4 and np.median(err) < 1e-6, (float(err.max()), float(np.median(err)))


def test_invalid_arguments_launch_nothing(ctx, scene_descs):
    torch = _torch()
    lib = ctx.lib
    sc = rt.Scene(ctx, scene_descs["earth_emitter"])
    w, h = 32, 16
    p = rt.default_params(width=w, height=h)
    acc = torch.full((h, w, 4), 7.0, dtype=torch.float32, device="cuda")
    err = torch.full((h, w), 7.0, dtype=torch.float32, device="cuda")
    out = np.empty((h, w, 3), np.float32)
    ptr, eptr = C.c_void_p(acc.data_ptr()), C.c_void_p(err.data_ptr())
    torch.cuda.synchronize()
    bad = [dict(min_spp=0), dict(min_spp=5), dict(step_spp=-2), dict(step_spp=3), dict(max_spp=18), dict(max_spp=2),
           dict(threshold=float("nan")), dict(threshold=-1.0)]
    for kw in bad:
        a = rt.default_adaptive_params(**kw)
        assert lib.rt_render_adaptive_device(ctx._h, sc._h, C.byref(p), C.byref(a), ptr, eptr, None, None) == capi.RT_ERR_INVALID_ARG, kw
        assert lib.rt_render_adaptive(ctx._h, sc._h, C.byref(p), C.byref(a), out.ctypes.data, None, None) == capi.RT_ERR_INVALID_ARG, kw
    ok = rt.default_adaptive_params()
    calls = [
        lambda: lib.rt_render_adaptive_device(None, sc._h, C.byref(p), C.byref(ok), ptr, eptr, None, None),
        lambda: lib.rt_render_adaptive_device(ctx._h, None, C.byref(p), C.byref(ok), ptr, eptr, None, None),
        lambda: lib.rt_render_adaptive_device(ctx._h, sc._h, None, C.byref(ok), ptr, eptr, None, None),
        lambda: lib.rt_render_adaptive_device(ctx._h, sc._h, C.byref(p), None, ptr, eptr, None, None),
        lambda: lib.rt_render_adaptive_device(ctx._h, sc._h, C.byref(p), C.byref(ok), None, eptr, None, None),
        lambda: lib.rt_render_adaptive(ctx._h, sc._h, C.byref(p), C.byref(ok), None, None, None),
        lambda: lib.rt_adaptive_error_device(ctx._h, None, w, h, eptr),
        lambda: lib.rt_adaptive_error_device(ctx._h, ptr, w, h, None),
        lambda: lib.rt_adaptive_error_device(ctx._h, ptr, 0, h, eptr),
    ]
    for k, call in enumerate(calls):
        assert call() == capi.RT_ERR_INVALID_ARG, k
    ctx.synchronize()
    assert (acc.cpu().numpy() == 7.0).all() and (err.cpu().numpy() == 7.0).all()


def _run_app(tmp_path, *args):
    exe = ROOT / "apps" / "render_scene"
    return subprocess.run([str(exe), "--scene", "earth_emitter", "--earth", str(ROOT / "assets" / "earth_stb.ppm"), *args],
                          capture_output=True, text=True, cwd=tmp_path)


def _ppm(path):
    raw = path.read_bytes()
    head = raw.split(b"\n", 3)
    w, h = map(int, head[1].split())
    return np.frombuffer(head[3], np.uint8).reshape(h, w, 3)


def test_app_adaptive_matches_the_binding(ctx, tmp_path):
    from raytracing_renderer_cuda_b200.assets import load_earth

    sc = rt.Scene(ctx, rt.SceneDesc.builtin("earth_emitter", load_earth()))
    # threshold 0: the count map is fixed (every pixel 2, 4, ..., 32 samples, the default cap 16 x --spp), so the file is
    # the binding's frame through rt_write_jpg byte for byte
    out = tmp_path / "a.jpg"
    r = _run_app(tmp_path, "--width", "200", "--height", "100", "--spp", "2", "--adaptive", "0", "--out", str(out))
    assert r.returncode == 0 and "16 passes" in r.stdout and "mean 32.00 samples per pixel" in r.stdout, (r.stdout, r.stderr)
    img, _, _, _ = sc.render_adaptive(rt.default_params(width=200, height=100),
                                      rt.default_adaptive_params(min_spp=2, step_spp=2, max_spp=32, threshold=0.0))
    assert out.read_bytes() == capi.jpeg_encode(ctx, rt.quantize_rgb8(img), 100)
    # a threshold between: the same frame, up to pixels whose error lies within float-addition order of the threshold
    r = _run_app(tmp_path, "--width", "200", "--height", "100", "--spp", "4", "--adaptive", "0.02", "--max-spp", "20", "--out",
                 str(tmp_path / "b.ppm"))
    assert r.returncode == 0, r.stderr
    img, _, _, passes = sc.render_adaptive(rt.default_params(width=200, height=100),
                                           rt.default_adaptive_params(min_spp=4, step_spp=4, max_spp=20, threshold=0.02))
    assert f"{passes} passes" in r.stdout
    assert (_ppm(tmp_path / "b.ppm") == rt.quantize_rgb8(img)).all(axis=2).mean() >= 0.999
    r = _run_app(tmp_path, "--width", "64", "--height", "32", "--spp", "4", "--adaptive", "0.02", "--denoise", "--out", str(tmp_path / "c.ppm"))
    assert r.returncode == 0 and "denoised" in r.stdout, r.stderr
    assert (tmp_path / "c.ppm").stat().st_size > 64 * 32 * 3
    for extra in (["--gpus", "2"], ["--passes", "3"]):
        r = _run_app(tmp_path, "--width", "64", "--height", "32", "--spp", "4", "--adaptive", "0.02", *extra, "--out", str(tmp_path / "d.ppm"))
        assert r.returncode != 0 and "--adaptive" in (r.stdout + r.stderr)
