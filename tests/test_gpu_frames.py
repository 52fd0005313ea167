"""Frame sequences on the B200: every frame of a batch against the single render of a scene whose camera is that frame's
camera, with the frame's sample offset (on every kernel granularity, the megakernel, emitter sampling, with and without the
tail kernel, a ragged size, one frame, and batches of many small frames), a motion sequence of perlin_motion, the device
entry adding into its accumulator, the host entry against rt_render, argument checks and the C++ app's --frames."""
import ctypes as C
import subprocess

import numpy as np
import pytest

import raytracing_renderer_cuda_b200 as rt
from raytracing_renderer_cuda_b200 import capi
from tests.conftest import ROOT

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    return rt.Context(0)


def _torch():
    import torch

    return torch


def _fresh_desc(name, earth):
    """A builtin description of the test's own: its camera is overwritten frame by frame (rt_scene_create copies it)."""
    if name == "earth_emitter":
        return rt.SceneDesc.builtin(name, earth)
    if name == "random_spheres":
        return rt.SceneDesc.builtin(name, n=5000)
    return rt.SceneDesc.builtin(name)


def _frames_device(ctx, sc, p, cams, prefill=None):
    """(accumulators [K, H, W, 4], stats) of rt_render_frames_device into a zeroed (or prefilled) device buffer."""
    torch = _torch()
    shape = (len(cams), p.height, p.width, 4)
    acc = torch.zeros(shape, dtype=torch.float32, device="cuda") if prefill is None else torch.from_numpy(prefill).cuda()
    torch.cuda.synchronize()
    st = sc.render_frames_device(p, cams, acc.data_ptr(), want_stats=True)
    ctx.synchronize()
    return acc.cpu().numpy(), st


def _singles(ctx, desc, p, cams):
    """Frame f rendered alone: a scene whose camera is cams[f], samples from p.sample_offset + f * p.spp."""
    accs, rays, saved = [], 0, capi.rt_camera.from_buffer_copy(desc.desc.camera)
    for f, cam in enumerate(cams):
        desc.desc.camera = cam
        sc = rt.Scene(ctx, desc)
        q = capi.rt_render_params.from_buffer_copy(p)
        q.sample_offset = p.sample_offset + f * p.spp
        acc, st = sc.render_accum(q)
        sc.close()
        accs.append(acc)
        rays += st.rays
    desc.desc.camera = saved
    return np.stack(accs), rays


def _assert_same_frames(got, want):
    assert np.array_equal(got[..., 3], want[..., 3])
    assert np.allclose(got, want, rtol=1e-5, atol=1e-5), float(np.abs(got - want).max())


CASES = {  # name: (scene, size, spp, frames, orbit degrees, extra render params)
    "c1_list_cta": ("earth_emitter", (96, 48), 4, 3, 30.0, {}),
    "c2_bvh_warp": ("book1_final", (80, 45), 4, 3, 30.0, {}),
    "spheres5000_pt": ("random_spheres", (64, 36), 4, 3, 30.0, {}),
    "c1_megakernel": ("earth_emitter", (96, 48), 4, 3, 30.0, {"pipeline": capi.RT_PIPE_MEGAKERNEL}),
    "c1_emitter_sampling": ("earth_emitter", (96, 48), 4, 3, 30.0, {"flags": capi.RT_RENDER_EMITTER_SAMPLING}),
    "c2_emitter_sampling": ("book1_final", (80, 45), 4, 3, 30.0, {"flags": capi.RT_RENDER_EMITTER_SAMPLING}),
    "c1_ragged": ("earth_emitter", (67, 31), 4, 3, 30.0, {}),
    "c1_one_frame": ("earth_emitter", (96, 48), 4, 1, 30.0, {}),
    # 40 frames of 64x32x2: every generation of the pool holds paths of many frames
    "c1_many_small_frames": ("earth_emitter", (64, 32), 2, 40, 90.0, {}),
    "c2_many_small_frames": ("book1_final", (64, 32), 2, 40, 90.0, {}),
}


@pytest.mark.parametrize("tail", ["default", "0"])
@pytest.mark.parametrize("case", list(CASES))
def test_batch_equals_the_single_frames(ctx, earth, monkeypatch, case, tail):
    name, (w, h), spp, k, degrees, extra = CASES[case]
    if tail == "0":
        if extra.get("pipeline") == capi.RT_PIPE_MEGAKERNEL or name == "random_spheres":
            pytest.skip("no tail kernel on this path")
        monkeypatch.setenv("RT_WF_TAIL_PATHS", "0")
    desc = _fresh_desc(name, earth)
    sc = rt.Scene(ctx, desc)
    if name == "random_spheres":
        assert sc.info().n_spheres >= 4096  # the persistent-lane kernel
    p = rt.default_params(width=w, height=h, spp=spp, sample_offset=3, **extra)
    cams = rt.orbit_cameras(desc.desc.camera, k, degrees)
    got, st = _frames_device(ctx, sc, p, cams)
    want, rays = _singles(ctx, desc, p, cams)
    assert (got[..., 3] == spp).all()
    _assert_same_frames(got, want)
    assert st.paths == w * h * spp * k and st.rays == rays
    if k > 1:
        assert not np.array_equal(got[0], got[1])


def test_motion_sequence_of_a_still_camera(ctx, earth):
    desc = _fresh_desc("perlin_motion", earth)
    sc = rt.Scene(ctx, desc)
    base = desc.desc.camera
    assert base.time1 > base.time0  # the moving spheres move within the shutter
    p = rt.default_params(width=80, height=40, spp=8)
    cams = rt.orbit_cameras(base, 3, 0.0)
    assert all(list(c.lookfrom) == list(base.lookfrom) for c in cams)
    got, st = _frames_device(ctx, sc, p, cams)
    want, rays = _singles(ctx, desc, p, cams)
    _assert_same_frames(got, want)
    assert st.rays == rays
    for a in range(3):
        for b in range(a + 1, 3):
            assert not np.allclose(got[a], got[b])


def test_device_entry_adds_into_the_accumulator(ctx, scene_descs):
    sc = rt.Scene(ctx, scene_descs["earth_emitter"])
    p = rt.default_params(width=64, height=32, spp=4)
    cams = rt.orbit_cameras(scene_descs["earth_emitter"].desc.camera, 3, 20.0)
    rng = np.random.default_rng(7)
    prefill = np.empty((3, 32, 64, 4), np.float32)
    prefill[..., :3] = rng.random((3, 32, 64, 3), dtype=np.float32)
    prefill[..., 3] = rng.integers(1, 5, (3, 32, 64))
    batch, _ = _frames_device(ctx, sc, p, cams)
    got, _ = _frames_device(ctx, sc, p, cams, prefill=prefill)
    assert np.array_equal(got[..., 3], prefill[..., 3] + batch[..., 3])
    assert np.allclose(got, prefill + batch, rtol=1e-5, atol=1e-5)


def test_host_entry_equals_rt_render_per_frame(ctx, earth):
    desc = _fresh_desc("book1_final", earth)
    sc = rt.Scene(ctx, desc)
    p = rt.default_params(width=80, height=45, spp=4, sample_offset=5)
    cams = rt.orbit_cameras(desc.desc.camera, 4, 60.0)
    rgb, st = sc.render_frames(p, cams)
    assert rgb.shape == (4, 45, 80, 3) and st.paths == 80 * 45 * 4 * 4 and st.ms_tonemap > 0
    for f, cam in enumerate(cams):
        desc.desc.camera = cam
        one = rt.Scene(ctx, desc)
        want, _ = one.render(rt.default_params(width=80, height=45, spp=4, sample_offset=5 + 4 * f))
        one.close()
        assert np.allclose(rgb[f], want, rtol=1e-5, atol=1e-5), f


def test_zero_spp_adds_nothing(ctx, scene_descs):
    sc = rt.Scene(ctx, scene_descs["earth_emitter"])
    cams = rt.orbit_cameras(scene_descs["earth_emitter"].desc.camera, 2, 10.0)
    prefill = np.full((2, 8, 16, 4), 0.5, np.float32)
    got, st = _frames_device(ctx, sc, rt.default_params(width=16, height=8, spp=0), cams, prefill=prefill)
    assert np.array_equal(got, prefill) and st.paths == 0 and st.rays == 0


def test_invalid_arguments_leave_the_buffers_untouched(ctx, scene_descs):
    torch = _torch()
    lib = capi.load_library()
    sc = rt.Scene(ctx, scene_descs["earth_emitter"])
    p = rt.default_params(width=16, height=8, spp=4)
    cams = (capi.rt_camera * 3)(*rt.orbit_cameras(scene_descs["earth_emitter"].desc.camera, 3, 10.0))
    nan_cams = (capi.rt_camera * 3)(*cams)
    nan_cams[1].lookat[0] = float("nan")
    overflow = rt.default_params(width=16, height=8, spp=1 << 29, sample_offset=(1 << 29) + 1)
    acc = torch.full((3, 8, 16, 4), 7.0, dtype=torch.float32, device="cuda")
    out = np.full((3, 8, 16, 3), 7.0, np.float32)
    torch.cuda.synchronize()
    bad = [(C.byref(p), nan_cams, 3), (C.byref(p), cams, 0), (C.byref(overflow), cams, 3), (C.byref(p), None, 3), (None, cams, 3)]
    for k, (params, cameras, n) in enumerate(bad):
        assert lib.rt_render_frames_device(ctx._h, sc._h, params, cameras, n, C.c_void_p(acc.data_ptr()), None) == capi.RT_ERR_INVALID_ARG, k
        assert lib.rt_render_frames(ctx._h, sc._h, params, cameras, n, out.ctypes.data, None) == capi.RT_ERR_INVALID_ARG, k
    assert lib.rt_render_frames_device(ctx._h, sc._h, C.byref(p), cams, 3, None, None) == capi.RT_ERR_INVALID_ARG
    assert lib.rt_render_frames(ctx._h, sc._h, C.byref(p), cams, 3, None, None) == capi.RT_ERR_INVALID_ARG
    ctx.synchronize()
    assert (acc == 7.0).all().item() and (out == 7.0).all()
    with pytest.raises(capi.RtError):
        sc.render_frames(p, list(nan_cams))


def _run_app(tmp_path, *args):
    exe = ROOT / "apps" / "render_scene"
    return subprocess.run([str(exe), "--scene", "earth_emitter", "--earth", str(ROOT / "assets" / "earth_stb.ppm"), *args],
                          capture_output=True, text=True, cwd=tmp_path)


def _ppm(path):
    raw = path.read_bytes()
    head = raw.split(b"\n", 3)
    w, h = map(int, head[1].split())
    return np.frombuffer(head[3], np.uint8).reshape(h, w, 3)


def test_app_frames_match_the_binding(ctx, scene_descs, tmp_path):
    desc = scene_descs["earth_emitter"]
    sc = rt.Scene(ctx, desc)
    r = _run_app(tmp_path, "--width", "96", "--height", "48", "--spp", "4", "--frames", "3", "--orbit", "30", "--out",
                 str(tmp_path / "seq.ppm"))
    assert r.returncode == 0 and "3 frames" in r.stdout, (r.stdout, r.stderr)
    rgb, _ = sc.render_frames(rt.default_params(width=96, height=48, spp=4), rt.orbit_cameras(desc.desc.camera, 3, 30.0))
    for f in range(3):
        # float sums in another order may move a channel across a quantisation step in a rare pixel
        assert (_ppm(tmp_path / f"seq_{f:04d}.ppm") == rt.quantize_rgb8(rgb[f])).all(axis=2).mean() >= 0.999, f
    assert not (tmp_path / "seq_0003.ppm").exists()
    r = _run_app(tmp_path, "--width", "96", "--height", "48", "--spp", "4", "--frames", "3", "--orbit", "30", "--out",
                 str(tmp_path / "seq.jpg"))
    assert r.returncode == 0, r.stderr
    for f in range(3):
        img, _ = capi.jpeg_decode(ctx, (tmp_path / f"seq_{f:04d}.jpg").read_bytes())
        assert img.shape == (48, 96, 3)
    for extra in (["--gpus", "2"], ["--passes", "3"], ["--denoise"], ["--adaptive", "0.1"]):
        r = _run_app(tmp_path, "--width", "64", "--height", "32", "--spp", "4", "--frames", "3", *extra, "--out", str(tmp_path / "x.ppm"))
        assert r.returncode != 0 and "--frames" in (r.stdout + r.stderr)
