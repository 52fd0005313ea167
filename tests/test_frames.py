"""Frame sequences without a device: rt_orbit_cameras against a numpy float64 restatement of its formula, its properties and
argument checks, the argument checks of rt_render_frames / rt_render_frames_device (which run before any device work) and
the ABI symbols."""
import ctypes as C

import numpy as np
import pytest

import raytracing_renderer_cuda_b200 as rt
from raytracing_renderer_cuda_b200 import capi


def _camera(lookfrom=(13.0, 2.0, 3.0), lookat=(0.0, 0.0, 0.0), up=(0.0, 1.0, 0.0), t0=0.0, t1=1.0):
    return capi.rt_camera(lookfrom, lookat, up, 20.0, 2.0, 0.1, 10.0, t0, t1)


def orbit_reference(base, n, degrees):
    """Frame k: lookfrom rotated by k * degrees / n about the axis through lookat along up (Rodrigues, right-hand rule), the
    shutter [t0 + k (t1 - t0) / n, t0 + (k + 1) (t1 - t0) / n]; float64 throughout, one rounding to float32 at the end."""
    lf, la, up = (np.array(v, np.float32).astype(np.float64) for v in (base.lookfrom, base.lookat, base.up))
    a = up / np.sqrt(np.sum(up * up))
    v = lf - la
    t0, t1 = np.float64(np.float32(base.time0)), np.float64(np.float32(base.time1))
    out = []
    for k in range(n):
        th = np.float64(np.float32(degrees)) * k / n * (np.pi / 180.0)
        c, s = np.cos(th), np.sin(th)
        vr = v * c + np.cross(a, v) * s + a * np.dot(a, v) * (1.0 - c)
        out.append((np.float32(la + vr), np.float32(t0 + (t1 - t0) * k / n), np.float32(t0 + (t1 - t0) * (k + 1) / n)))
    return out


def _f32(v):
    return np.array(v, np.float32)


@pytest.mark.parametrize("degrees", [0.0, 30.0, 360.0, -45.0, 720.0])
@pytest.mark.parametrize("n", [1, 3, 8, 32])
@pytest.mark.parametrize("up", [(0.0, 1.0, 0.0), (0.3, 2.0, -0.5)])
def test_orbit_matches_the_restatement(degrees, n, up):
    base = _camera(lookfrom=(13.0, 2.0, 3.0), lookat=(0.5, -0.25, 1.0), up=up, t0=0.25, t1=1.75)
    got = rt.orbit_cameras(base, n, degrees)
    want = orbit_reference(base, n, degrees)
    assert len(got) == n
    for cam, (lf, t0, t1) in zip(got, want):
        # (libm and numpy may round sin / cos of the same double differently in the last bit)
        assert np.allclose(_f32(cam.lookfrom), lf, rtol=0, atol=4e-6 * np.abs(lf).max())
        assert np.float32(cam.time0) == t0 and np.float32(cam.time1) == t1
        for field in ("lookat", "up"):
            assert np.array_equal(_f32(getattr(cam, field)), _f32(getattr(base, field)))
        for field in ("vfov", "aspect", "aperture", "focus_dist"):
            assert getattr(cam, field) == getattr(base, field)


def test_orbit_rotates_right_handed_about_up():
    got = rt.orbit_cameras(_camera(lookfrom=(1.0, 0.0, 0.0)), 4, 360.0)
    # +90 degrees about +y takes +x to -z
    assert np.allclose(_f32(got[1].lookfrom), (0.0, 0.0, -1.0), atol=1e-7)
    assert np.allclose(_f32(got[2].lookfrom), (-1.0, 0.0, 0.0), atol=1e-7)


def test_orbit_zero_degrees_keeps_lookfrom_and_distance_is_preserved():
    base = _camera(lookfrom=(13.0, 2.0, 3.0), lookat=(0.5, -0.25, 1.0), up=(0.3, 2.0, -0.5))
    for cam in rt.orbit_cameras(base, 7, 0.0):
        assert np.array_equal(_f32(cam.lookfrom), _f32(base.lookfrom))
    d0 = np.linalg.norm(_f32(base.lookfrom).astype(np.float64) - _f32(base.lookat))
    for cam in rt.orbit_cameras(base, 9, 250.0):
        d = np.linalg.norm(_f32(cam.lookfrom).astype(np.float64) - _f32(cam.lookat))
        assert abs(d - d0) <= 4e-7 * d0


@pytest.mark.parametrize("t0,t1,n", [(0.0, 1.0, 3), (0.25, 1.75, 7), (0.0, 0.0, 5), (1.0, 0.1, 6), (0.0, 1.0, 40)])
def test_orbit_shutter_windows_tile_the_base_window(t0, t1, n):
    cams = rt.orbit_cameras(_camera(t0=t0, t1=t1), n, 10.0)
    assert cams[0].time0 == np.float32(t0) and cams[-1].time1 == np.float32(t1)
    for a, b in zip(cams, cams[1:]):
        assert a.time1 == b.time0


def test_orbit_of_one_frame_is_the_base_camera():
    base = _camera(lookfrom=(13.0, 2.0, 3.0), lookat=(0.5, -0.25, 1.0), up=(0.3, 2.0, -0.5), t0=0.25, t1=1.75)
    (cam,) = rt.orbit_cameras(base, 1, 123.0)
    assert bytes(cam) == bytes(base)


def test_orbit_argument_checks():
    lib = capi.load_library()
    base = _camera()
    out = (capi.rt_camera * 4)()
    assert lib.rt_orbit_cameras(None, 4, 10.0, out) == capi.RT_ERR_INVALID_ARG
    assert lib.rt_orbit_cameras(C.byref(base), 4, 10.0, None) == capi.RT_ERR_INVALID_ARG
    for n in (0, -1):
        assert lib.rt_orbit_cameras(C.byref(base), n, 10.0, out) == capi.RT_ERR_INVALID_ARG
    for deg in (float("nan"), float("inf")):
        assert lib.rt_orbit_cameras(C.byref(base), 4, deg, out) == capi.RT_ERR_INVALID_ARG
    for bad in (_camera(up=(0.0, 0.0, 0.0)), _camera(lookfrom=(float("nan"), 0.0, 0.0)), _camera(t1=float("inf"))):
        assert lib.rt_orbit_cameras(C.byref(bad), 4, 10.0, out) == capi.RT_ERR_INVALID_ARG
    assert bytes(out) == bytes((capi.rt_camera * 4)())  # nothing written on a rejected call
    with pytest.raises(capi.RtError):
        rt.orbit_cameras(base, 0, 10.0)


def test_frame_entries_are_exported():
    lib = capi.load_library()
    for name in ("rt_render_frames_device", "rt_render_frames", "rt_orbit_cameras"):
        assert name in capi.EXPORTED_SYMBOLS and hasattr(lib, name)
    assert hasattr(rt.Scene, "render_frames") and hasattr(rt.Scene, "render_frames_device")


def test_bad_frame_arguments_are_rejected_before_any_device_work():
    """The argument checks run before the context or the scene is read: the dummy handles below are never dereferenced,
    so an invalid-argument status shows that nothing reached the device."""
    lib = capi.load_library()
    dummy = C.c_void_p(1)
    p = rt.default_params(width=16, height=8, spp=4)
    cams = (capi.rt_camera * 3)(*rt.orbit_cameras(_camera(), 3, 30.0))
    nan_cams = (capi.rt_camera * 3)(*cams)
    nan_cams[2].focus_dist = float("nan")
    out = np.zeros((3, 8, 16, 3), np.float32)

    def both(ctx, scene, params, cameras, n, buf):
        return (lib.rt_render_frames(ctx, scene, params, cameras, n, buf, None),
                lib.rt_render_frames_device(ctx, scene, params, cameras, n, buf, None))

    cases = [
        (None, dummy, C.byref(p), cams, 3, out.ctypes.data),
        (dummy, None, C.byref(p), cams, 3, out.ctypes.data),
        (dummy, dummy, None, cams, 3, out.ctypes.data),
        (dummy, dummy, C.byref(p), None, 3, out.ctypes.data),
        (dummy, dummy, C.byref(p), cams, 3, None),
        (dummy, dummy, C.byref(p), cams, 0, out.ctypes.data),
        (dummy, dummy, C.byref(p), cams, -2, out.ctypes.data),
        (dummy, dummy, C.byref(p), nan_cams, 3, out.ctypes.data),
        (dummy, dummy, C.byref(rt.default_params(width=0)), cams, 3, out.ctypes.data),
        (dummy, dummy, C.byref(rt.default_params(spp=-1)), cams, 3, out.ctypes.data),
        # samples [offset, offset + 3 * spp) must stay below 2^31
        (dummy, dummy, C.byref(rt.default_params(spp=1 << 29, sample_offset=(1 << 29) + 1)), cams, 3, out.ctypes.data),
        (dummy, dummy, C.byref(rt.default_params(spp=(1 << 30), sample_offset=0)), cams, 2, out.ctypes.data),
    ]
    for k, args in enumerate(cases):
        assert both(*args) == (capi.RT_ERR_INVALID_ARG, capi.RT_ERR_INVALID_ARG), k
    assert not out.any()
