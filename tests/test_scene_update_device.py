"""Scene updates from device memory without a device: the exported entry, the NULL checks that run before any device work,
and the rt_sphere records sphere_records builds."""
import ctypes as C

import numpy as np
import pytest

import raytracing_renderer_cuda_b200 as rt
from raytracing_renderer_cuda_b200 import capi


def test_device_update_entry_is_exported():
    lib = capi.load_library()
    assert "rt_scene_update_device" in capi.EXPORTED_SYMBOLS and hasattr(lib, "rt_scene_update_device")
    assert rt.Scene.update_device.__doc__


@pytest.mark.parametrize("n", [0, 3])
def test_null_arguments_are_rejected_before_any_device_work(n):
    lib = capi.load_library()
    ms = C.c_float(-1.0)
    bogus = C.c_void_p(0x1000)  # never dereferenced: the NULL check of another argument comes first
    cases = [(None, bogus, bogus, bogus), (bogus, None, bogus, bogus), (None, None, None, None)]
    if n:  # NULL record pointers are an error only when there are records
        cases += [(bogus, bogus, None, bogus), (bogus, bogus, bogus, None), (bogus, bogus, None, None)]
    for ctx, scene, idx, sph in cases:
        ms.value = -1.0
        assert lib.rt_scene_update_device(ctx, scene, idx, sph, n, C.byref(ms)) == capi.RT_ERR_INVALID_ARG
        assert b"NULL" in lib.rt_last_error()
        assert ms.value == 0.0


def test_sphere_records_lay_out_the_fields_of_rt_sphere():
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(1)
    n = 5
    c0 = rng.normal(size=(n, 3)).astype(np.float32)
    c1 = rng.normal(size=(n, 3)).astype(np.float32)
    r = rng.uniform(0.1, 2.0, n).astype(np.float32)
    t1 = rng.uniform(1.0, 2.0, n).astype(np.float32)
    mat = np.arange(n, dtype=np.int64) + 7
    ids = np.array([0, 1, 2**31 - 1, 2**31, 2**32 - 1], np.int64)

    want = np.zeros(n, capi.SPHERE_DTYPE)
    want["center0"], want["radius"], want["center1"] = c0, r, c1
    want["time0"], want["time1"] = 0.25, t1
    want["material"], want["id"], want["flags"] = mat, ids, capi.RT_SPHERE_MOVING
    got = capi.sphere_records(torch.from_numpy(c0), torch.from_numpy(r), torch.from_numpy(c1), 0.25, torch.from_numpy(t1),
                              torch.from_numpy(mat), torch.from_numpy(ids))
    assert got.dtype == torch.float32 and tuple(got.shape) == (n, 12) and got.device.type == "cpu"
    assert got.numpy().tobytes() == want.tobytes()

    # static spheres: center1 = center0, flags 0; scalar fields broadcast; flags given explicitly win
    want = np.zeros(n, capi.SPHERE_DTYPE)
    want["center0"] = want["center1"] = c0
    want["radius"], want["material"], want["id"] = 1.5, 3, 2**32 - 2
    got = capi.sphere_records(torch.from_numpy(c0), 1.5, material=3, id=2**32 - 2)
    assert got.numpy().tobytes() == want.tobytes()
    want["flags"] = capi.RT_SPHERE_INSIDE
    got = capi.sphere_records(torch.from_numpy(c0), 1.5, material=3, id=2**32 - 2, flags=capi.RT_SPHERE_INSIDE)
    assert got.numpy().tobytes() == want.tobytes()


def test_update_device_refuses_tensors_of_the_wrong_kind_before_the_call():
    torch = pytest.importorskip("torch")

    class _Scene(rt.Scene):  # no context, no scene: only the argument checks of the binding run
        def __init__(self):
            self.ctx = type("Ctx", (), {"device": 0})()
            self.lib = None

    sc = _Scene()
    idx = torch.zeros(2, dtype=torch.int32)
    rec = torch.zeros((2, 12), dtype=torch.float32)
    with pytest.raises(TypeError):
        sc.update_device(np.zeros(2, np.uint32), rec)
    with pytest.raises(TypeError):
        sc.update_device(idx.to(torch.int64), rec)
    with pytest.raises(TypeError):
        sc.update_device(idx, rec.to(torch.float64))
    with pytest.raises(ValueError):
        sc.update_device(idx, rec[:, :11])
    with pytest.raises(ValueError):
        sc.update_device(idx, torch.zeros((3, 12), dtype=torch.float32))
    with pytest.raises(ValueError):
        sc.update_device(idx, torch.zeros((2, 12), dtype=torch.uint8))
    with pytest.raises(ValueError):  # a CPU tensor is not on the context's device
        sc.update_device(idx, rec)
