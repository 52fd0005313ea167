"""Scene updates without a device: the exported entries, the rt_scene_edit layout against the binding, and the NULL checks
that run before any device work."""
import ctypes as C

import numpy as np

import raytracing_renderer_cuda_b200 as rt
from raytracing_renderer_cuda_b200 import capi


def test_update_entries_are_exported():
    lib = capi.load_library()
    for name in ("rt_scene_update", "rt_multi_update_scene"):
        assert name in capi.EXPORTED_SYMBOLS and hasattr(lib, name)


def test_scene_edit_layout_matches_the_binding():
    lib = capi.load_library()
    assert lib.rt_abi_sizeof(b"rt_scene_edit") == C.sizeof(capi.rt_scene_edit)
    # the C declaration: pointer, pointer, uint32 (padded), pointer, pointer, uint32 (padded), pointer
    p = C.sizeof(C.c_void_p)
    want = {"sphere_index": 0, "spheres": p, "n_spheres": 2 * p, "material_index": 3 * p, "materials": 4 * p, "n_materials": 5 * p,
            "camera": 6 * p}
    assert {f: getattr(capi.rt_scene_edit, f).offset for f, _ in capi.rt_scene_edit._fields_} == want
    assert C.sizeof(capi.rt_scene_edit) == 7 * p


def test_null_arguments_are_rejected_before_any_device_work():
    lib = capi.load_library()
    edit = capi.rt_scene_edit()
    ms = C.c_float(-1.0)
    bogus = C.c_void_p(0x1000)  # never dereferenced: the NULL check of another argument comes first
    for ctx, scene, e in ((None, bogus, C.byref(edit)), (bogus, None, C.byref(edit)), (bogus, bogus, None), (None, None, None)):
        assert lib.rt_scene_update(ctx, scene, e, C.byref(ms)) == capi.RT_ERR_INVALID_ARG
        assert b"NULL" in lib.rt_last_error()
        assert ms.value == 0.0
    assert lib.rt_multi_update_scene(None, C.byref(edit)) == capi.RT_ERR_INVALID_ARG
    assert lib.rt_multi_update_scene(bogus, None) == capi.RT_ERR_INVALID_ARG


def test_edit_builder_points_at_its_arrays():
    sph = np.zeros(3, capi.SPHERE_DTYPE)
    sph["radius"] = [1.0, 2.0, 3.0]
    mats = [capi.rt_material(capi.RT_MAT_METAL, -1, (0.5, 0.5, 0.5), 0.1)]
    cam = capi.rt_camera((1.0, 2.0, 3.0), (0.0, 0.0, 0.0), (0.0, 1.0, 0.0), 20.0, 2.0, 0.0, 10.0, 0.0, 1.0)
    edit, keep = capi.scene_edit([4, 0, 2], sph, [1], mats, cam)
    assert edit.n_spheres == 3 and edit.n_materials == 1
    assert [edit.sphere_index[k] for k in range(3)] == [4, 0, 2]
    assert [edit.spheres[k].radius for k in range(3)] == [1.0, 2.0, 3.0]
    assert edit.material_index[0] == 1 and edit.materials[0].kind == capi.RT_MAT_METAL
    assert list(edit.camera.contents.lookfrom) == [1.0, 2.0, 3.0]
    empty, _ = capi.scene_edit()
    assert empty.n_spheres == 0 and empty.n_materials == 0 and not empty.camera
    assert rt.Scene.update.__doc__
