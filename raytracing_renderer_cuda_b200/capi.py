"""ctypes binding of include/rt_api.h (librt_b200.so).

Test / bench orchestration only: the product is the shared library and the C++
facade in include/rt/.  Every structure below mirrors the C declaration of the
same name field by field; `check_layout()` compares sizes with the library's
own `rt_abi_sizeof` so a drifted binding fails loudly instead of corrupting memory.

There is no fallback: if the library is missing, or no sm_100 device is usable,
the calls raise.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import numpy as np

_PKG = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ["RT_B200_LIB"]) if os.environ.get("RT_B200_LIB") else _PKG / "librt_b200.so"  # override: A/B library variants

RT_INVALID_ID = 0xFFFFFFFF
RT_OK = 0
RT_ERR_INVALID_ARG, RT_ERR_CUDA, RT_ERR_OOM, RT_ERR_UNSUPPORTED, RT_ERR_NO_DEVICE, RT_ERR_IO = 1, 2, 3, 4, 5, 6
STATUS_NAMES = {0: "RT_OK", 1: "RT_ERR_INVALID_ARG", 2: "RT_ERR_CUDA", 3: "RT_ERR_OOM", 4: "RT_ERR_UNSUPPORTED",
                5: "RT_ERR_NO_DEVICE", 6: "RT_ERR_IO"}

RT_MAT_LAMBERTIAN, RT_MAT_METAL, RT_MAT_DIELECTRIC, RT_MAT_EMITTER = 0, 1, 2, 3
(RT_TEX_CONSTANT, RT_TEX_CHECKER, RT_TEX_NOISE_PERLIN, RT_TEX_NOISE_TURBULANCE, RT_TEX_NOISE_MARBLE, RT_TEX_WOOD,
 RT_TEX_IMAGE) = range(7)
RT_BVH_AUTO, RT_BVH_NONE, RT_BVH_HOST_SAH, RT_BVH_GPU_LBVH = 0, 1, 2, 3
RT_PIPE_AUTO, RT_PIPE_WAVEFRONT, RT_PIPE_MEGAKERNEL = 0, 1, 2
RT_RENDER_EMITTER_SAMPLING = 1  # rt_render_params.flags
RT_MAX_LIGHTS = 16
RT_SPHERE_MOVING, RT_SPHERE_INSIDE = 1, 2


class RtError(RuntimeError):
    def __init__(self, status: int, msg: str):
        super().__init__(f"{STATUS_NAMES.get(status, status)}: {msg}")
        self.status = status


class rt_sphere(C.Structure):
    _fields_ = [("center0", C.c_float * 3), ("radius", C.c_float), ("center1", C.c_float * 3), ("time0", C.c_float),
                ("time1", C.c_float), ("material", C.c_uint32), ("id", C.c_uint32), ("flags", C.c_uint32)]


class rt_material(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("texture", C.c_int32), ("albedo", C.c_float * 3), ("param", C.c_float)]


class rt_texture(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("even", C.c_int32), ("odd", C.c_int32), ("image", C.c_int32),
                ("color1", C.c_float * 3), ("color2", C.c_float * 3), ("density", C.c_float), ("hardness", C.c_float)]


class rt_jpeg_component(C.Structure):
    _fields_ = [("h", C.c_int32), ("v", C.c_int32), ("tq", C.c_int32), ("x", C.c_int32), ("y", C.c_int32), ("w2", C.c_int32),
                ("h2", C.c_int32), ("blocks_w", C.c_int32), ("blocks_h", C.c_int32), ("coeff", C.POINTER(C.c_int16))]


class rt_jpeg_coefficients(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("n_comp", C.c_int32), ("h_max", C.c_int32), ("v_max", C.c_int32),
                ("progressive", C.c_int32), ("is_rgb", C.c_int32), ("comp", rt_jpeg_component * 3), ("dequant", (C.c_uint16 * 64) * 4)]


class rt_image(C.Structure):
    _fields_ = [("rgb", C.POINTER(C.c_float)), ("width", C.c_int32), ("height", C.c_int32)]


class rt_camera(C.Structure):
    _fields_ = [("lookfrom", C.c_float * 3), ("lookat", C.c_float * 3), ("up", C.c_float * 3), ("vfov", C.c_float),
                ("aspect", C.c_float), ("aperture", C.c_float), ("focus_dist", C.c_float), ("time0", C.c_float),
                ("time1", C.c_float)]


class rt_scene_desc(C.Structure):
    _fields_ = [("spheres", C.POINTER(rt_sphere)), ("n_spheres", C.c_uint32),
                ("materials", C.POINTER(rt_material)), ("n_materials", C.c_uint32),
                ("textures", C.POINTER(rt_texture)), ("n_textures", C.c_uint32),
                ("images", C.POINTER(rt_image)), ("n_images", C.c_uint32),
                ("camera", rt_camera), ("bvh_mode", C.c_uint32)]


class rt_render_params(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("spp", C.c_int32), ("sample_offset", C.c_int32),
                ("max_depth", C.c_int32), ("seed", C.c_uint32), ("tmin", C.c_float), ("world", C.c_float * 3),
                ("bloom", C.c_float), ("pipeline", C.c_uint32), ("flags", C.c_uint32)]


class rt_stats(C.Structure):
    _fields_ = [("paths", C.c_uint64), ("rays", C.c_uint64), ("ms_total", C.c_float), ("ms_tonemap", C.c_float),
                ("ms_h2d", C.c_float), ("ms_d2h", C.c_float), ("launches", C.c_uint32), ("iterations", C.c_uint32)]


class rt_scene_info(C.Structure):
    _fields_ = [("n_spheres", C.c_uint32), ("n_nodes", C.c_uint32), ("bvh_mode", C.c_uint32), ("bvh_depth", C.c_uint32),
                ("ms_build", C.c_float), ("ms_upload", C.c_float), ("sah_cost", C.c_float),
                ("device_bytes", C.c_uint64)]


class rt_ray(C.Structure):
    _fields_ = [("origin", C.c_float * 3), ("direction", C.c_float * 3), ("time", C.c_float)]


class rt_hit(C.Structure):
    _fields_ = [("t", C.c_float), ("id", C.c_uint32), ("p", C.c_float * 3), ("n", C.c_float * 3), ("u", C.c_float),
                ("v", C.c_float)]


class rt_shade_sample(C.Structure):
    _fields_ = [("id", C.c_uint32), ("continues", C.c_uint32), ("t", C.c_float), ("emitted", C.c_float * 3),
                ("attenuation", C.c_float * 3), ("scattered", rt_ray)]


class rt_denoise_params(C.Structure):
    _fields_ = [("iterations", C.c_int32), ("feature_spp", C.c_int32), ("sigma_color", C.c_float), ("sigma_normal", C.c_float),
                ("sigma_depth", C.c_float), ("sigma_albedo", C.c_float)]


class rt_adaptive_params(C.Structure):
    _fields_ = [("min_spp", C.c_int32), ("step_spp", C.c_int32), ("max_spp", C.c_int32), ("threshold", C.c_float)]


RAY_DTYPE = np.dtype([("origin", "<f4", 3), ("direction", "<f4", 3), ("time", "<f4")])
HIT_DTYPE = np.dtype([("t", "<f4"), ("id", "<u4"), ("p", "<f4", 3), ("n", "<f4", 3), ("u", "<f4"), ("v", "<f4")])
SHADE_DTYPE = np.dtype([("id", "<u4"), ("continues", "<u4"), ("t", "<f4"), ("emitted", "<f4", 3), ("attenuation", "<f4", 3),
                        ("scattered", RAY_DTYPE)])
assert RAY_DTYPE.itemsize == C.sizeof(rt_ray) and HIT_DTYPE.itemsize == C.sizeof(rt_hit)
assert SHADE_DTYPE.itemsize == C.sizeof(rt_shade_sample)

# every symbol include/rt_api.h declares: name -> (restype, argtypes)
_VP = C.c_void_p
_SIGNATURES = {
    "rt_api_version": (C.c_int, []),
    "rt_abi_sizeof": (C.c_size_t, [C.c_char_p]),
    "rt_last_error": (C.c_char_p, []),
    "rt_default_render_params": (None, [C.POINTER(rt_render_params)]),
    "rt_context_create": (C.c_int, [C.c_int, C.POINTER(_VP)]),
    "rt_context_destroy": (None, [_VP]),
    "rt_context_set_stream": (C.c_int, [_VP, _VP]),
    "rt_context_synchronize": (C.c_int, [_VP]),
    "rt_scene_create": (C.c_int, [_VP, C.POINTER(rt_scene_desc), C.POINTER(_VP)]),
    "rt_scene_destroy": (None, [_VP]),
    "rt_scene_get_info": (C.c_int, [_VP, C.POINTER(rt_scene_info)]),
    "rt_trace_primary": (C.c_int, [_VP, _VP, _VP, C.c_size_t, C.c_float, C.c_int, _VP]),
    "rt_selftest_rz": (C.c_int, [_VP, _VP, _VP, C.c_size_t, _VP]),
    "rt_selftest_exclusive_sum": (C.c_int, [_VP, _VP, _VP, C.c_size_t, C.c_int32, C.c_int32, C.POINTER(C.c_int32)]),
    "rt_selftest_sort_pairs": (C.c_int, [_VP, _VP, _VP, C.c_size_t, C.c_int32, _VP, _VP, C.POINTER(C.c_int32),
                                         C.POINTER(C.c_int32)]),
    "rt_shade_probe": (C.c_int, [_VP, _VP, _VP, C.c_size_t, C.POINTER(rt_render_params), C.c_int, _VP]),
    "rt_render": (C.c_int, [_VP, _VP, C.POINTER(rt_render_params), _VP, C.POINTER(rt_stats)]),
    "rt_render_accum": (C.c_int, [_VP, _VP, C.POINTER(rt_render_params), _VP, C.POINTER(rt_stats)]),
    "rt_render_accum_device": (C.c_int, [_VP, _VP, C.POINTER(rt_render_params), _VP, C.POINTER(rt_stats)]),
    "rt_render_progressive": (C.c_int, [_VP, _VP, C.POINTER(rt_render_params), C.c_int32, _VP, _VP, _VP, C.POINTER(rt_stats)]),
    "rt_tonemap_device": (C.c_int, [_VP, _VP, C.c_int32, C.c_int32, _VP, _VP]),
    "rt_default_denoise_params": (None, [C.POINTER(rt_denoise_params)]),
    "rt_render_features_device": (C.c_int, [_VP, _VP, C.POINTER(rt_render_params), C.c_int32, _VP]),
    "rt_denoise_device": (C.c_int, [_VP, _VP, _VP, C.c_int32, C.c_int32, C.POINTER(rt_denoise_params), _VP, _VP]),
    "rt_render_denoised": (C.c_int, [_VP, _VP, C.POINTER(rt_render_params), C.POINTER(rt_denoise_params), _VP, C.POINTER(rt_stats)]),
    "rt_default_adaptive_params": (None, [C.POINTER(rt_adaptive_params)]),
    "rt_adaptive_error_device": (C.c_int, [_VP, _VP, C.c_int32, C.c_int32, _VP]),
    "rt_render_adaptive_device": (C.c_int, [_VP, _VP, C.POINTER(rt_render_params), C.POINTER(rt_adaptive_params), _VP, _VP,
                                            C.POINTER(C.c_int32), C.POINTER(rt_stats)]),
    "rt_render_adaptive": (C.c_int, [_VP, _VP, C.POINTER(rt_render_params), C.POINTER(rt_adaptive_params), _VP, _VP,
                                     C.POINTER(rt_stats)]),
    "rt_render_frames_device": (C.c_int, [_VP, _VP, C.POINTER(rt_render_params), C.POINTER(rt_camera), C.c_int32, _VP,
                                          C.POINTER(rt_stats)]),
    "rt_render_frames": (C.c_int, [_VP, _VP, C.POINTER(rt_render_params), C.POINTER(rt_camera), C.c_int32, _VP, C.POINTER(rt_stats)]),
    "rt_orbit_cameras": (C.c_int, [C.POINTER(rt_camera), C.c_int32, C.c_float, C.POINTER(rt_camera)]),
    "rt_reduce_tonemap_peers": (C.c_int, [_VP, C.POINTER(_VP), C.c_int32, _VP, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                          _VP, _VP, _VP]),
    "rt_shard_samples": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "rt_shard_rows": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "rt_multi_create": (C.c_int, [C.POINTER(C.c_int32), C.c_int32, C.POINTER(_VP)]),
    "rt_multi_size": (C.c_int32, [_VP]),
    "rt_multi_set_scene": (C.c_int, [_VP, C.POINTER(rt_scene_desc)]),
    "rt_multi_render": (C.c_int, [_VP, C.POINTER(rt_render_params), _VP, _VP, C.POINTER(rt_stats), C.POINTER(C.c_float)]),
    "rt_multi_read_accum": (C.c_int, [_VP, C.c_int32, _VP]),
    "rt_multi_destroy": (None, [_VP]),
    "rt_group_create": (C.c_int, [_VP, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(_VP)]),
    "rt_group_export": (C.c_int, [_VP, _VP]),
    "rt_group_connect": (C.c_int, [_VP, _VP]),
    "rt_group_accum": (_VP, [_VP]),
    "rt_group_begin_frame": (C.c_int, [_VP]),
    "rt_group_finish_frame": (C.c_int, [_VP, C.c_int32, C.POINTER(C.c_float)]),
    "rt_group_read_frame": (C.c_int, [_VP, _VP, _VP]),
    "rt_group_read_accum": (C.c_int, [_VP, _VP]),
    "rt_group_destroy": (None, [_VP]),
    "rt_quantize_rgb8": (C.c_int, [_VP, C.c_int32, C.c_int32, _VP]),
    "rt_write_ppm": (C.c_int, [C.c_char_p, C.c_int32, C.c_int32, _VP]),
    "rt_read_ppm_f32": (C.c_int, [C.c_char_p, C.POINTER(C.POINTER(C.c_float)), C.POINTER(C.c_int32),
                                  C.POINTER(C.c_int32)]),
    "rt_jpeg_parse": (C.c_int, [_VP, C.c_size_t, C.POINTER(C.POINTER(rt_jpeg_coefficients))]),
    "rt_jpeg_coefficients_free": (None, [C.POINTER(rt_jpeg_coefficients)]),
    "rt_jpeg_decode": (C.c_int, [_VP, _VP, C.c_size_t, C.POINTER(C.POINTER(C.c_float)), C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                 C.POINTER(C.c_int32), C.POINTER(C.c_float)]),
    "rt_image_load": (C.c_int, [_VP, C.c_char_p, C.POINTER(C.POINTER(C.c_float)), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "rt_image_to_rgb": (C.c_int, [_VP, C.c_int32, C.c_int32, C.c_int32, _VP]),
    "rt_free": (None, [_VP]),
    "rt_jpeg_max_bytes": (C.c_size_t, [C.c_int32, C.c_int32]),
    "rt_jpeg_encode_device": (C.c_int, [_VP, _VP, C.c_int32, C.c_int32, C.c_int32, _VP, C.c_size_t, C.POINTER(C.c_size_t),
                                        C.POINTER(C.c_float)]),
    "rt_jpeg_encode": (C.c_int, [_VP, _VP, C.c_int32, C.c_int32, C.c_int32, _VP, C.c_size_t, C.POINTER(C.c_size_t)]),
    "rt_write_jpg": (C.c_int, [_VP, C.c_char_p, C.c_int32, C.c_int32, _VP, C.c_int32]),
    "rt_render_jpeg": (C.c_int, [_VP, _VP, C.POINTER(rt_render_params), C.c_int32, _VP, C.c_size_t, C.POINTER(C.c_size_t),
                                 C.POINTER(rt_stats)]),
    "rt_builtin_scene": (C.c_int, [C.c_char_p, _VP, C.c_int32, C.c_int32, C.c_uint32, C.c_uint32,
                                   C.POINTER(C.POINTER(rt_scene_desc))]),
    "rt_scene_desc_free": (None, [C.POINTER(rt_scene_desc)]),
    "rt_scene_desc_from_json": (C.c_int, [_VP, C.c_char_p, C.c_char_p, C.POINTER(rt_render_params),
                                          C.POINTER(C.POINTER(rt_scene_desc))]),
    "rt_scene_desc_from_json_file": (C.c_int, [_VP, C.c_char_p, C.POINTER(rt_render_params), C.POINTER(C.POINTER(rt_scene_desc))]),
    "rt_scene_desc_save": (C.c_int, [C.POINTER(rt_scene_desc), C.c_char_p]),
    "rt_scene_desc_load": (C.c_int, [C.c_char_p, C.POINTER(C.POINTER(rt_scene_desc))]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def load_library(path: os.PathLike | None = None) -> C.CDLL:
    """dlopen librt_b200.so (built in-tree by `make lib` / __graft_entry__.build()).  No fallback."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = Path(path) if path else LIB_PATH
    if not p.exists():
        raise FileNotFoundError(f"{p} not found: build it with `make lib` (there is no CPU fallback)")
    lib = C.CDLL(str(p))
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    if path is None:
        _lib = lib
    check_layout(lib)
    return lib


def check_layout(lib: C.CDLL) -> None:
    for cls in (rt_jpeg_component, rt_jpeg_coefficients, rt_sphere, rt_material, rt_texture, rt_image, rt_camera, rt_scene_desc, rt_render_params, rt_stats,
                rt_scene_info, rt_ray, rt_hit, rt_shade_sample, rt_denoise_params, rt_adaptive_params):
        want = lib.rt_abi_sizeof(cls.__name__.encode())
        if want != C.sizeof(cls):
            raise RuntimeError(f"ABI drift: sizeof({cls.__name__}) is {want} in the library, {C.sizeof(cls)} here")


def _check(lib: C.CDLL, status: int) -> None:
    if status != RT_OK:
        raise RtError(status, (lib.rt_last_error() or b"").decode(errors="replace"))


def _f32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float32)


class SceneDesc:
    """Owns (or borrows) a rt_scene_desc.  Built-in scenes come from the C++ facade via rt_builtin_scene."""

    def __init__(self, ptr, lib, keepalive=None):
        self._ptr = ptr
        self._lib = lib
        self._keep = keepalive

    @classmethod
    def builtin(cls, name: str, image: np.ndarray | None = None, n: int = 0, bvh_mode: int = RT_BVH_AUTO) -> "SceneDesc":
        lib = load_library()
        out = C.POINTER(rt_scene_desc)()
        if image is not None:
            image = _f32(image)
            h, w = image.shape[:2]
            st = lib.rt_builtin_scene(name.encode(), image.ctypes.data, w, h, n, bvh_mode, C.byref(out))
        else:
            st = lib.rt_builtin_scene(name.encode(), None, 0, 0, n, bvh_mode, C.byref(out))
        _check(lib, st)
        return cls(out, lib)

    @classmethod
    def load(cls, path: str) -> "SceneDesc":
        lib = load_library()
        out = C.POINTER(rt_scene_desc)()
        _check(lib, lib.rt_scene_desc_load(str(path).encode(), C.byref(out)))
        return cls(out, lib)

    @classmethod
    def from_json(cls, text: str, base_dir: str = "", params: "rt_render_params | None" = None, ctx: "Context | None" = None) -> "SceneDesc":
        """rt_scene_desc_from_json: the runtime scene front-end (format: include/rt/scene_json.hpp).  JPEG image files need `ctx`."""
        lib = load_library()
        out = C.POINTER(rt_scene_desc)()
        _check(lib, lib.rt_scene_desc_from_json(ctx._h if ctx is not None else None, text.encode(), str(base_dir).encode(), C.byref(params) if params is not None else None,
                                                C.byref(out)))
        return cls(out, lib)

    @classmethod
    def from_json_file(cls, path: str, params: "rt_render_params | None" = None, ctx: "Context | None" = None) -> "SceneDesc":
        lib = load_library()
        out = C.POINTER(rt_scene_desc)()
        _check(lib, lib.rt_scene_desc_from_json_file(ctx._h if ctx is not None else None, str(path).encode(), C.byref(params) if params is not None else None, C.byref(out)))
        return cls(out, lib)

    def save(self, path: str) -> None:
        _check(self._lib, self._lib.rt_scene_desc_save(self._ptr, str(path).encode()))

    @property
    def desc(self) -> rt_scene_desc:
        return self._ptr.contents

    def set_bvh_mode(self, mode: int) -> None:
        self._ptr.contents.bvh_mode = mode

    def spheres(self) -> np.ndarray:
        d = self.desc
        return np.ctypeslib.as_array(C.cast(d.spheres, C.POINTER(C.c_uint8)), (d.n_spheres * C.sizeof(rt_sphere),)).view(
            SPHERE_DTYPE).copy() if d.n_spheres else np.zeros(0, SPHERE_DTYPE)

    def __del__(self):
        if getattr(self, "_ptr", None) and self._keep is None:
            try:
                self._lib.rt_scene_desc_free(self._ptr)
            except Exception:
                pass
            self._ptr = None


SPHERE_DTYPE = np.dtype([("center0", "<f4", 3), ("radius", "<f4"), ("center1", "<f4", 3), ("time0", "<f4"),
                         ("time1", "<f4"), ("material", "<u4"), ("id", "<u4"), ("flags", "<u4")])
assert SPHERE_DTYPE.itemsize == C.sizeof(rt_sphere)


def default_params(**kw) -> rt_render_params:
    lib = load_library()
    p = rt_render_params()
    lib.rt_default_render_params(C.byref(p))
    for k, v in kw.items():
        if k == "world":
            p.world[:] = v
        else:
            setattr(p, k, v)
    return p


def default_denoise_params(**kw) -> rt_denoise_params:
    """rt_default_denoise_params with fields overridden by keyword."""
    lib = load_library()
    d = rt_denoise_params()
    lib.rt_default_denoise_params(C.byref(d))
    for k, v in kw.items():
        setattr(d, k, v)
    return d


def default_adaptive_params(**kw) -> rt_adaptive_params:
    """rt_default_adaptive_params with fields overridden by keyword."""
    lib = load_library()
    a = rt_adaptive_params()
    lib.rt_default_adaptive_params(C.byref(a))
    for k, v in kw.items():
        setattr(a, k, v)
    return a


class Context:
    """One CUDA device + one stream (one process per GPU)."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        self._h = _VP()
        _check(self.lib, self.lib.rt_context_create(device, C.byref(self._h)))
        self.device = device
        # open scenes and groups of this context, handle -> destroy entry: they must be destroyed before the context, and
        # when the garbage collector finds a context and its scenes unreachable together it finalises them in no
        # particular order
        self._open: dict[int, object] = {}

    def set_stream(self, cuda_stream: int) -> None:
        _check(self.lib, self.lib.rt_context_set_stream(self._h, _VP(cuda_stream)))

    def synchronize(self) -> None:
        _check(self.lib, self.lib.rt_context_synchronize(self._h))

    def close(self) -> None:
        if self._h:
            for h, destroy in self._open.items():
                destroy(_VP(h))
            self._open.clear()
            self.lib.rt_context_destroy(self._h)
            self._h = _VP()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Scene:
    def __init__(self, ctx: Context, desc: SceneDesc):
        self.ctx = ctx
        self.lib = ctx.lib
        self._h = _VP()
        _check(self.lib, self.lib.rt_scene_create(ctx._h, desc._ptr, C.byref(self._h)))
        ctx._open[self._h.value] = self.lib.rt_scene_destroy

    def info(self) -> rt_scene_info:
        i = rt_scene_info()
        _check(self.lib, self.lib.rt_scene_get_info(self._h, C.byref(i)))
        return i

    def trace_primary(self, rays: np.ndarray, tmin: float = 1e-5, use_bvh: bool | int = True) -> np.ndarray:
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        hits = np.zeros(rays.shape[0], dtype=HIT_DTYPE)
        _check(self.lib, self.lib.rt_trace_primary(self.ctx._h, self._h, rays.ctypes.data, rays.shape[0], tmin,
                                                   int(use_bvh), hits.ctypes.data))
        return hits

    def shade_probe(self, rays: np.ndarray, params: rt_render_params, use_bvh: bool = True) -> np.ndarray:
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        out = np.zeros(rays.shape[0], dtype=SHADE_DTYPE)
        _check(self.lib, self.lib.rt_shade_probe(self.ctx._h, self._h, rays.ctypes.data, rays.shape[0], C.byref(params),
                                                 int(use_bvh), out.ctypes.data))
        return out

    def render(self, params: rt_render_params, out: np.ndarray | None = None):
        """rt_render: HOST float RGB [H, W, 3], reference framebuffer layout (row 0 = bottom)."""
        if out is None:
            out = np.empty((params.height, params.width, 3), dtype=np.float32)
        st = rt_stats()
        _check(self.lib, self.lib.rt_render(self.ctx._h, self._h, C.byref(params), out.ctypes.data, C.byref(st)))
        return out, st

    def render_accum(self, params: rt_render_params):
        out = np.empty((params.height, params.width, 4), dtype=np.float32)
        st = rt_stats()
        _check(self.lib, self.lib.rt_render_accum(self.ctx._h, self._h, C.byref(params), out.ctypes.data, C.byref(st)))
        return out, st

    def render_accum_device(self, params: rt_render_params, accum_ptr: int, want_stats: bool = False, ctx: "Context | None" = None):
        """rt_render_accum_device; `ctx` renders this scene through ANOTHER context of the same device (frame pipelines)."""
        st = rt_stats() if want_stats else None
        _check(self.lib, self.lib.rt_render_accum_device((ctx or self.ctx)._h, self._h, C.byref(params), _VP(accum_ptr),
                                                         C.byref(st) if st is not None else None))
        return st

    def render_progressive(self, params: rt_render_params, passes: int, on_pass=None):
        """rt_render_progressive: `passes` x params.spp samples into one accumulator; on_pass(pass, spp_so_far, rgb[H,W,3])
        is called after every pass (return True to stop).  Returns (final frame, stats)."""
        out = np.empty((params.height, params.width, 3), dtype=np.float32)
        CB = C.CFUNCTYPE(C.c_int, C.c_int32, C.c_int32, C.POINTER(C.c_float), _VP)

        def _cb(k, spp, rgb, _user):
            return 1 if (on_pass and on_pass(int(k), int(spp), out)) else 0

        cb = CB(_cb)
        st = rt_stats()
        _check(self.lib, self.lib.rt_render_progressive(self.ctx._h, self._h, C.byref(params), passes, out.ctypes.data,
                                                        C.cast(cb, _VP), None, C.byref(st)))
        return out, st

    def render_jpeg(self, params: rt_render_params, quality: int = 100, out: np.ndarray | None = None):
        """rt_render_jpeg: render -> finalise -> flip/quantise -> JPEG on the device; returns (file bytes, stats)."""
        cap = self.lib.rt_jpeg_max_bytes(params.width, params.height)
        if out is None:
            out = np.empty(cap, dtype=np.uint8)
        n = C.c_size_t(0)
        st = rt_stats()
        _check(self.lib, self.lib.rt_render_jpeg(self.ctx._h, self._h, C.byref(params), quality, out.ctypes.data, out.size,
                                                 C.byref(n), C.byref(st)))
        return out[:n.value], st

    def render_denoised(self, params: rt_render_params, denoise: "rt_denoise_params | None" = None):
        """rt_render_denoised: render + features + à-trous filter + finalisation; HOST float RGB [H, W, 3] (layout of render)."""
        d = denoise if denoise is not None else default_denoise_params()
        out = np.empty((params.height, params.width, 3), dtype=np.float32)
        st = rt_stats()
        _check(self.lib, self.lib.rt_render_denoised(self.ctx._h, self._h, C.byref(params), C.byref(d), out.ctypes.data, C.byref(st)))
        return out, st

    def render_features_device(self, params: rt_render_params, feature_spp: int, features_ptr: int) -> None:
        """rt_render_features_device: first-hit features of feature_spp camera samples per pixel into 2*W*H float4 of device
        memory (plane 0: mean normal, mean distance; plane 1: mean albedo, hit fraction)."""
        _check(self.lib, self.lib.rt_render_features_device(self.ctx._h, self._h, C.byref(params), feature_spp, _VP(features_ptr)))

    def render_adaptive(self, params: rt_render_params, adaptive: "rt_adaptive_params | None" = None):
        """rt_render_adaptive: returns (HOST float RGB [H, W, 3] in the layout of render, samples per pixel [H, W] int32, stats,
        passes run)."""
        a = adaptive if adaptive is not None else default_adaptive_params()
        out = np.empty((params.height, params.width, 3), dtype=np.float32)
        spp = np.empty((params.height, params.width), dtype=np.int32)
        st = rt_stats()
        _check(self.lib, self.lib.rt_render_adaptive(self.ctx._h, self._h, C.byref(params), C.byref(a), out.ctypes.data, spp.ctypes.data,
                                                     C.byref(st)))
        return out, spp, st, 1 + (int(spp.max()) - a.min_spp) // a.step_spp  # one pass per sample level up to the largest count

    def render_adaptive_device(self, params: rt_render_params, adaptive: "rt_adaptive_params | None", accum_ptr: int,
                               error_ptr: int = 0, want_stats: bool = False):
        """rt_render_adaptive_device: writes the finished accumulator (W*H float4) to accum_ptr and, if error_ptr, the final
        windowed error map (W*H float) there.  Returns (passes run, stats or None)."""
        a = adaptive if adaptive is not None else default_adaptive_params()
        st = rt_stats() if want_stats else None
        passes = C.c_int32(0)
        _check(self.lib, self.lib.rt_render_adaptive_device(self.ctx._h, self._h, C.byref(params), C.byref(a), _VP(accum_ptr),
                                                            _VP(error_ptr or None), C.byref(passes), C.byref(st) if st is not None else None))
        return passes.value, st

    def render_frames(self, params: rt_render_params, cameras):
        """rt_render_frames: frame f of the sequence looks through cameras[f] (a sequence of rt_camera, e.g. from orbit_cameras)
        with samples params.sample_offset + f * params.spp + [0, spp).  Returns (HOST float RGB [K, H, W, 3], frame f in the
        layout of render, stats)."""
        cams = _camera_array(cameras)
        out = np.empty((len(cams), params.height, params.width, 3), dtype=np.float32)
        st = rt_stats()
        _check(self.lib, self.lib.rt_render_frames(self.ctx._h, self._h, C.byref(params), cams, len(cams), out.ctypes.data, C.byref(st)))
        return out, st

    def render_frames_device(self, params: rt_render_params, cameras, accum_ptr: int, want_stats: bool = False):
        """rt_render_frames_device: ADDS frame f into accum_ptr + f * W * H float4 (device).  Returns stats or None."""
        cams = _camera_array(cameras)
        st = rt_stats() if want_stats else None
        _check(self.lib, self.lib.rt_render_frames_device(self.ctx._h, self._h, C.byref(params), cams, len(cams), _VP(accum_ptr),
                                                          C.byref(st) if st is not None else None))
        return st

    def close(self) -> None:
        if self._h:
            if self.ctx._open.pop(self._h.value, None):  # (else the context has been closed and destroyed the scene with it)
                self.lib.rt_scene_destroy(self._h)
            self._h = _VP()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _camera_array(cameras):
    cams = list(cameras)
    return (rt_camera * len(cams))(*cams)


def orbit_cameras(base: rt_camera, n: int, degrees: float):
    """rt_orbit_cameras: n cameras, frame k = base with lookfrom rotated by k * degrees / n about the axis through lookat along
    up and the k-th of n equal shutter windows of [base.time0, base.time1].  Needs no device."""
    lib = load_library()
    out = (rt_camera * max(int(n), 1))()
    _check(lib, lib.rt_orbit_cameras(C.byref(base), int(n), float(degrees), out))
    return list(out)


def tonemap_device(ctx: Context, accum_ptr: int, width: int, height: int, out_rgb_ptr: int = 0, out_rgb8_ptr: int = 0):
    _check(ctx.lib, ctx.lib.rt_tonemap_device(ctx._h, _VP(accum_ptr), width, height, _VP(out_rgb_ptr or None),
                                              _VP(out_rgb8_ptr or None)))


def denoise_device(ctx: Context, accum_ptr: int, features_ptr: int, width: int, height: int, denoise: "rt_denoise_params | None" = None,
                   out_rgb_ptr: int = 0, out_rgb8_ptr: int = 0):
    """rt_denoise_device: à-trous filter of a device accumulator guided by device features, finalised as tonemap_device."""
    d = denoise if denoise is not None else default_denoise_params()
    _check(ctx.lib, ctx.lib.rt_denoise_device(ctx._h, _VP(accum_ptr), _VP(features_ptr), width, height, C.byref(d),
                                              _VP(out_rgb_ptr or None), _VP(out_rgb8_ptr or None)))


def adaptive_error_device(ctx: Context, planes_ptr: int, width: int, height: int, error_ptr: int) -> None:
    """rt_adaptive_error_device: windowed error map (W*H float) of a two-plane accumulator (2*W*H float4, plane A then B)."""
    _check(ctx.lib, ctx.lib.rt_adaptive_error_device(ctx._h, _VP(planes_ptr), width, height, _VP(error_ptr)))


RT_GROUP_HANDLE_BYTES = 192


def selftest_rz(ctx: "Context", x: np.ndarray, y: np.ndarray) -> np.ndarray:
    """rt_selftest_rz -> [n, 4] float32: div_rz(x, y), __fdiv_rz(x, y), sqrt_rz(x), __fsqrt_rz(x)."""
    x, y = np.ascontiguousarray(x, np.float32), np.ascontiguousarray(y, np.float32)
    out = np.empty((x.size, 4), np.float32)
    _check(ctx.lib, ctx.lib.rt_selftest_rz(ctx._h, x.ctypes.data, y.ctypes.data, x.size, out.ctypes.data))
    return out


def selftest_exclusive_sum(ctx: "Context", values: np.ndarray, in_place: bool = False, out: np.ndarray | None = None):
    """rt_selftest_exclusive_sum on a uint32 or uint64 array -> (exclusive prefix sums, overrun).  `out` (same dtype and
    size) receives the sums when given."""
    values = np.ascontiguousarray(values)
    assert values.dtype in (np.uint32, np.uint64), values.dtype
    if out is None:
        out = np.empty_like(values)
    assert out.dtype == values.dtype and out.size == values.size and out.flags.c_contiguous
    overrun = C.c_int32(-1)
    _check(ctx.lib, ctx.lib.rt_selftest_exclusive_sum(ctx._h, values.ctypes.data, out.ctypes.data, values.size, values.itemsize,
                                                      int(in_place), C.byref(overrun)))
    return out, bool(overrun.value)


def selftest_sort_pairs(ctx: "Context", keys: np.ndarray, vals: np.ndarray, passes: int):
    """rt_selftest_sort_pairs -> (sorted uint64 keys, uint32 values, in_alt, overrun): stable by the key bits
    [0, 8 * passes)."""
    keys, vals = np.ascontiguousarray(keys, np.uint64), np.ascontiguousarray(vals, np.uint32)
    assert keys.size == vals.size
    k_out, v_out = np.empty_like(keys), np.empty_like(vals)
    in_alt, overrun = C.c_int32(-1), C.c_int32(-1)
    _check(ctx.lib, ctx.lib.rt_selftest_sort_pairs(ctx._h, keys.ctypes.data, vals.ctypes.data, keys.size, passes, k_out.ctypes.data,
                                                   v_out.ctypes.data, C.byref(in_alt), C.byref(overrun)))
    return k_out, v_out, bool(in_alt.value), bool(overrun.value)


def shard_samples(spp_total: int, rank: int, world: int):
    """rt_shard_samples: (first sample index, sample count) of `rank`."""
    lib = load_library()
    first, count = C.c_int32(), C.c_int32()
    _check(lib, lib.rt_shard_samples(spp_total, rank, world, C.byref(first), C.byref(count)))
    return first.value, count.value


def shard_rows(height: int, rank: int, world: int):
    """rt_shard_rows: [row_begin, row_end) of the band `rank` reduces."""
    lib = load_library()
    a, b = C.c_int32(), C.c_int32()
    _check(lib, lib.rt_shard_rows(height, rank, world, C.byref(a), C.byref(b)))
    return a.value, b.value


class Multi:
    """rt_multi_*: ONE process driving n devices (sample-sharded render + fused NVLink reduce)."""

    def __init__(self, devices=None):
        self.lib = load_library()
        self._h = _VP()
        if devices is None:
            _check(self.lib, self.lib.rt_multi_create(None, 0, C.byref(self._h)))
        else:
            arr = (C.c_int32 * len(devices))(*devices)
            _check(self.lib, self.lib.rt_multi_create(arr, len(devices), C.byref(self._h)))
        self.size = int(self.lib.rt_multi_size(self._h))

    def set_scene(self, desc: "SceneDesc") -> None:
        _check(self.lib, self.lib.rt_multi_set_scene(self._h, desc._ptr))

    def render(self, params: rt_render_params, want_rgb8: bool = False):
        rgb = np.empty((params.height, params.width, 3), np.float32)
        rgb8 = np.empty((params.height, params.width, 3), np.uint8) if want_rgb8 else None
        st, ms = rt_stats(), C.c_float()
        _check(self.lib, self.lib.rt_multi_render(self._h, C.byref(params), rgb.ctypes.data, rgb8.ctypes.data if want_rgb8 else None,
                                                  C.byref(st), C.byref(ms)))
        return rgb, rgb8, st, ms.value

    def read_accum(self, member: int, width: int, height: int) -> np.ndarray:
        out = np.empty((height, width, 4), np.float32)
        _check(self.lib, self.lib.rt_multi_read_accum(self._h, member, out.ctypes.data))
        return out

    def close(self) -> None:
        if self._h:
            self.lib.rt_multi_destroy(self._h)
            self._h = _VP()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Group:
    """rt_group_*: this process's member of a one-process-per-GPU group.  `exchange(blob) -> [blob of rank 0, ...]`
    moves the IPC handle blobs between the processes (e.g. torch.distributed.all_gather_object)."""

    def __init__(self, ctx: "Context", rank: int, world: int, width: int, height: int, exchange):
        self.lib, self.ctx, self.rank, self.world, self.width, self.height = ctx.lib, ctx, rank, world, width, height
        self._h = _VP()
        _check(self.lib, self.lib.rt_group_create(ctx._h, rank, world, width, height, C.byref(self._h)))
        ctx._open[self._h.value] = self.lib.rt_group_destroy
        blob = C.create_string_buffer(RT_GROUP_HANDLE_BYTES)
        _check(self.lib, self.lib.rt_group_export(self._h, blob))
        if world > 1:
            table = b"".join(bytes(b) for b in exchange(bytes(blob.raw)))
            assert len(table) == world * RT_GROUP_HANDLE_BYTES
            _check(self.lib, self.lib.rt_group_connect(self._h, C.create_string_buffer(table, len(table))))
        self.accum_ptr = int(self.lib.rt_group_accum(self._h))

    def begin_frame(self) -> None:
        _check(self.lib, self.lib.rt_group_begin_frame(self._h))

    def finish_frame(self, want_rgb8: bool = False, timed: bool = False) -> float:
        ms = C.c_float()
        _check(self.lib, self.lib.rt_group_finish_frame(self._h, int(want_rgb8), C.byref(ms) if timed else None))
        return ms.value

    def read_frame(self, out_rgb: "np.ndarray | None" = None, out_rgb8: "np.ndarray | None" = None) -> None:
        _check(self.lib, self.lib.rt_group_read_frame(self._h, out_rgb.ctypes.data if out_rgb is not None else None,
                                                      out_rgb8.ctypes.data if out_rgb8 is not None else None))

    def read_accum(self) -> np.ndarray:
        out = np.empty((self.height, self.width, 4), np.float32)
        _check(self.lib, self.lib.rt_group_read_accum(self._h, out.ctypes.data))
        return out

    def close(self) -> None:
        if self._h:
            if self.ctx._open.pop(self._h.value, None):  # (else the context has been closed and destroyed the group with it)
                self.lib.rt_group_destroy(self._h)
            self._h = _VP()


def reduce_tonemap_peers(ctx: Context, peer_ptrs, multicast_ptr: int, width: int, height: int, row_begin: int, row_end: int,
                         out_rgb_ptr: int = 0, out_rgb8_ptr: int = 0, out_sum_ptr: int = 0) -> None:
    """rt_reduce_tonemap_peers: fused NVLink reduce (+ NVLS multimem when multicast_ptr != 0) and tonemap."""
    n = len(peer_ptrs)
    arr = (_VP * n)(*[_VP(int(p)) for p in peer_ptrs])
    _check(ctx.lib, ctx.lib.rt_reduce_tonemap_peers(ctx._h, arr, n, _VP(multicast_ptr or None), width, height, row_begin, row_end,
                                                    _VP(out_rgb_ptr or None), _VP(out_rgb8_ptr or None), _VP(out_sum_ptr or None)))


def jpeg_encode(ctx: Context, rgb8: np.ndarray, quality: int = 100) -> bytes:
    """rt_jpeg_encode: stbi_write_jpg(.., w, h, 3, rgb8, quality) (main.cu:491) on the device; returns the file."""
    rgb8 = np.ascontiguousarray(rgb8, dtype=np.uint8)
    h, w = rgb8.shape[:2]
    cap = ctx.lib.rt_jpeg_max_bytes(w, h)
    out = np.empty(cap, dtype=np.uint8)
    n = C.c_size_t(0)
    _check(ctx.lib, ctx.lib.rt_jpeg_encode(ctx._h, rgb8.ctypes.data, w, h, quality, out.ctypes.data, cap, C.byref(n)))
    return out[:n.value].tobytes()


def jpeg_encode_device(ctx: Context, rgb8_ptr: int, width: int, height: int, quality: int, out: np.ndarray):
    """rt_jpeg_encode_device: device rgb8 -> file in `out` (host uint8 array); returns (n_bytes, device ms)."""
    n = C.c_size_t(0)
    ms = C.c_float(0)
    _check(ctx.lib, ctx.lib.rt_jpeg_encode_device(ctx._h, _VP(rgb8_ptr), width, height, quality, out.ctypes.data, out.size,
                                                  C.byref(n), C.byref(ms)))
    return n.value, ms.value


def jpeg_parse(file_bytes: bytes):
    """rt_jpeg_parse: host half of the JPEG reader.  Returns the owning pointer (free with jpeg_coefficients_free)."""
    lib = load_library()
    buf = np.frombuffer(file_bytes, dtype=np.uint8)
    out = C.POINTER(rt_jpeg_coefficients)()
    _check(lib, lib.rt_jpeg_parse(buf.ctypes.data, buf.size, C.byref(out)))
    return out


def jpeg_coefficients_free(ptr) -> None:
    load_library().rt_jpeg_coefficients_free(ptr)


def jpeg_decode(ctx: "Context", file_bytes: bytes):
    """rt_jpeg_decode: stbi_loadf(file, &w, &h, &ch, 0) (main.cu:376-380): returns ([H, W, ch] float32, device ms)."""
    buf = np.frombuffer(file_bytes, dtype=np.uint8)
    px = C.POINTER(C.c_float)()
    w, h, ch, ms = C.c_int32(), C.c_int32(), C.c_int32(), C.c_float()
    _check(ctx.lib, ctx.lib.rt_jpeg_decode(ctx._h, buf.ctypes.data, buf.size, C.byref(px), C.byref(w), C.byref(h), C.byref(ch), C.byref(ms)))
    out = np.ctypeslib.as_array(px, (h.value, w.value, ch.value)).copy()
    ctx.lib.rt_free(px)
    return out, ms.value


def image_to_rgb(data: np.ndarray) -> np.ndarray:
    """rt_image_to_rgb: [H, W, C] float image with C in 1..4 -> [H, W, 3] (what image_texture indexes)."""
    lib = load_library()
    data = _f32(data)
    if data.ndim == 2:
        data = data[..., None]
    h, w, c = data.shape
    out = np.empty((h, w, 3), dtype=np.float32)
    _check(lib, lib.rt_image_to_rgb(data.ctypes.data, w, h, c, out.ctypes.data))
    return out


def quantize_rgb8(rgb: np.ndarray) -> np.ndarray:
    """main.cu:475-488 on the host: Y flip + int(255.999f*c) & 255."""
    lib = load_library()
    rgb = _f32(rgb)
    h, w = rgb.shape[:2]
    out = np.empty((h, w, 3), dtype=np.uint8)
    _check(lib, lib.rt_quantize_rgb8(rgb.ctypes.data, w, h, out.ctypes.data))
    return out


def psnr(a: np.ndarray, b: np.ndarray, peak: float = 1.0) -> float:
    mse = float(np.mean((np.asarray(a, np.float64) - np.asarray(b, np.float64)) ** 2))
    return float("inf") if mse == 0 else 10.0 * np.log10(peak * peak / mse)
