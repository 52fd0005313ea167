"""B200-native path tracer behind the scene API of slimem/raytracing_renderer_cuda.

The product is `librt_b200.so` (hand-written sm_100a CUDA behind the C-ABI of
include/rt_api.h) plus the header-only C++ facade in include/rt/.  This package
only carries the ctypes binding used by tests/, bench.py and __graft_entry__.py.
"""
from . import capi  # noqa: F401
from .capi import (Context, Group, Multi, Scene, SceneDesc, adaptive_error_device, default_adaptive_params,  # noqa: F401
                   default_denoise_params, default_params, denoise_device, load_library, orbit_cameras, psnr, quantize_rgb8,
                   reduce_tonemap_peers, shard_rows, shard_samples, tonemap_device)
