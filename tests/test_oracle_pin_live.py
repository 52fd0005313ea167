"""Live pin of the oracle against the reference's own headers (oracle/_ref/libref_cpu.so).  Only where the
reference has been compiled (`make -C oracle ref REF=<reference checkout>`); elsewhere tests/test_oracle_golden.py
carries the same comparison through committed vectors."""
import numpy as np
import pytest

import raytracing_renderer_cuda_b200 as rt
from raytracing_renderer_cuda_b200 import capi
from tests.conftest import SCENES
from tests.oracle_api import REFCPU_SO, RefCpu, camera_rays, secondary_rays

needs_reference = pytest.mark.skipif(not REFCPU_SO.exists(), reason="oracle/_ref/libref_cpu.so not built (the reference's sources are not here)")


@pytest.fixture(scope="module")
def ref():
    return RefCpu()


@needs_reference
@pytest.mark.parametrize("name", SCENES)
def test_trace_matches_reference_headers(oracle, ref, scene_descs, name):
    d = scene_descs[name]
    rays = camera_rays(d, 20000, seed=3)
    want = ref.scene(d, use_bvh=False).trace(rays)
    got = oracle.scene(d).trace(rays, arith=0)
    assert got.tobytes() == want.tobytes()
    sec = secondary_rays(d, want, seed=4)
    want2 = ref.scene(d, use_bvh=False).trace(sec)
    assert oracle.scene(d).trace(sec, arith=0).tobytes() == want2.tobytes()
    # the reference's own BVH (bvh.h:75-155) returns what its brute-force list does
    bvh = ref.scene(d, use_bvh=True)
    for r, w in ((rays, want), (sec, want2)):
        b = bvh.trace(r)
        assert np.array_equal(b["id"], w["id"]) and np.array_equal(b["t"], w["t"])


@needs_reference
@pytest.mark.parametrize("name,size", [("earth_emitter", (96, 48, 8)), ("book1_final", (64, 36, 4)), ("perlin_motion", (64, 32, 4))])
def test_render_matches_reference_headers(oracle, ref, scene_descs, name, size):
    w, h, spp = size
    d = scene_descs[name]
    mean, fb, nrays = ref.scene(d, use_bvh=False).render(w, h, spp)
    acc, n2 = oracle.scene(d).render(rt.default_params(width=w, height=h, spp=spp), sampler=0, arith=0)
    assert n2 == nrays
    assert np.array_equal(oracle.tonemap(acc), fb)


def test_product_sampler_is_statistically_the_reference_sampler(oracle, scene_descs):
    """Sampler 1 (Philox + direct ball/disk sampling, what the CUDA path does) draws from the same
    distributions as sampler 0 (sequential generator + rejection): two renders of the same scene differ
    only by Monte-Carlo noise, i.e. no more than two reference-sampler renders with different seeds."""
    d = scene_descs["earth_emitter"]
    sc = oracle.scene(d)
    w, h, spp = 100, 50, 128
    a, _ = sc.render(rt.default_params(width=w, height=h, spp=spp), sampler=0)
    b, _ = sc.render(rt.default_params(width=w, height=h, spp=spp, seed=77), sampler=0)
    c, _ = sc.render(rt.default_params(width=w, height=h, spp=spp), sampler=1)
    ta, tb, tc = oracle.tonemap(a), oracle.tonemap(b), oracle.tonemap(c)
    noise = rt.psnr(ta, tb)
    assert rt.psnr(ta, tc) > noise - 0.5 and rt.psnr(tb, tc) > noise - 0.5, (noise, rt.psnr(ta, tc), rt.psnr(tb, tc))
    # and the mean image brightness agrees to well under the noise level
    assert abs(float(a[..., :3].mean()) - float(c[..., :3].mean())) / float(a[..., :3].mean()) < 5e-3
