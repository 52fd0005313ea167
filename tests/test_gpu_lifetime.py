"""Teardown order through the Python binding: an rt_scene must be destroyed before the rt_context it was created on,
whichever of the two Python objects goes first."""
import gc

import numpy as np
import pytest

import raytracing_renderer_cuda_b200 as rt

pytestmark = pytest.mark.gpu


def test_context_closed_before_its_scene(scene_descs):
    """Closing a context destroys the scenes still open on it; closing such a scene afterwards does nothing."""
    ctx = rt.Context(0)
    sc = rt.Scene(ctx, scene_descs["book1_final"])
    assert sc._h.value in ctx._open
    ctx.close()
    assert not ctx._open
    sc.close()
    assert not sc._h


def test_context_and_scene_collected_together(scene_descs):
    """A context and its scenes that become garbage in one reference cycle are finalised in no particular order; a
    context created afterwards renders normally."""
    for _ in range(3):
        ctx = rt.Context(0)
        cycle = [ctx, rt.Scene(ctx, scene_descs["book1_final"]), rt.Scene(ctx, scene_descs["perlin_motion"])]
        cycle.append(cycle)
        del ctx, cycle
        gc.collect()
    ctx = rt.Context(0)
    img, st = rt.Scene(ctx, scene_descs["book1_final"]).render(rt.default_params(width=32, height=16, spp=2))
    assert st.paths == 32 * 16 * 2 and np.isfinite(img).all()
