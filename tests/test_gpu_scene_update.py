"""Scene updates on the B200: a scene updated in place against rt_scene_create of the edited description, created fresh.

Closest hits (camera rays and secondary rays, every use_bvh both scenes have) must be bit-identical, and every walk of the
updated scene must equal its own brute-force list; renders must have equal sample and ray counts and sums equal up to the
order of float additions (the tolerance of test_gpu_frames.py).  Covers the constant-bank list, a brute-force list, host
SAH trees, a GPU LBVH with the outsized-sphere chain and the 4-wide and quantised forms; moves of 1 %, 10 % and 100 % of the
spheres, radius scaling, new motions and ids, and adversarial edits (everything on one point, a sphere far outside the old
root box, 50 successive edits, a moved caterpillar tree, an exact tie, an extent beyond the quantised range).  Also every
render pipeline, emitter sampling after material and sphere edits, camera edits through every host render entry, the
identity edit, stream ordering, rejected edits and the multi-GPU entry."""
import ctypes as C
import zlib

import numpy as np
import pytest

import raytracing_renderer_cuda_b200 as rt
from raytracing_renderer_cuda_b200 import capi
from tests.test_gpu_bvh_adversarial import _doc, caterpillar, grid_scene

pytestmark = pytest.mark.gpu

F32 = np.float32


@pytest.fixture(scope="module")
def ctx():
    return rt.Context(0)


# ------------------------------------------------------------------------------------------------------------ descriptions

def _materials(desc):
    d = desc.desc
    return [capi.rt_material.from_buffer_copy(d.materials[k]) for k in range(d.n_materials)]


def edited(desc, sphere_index=(), spheres=None, material_index=(), materials=None, camera=None):
    """A new description: `desc` with the edit applied (what rt_scene_update must match)."""
    d = desc.desc
    sph = desc.spheres()
    if len(sphere_index):
        sph[np.asarray(sphere_index, np.int64)] = spheres
    mats = _materials(desc)
    for k, m in zip(material_index, materials or ()):
        mats[k] = m
    mat_arr = (capi.rt_material * max(len(mats), 1))(*mats)
    sph = np.ascontiguousarray(sph)
    out = capi.rt_scene_desc()
    C.memmove(C.byref(out), C.byref(d), C.sizeof(out))
    out.spheres = sph.ctypes.data_as(C.POINTER(capi.rt_sphere))
    out.materials = mat_arr
    if camera is not None:
        out.camera = camera
    return rt.SceneDesc(C.pointer(out), desc._lib, keepalive=(sph, mat_arr, desc, out))


def from_list(sph, bvh, emitters=False, camera=None):
    return rt.SceneDesc.from_json(_doc(sph, bvh, camera, emitters))


SCENES = {  # name: description factory (earth: the image)
    "c1_list": lambda earth: rt.SceneDesc.builtin("earth_emitter", earth),
    "list20": lambda earth: rt.SceneDesc.builtin("random_spheres", n=20, bvh_mode=capi.RT_BVH_NONE),
    "c2_sah": lambda earth: rt.SceneDesc.builtin("book1_final", bvh_mode=capi.RT_BVH_HOST_SAH),
    "c3_sah": lambda earth: rt.SceneDesc.builtin("perlin_motion", bvh_mode=capi.RT_BVH_HOST_SAH),
    "lbvh5000": lambda earth: rt.SceneDesc.builtin("random_spheres", n=5000, bvh_mode=capi.RT_BVH_GPU_LBVH),
}


# ------------------------------------------------------------------------------------------------------------------- rays

def camera_rays(cam, n, seed):
    """From the camera's lookfrom, directions spread about the view direction."""
    rng = np.random.default_rng(seed)
    o = np.array(cam.lookfrom, np.float64)
    w = np.array(cam.lookat, np.float64) - o
    w /= np.linalg.norm(w)
    d = w[None] + rng.normal(scale=0.35, size=(n, 3))
    r = np.zeros(n, capi.RAY_DTYPE)
    r["origin"] = o.astype(F32)
    r["direction"] = d.astype(F32)
    r["time"] = rng.random(n).astype(F32)
    return r


def secondary_rays(hits, n, seed):
    """From the hit points of camera rays, random directions (misses start at the origin)."""
    rng = np.random.default_rng(seed)
    k = rng.integers(0, len(hits), n)
    r = np.zeros(n, capi.RAY_DTYPE)
    r["origin"] = np.where((hits["id"][k] != capi.RT_INVALID_ID)[:, None], hits["p"][k], 0.0)
    r["direction"] = rng.normal(size=(n, 3)).astype(F32)
    r["time"] = rng.random(n).astype(F32)
    return r


def towards(centres, n, dist, seed):
    rng = np.random.default_rng(seed)
    c = np.asarray(centres, np.float64)[rng.integers(0, len(centres), n)]
    u = rng.normal(size=(n, 3))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    r = np.zeros(n, capi.RAY_DTYPE)
    r["origin"] = (c + dist * u).astype(F32)
    r["direction"] = (-u + rng.normal(scale=0.02, size=(n, 3))).astype(F32)
    r["time"] = rng.random(n).astype(F32)
    return r


_PROBE = np.zeros(1, capi.RAY_DTYPE)
_PROBE["direction"] = (0.0, 0.0, 1.0)


def _walks(sc):
    forms = [0, 1, 2, 3] if sc.info().n_nodes else [0]
    out = []
    for u in forms:
        try:
            sc.trace_primary(_PROBE, use_bvh=u)
            out.append(u)
        except capi.RtError as e:
            assert e.status == capi.RT_ERR_INVALID_ARG
    return out


def _bytes(h):
    return h.view(np.uint8).reshape(len(h), -1)


def assert_same_hits(upd, fresh, rays):
    """Bit-identical (id, t, p, n, u, v) of the two scenes for every walk both have, and every walk of the updated scene
    equal to its list.  The list comparison leaves out the rays whose list hit even the freshly built tree does not
    reproduce: a tiny sphere seen from far away makes the float32 quadratic ill-conditioned, and the list can then report
    a hit outside the sphere's padded box (a property of the builders' padding, not of the update; at most 0.1 % of the
    rays)."""
    want = fresh.trace_primary(rays, use_bvh=0)
    mine = upd.trace_primary(rays, use_bvh=0)
    assert np.array_equal(_bytes(mine), _bytes(want)), int((_bytes(mine) != _bytes(want)).any(axis=1).sum())
    fresh_walks = set(_walks(fresh))
    for u in _walks(upd):
        got = _bytes(upd.trace_primary(rays, use_bvh=u))
        exact = np.ones(len(rays), bool)
        if u in fresh_walks:
            ref = _bytes(fresh.trace_primary(rays, use_bvh=u))
            diff = (got != ref).any(axis=1)
            assert not diff.any(), ("fresh", u, int(diff.sum()))
            exact = (ref == _bytes(want)).all(axis=1)
            assert exact.mean() >= 0.999, (u, int((~exact).sum()))
        bad = (got != _bytes(want)).any(axis=1) & exact
        assert not bad.any(), (u, int(bad.sum()))
    return want


def scene_rays(desc, sc, seed, n=4096):
    """Camera rays of the description and secondary rays from their hits in scene `sc`."""
    prim = camera_rays(desc.desc.camera, n, seed)
    return np.concatenate([prim, secondary_rays(sc.trace_primary(prim, use_bvh=0), n, seed + 1)])


def check_update(ctx, desc, idx=(), sph=None, midx=(), mats=None, cam=None, extra_rays=None):
    """Updates a scene of `desc`, compares it with a fresh scene of the edited description; returns both scenes."""
    upd = rt.Scene(ctx, desc)
    ms = upd.update(np.asarray(idx, np.uint32), sph, list(midx), mats, cam)
    assert ms >= 0.0
    new = edited(desc, idx, sph, midx, mats, cam)
    fresh = rt.Scene(ctx, new)
    rays = np.concatenate([camera_rays(new.desc.camera, 4096, 1)] + ([extra_rays] if extra_rays is not None else []))
    h = fresh.trace_primary(rays, use_bvh=0)
    rays = np.concatenate([rays, secondary_rays(h, 4096, 2)])
    assert_same_hits(upd, fresh, rays)
    return upd, fresh, new


# ------------------------------------------------------------------------------------------------------------------ edits

def _move(sph, frac, rng):
    """Jitter `frac` of the spheres (at least one) by up to one radius; a moving sphere keeps its motion vector."""
    n = len(sph)
    idx = np.sort(rng.choice(n, max(1, int(round(frac * n))), replace=False))
    new = sph[idx].copy()
    j = rng.uniform(-1, 1, (len(idx), 3)) * np.abs(new["radius"])[:, None]
    new["center0"] = (new["center0"] + j).astype(F32)
    new["center1"] = (new["center1"] + j).astype(F32)
    return idx, new


def _edit(kind, sph, rng):
    n = len(sph)
    if kind.startswith("move"):
        return _move(sph, {"move1": 0.01, "move10": 0.10, "move100": 1.0}[kind], rng)
    idx = np.arange(n)
    new = sph.copy()
    if kind in ("radius0.1", "radius50"):
        s = 0.1 if kind == "radius0.1" else 50.0
        new["radius"] = (new["radius"] * s).astype(F32)
    elif kind == "motion":
        mv = np.nonzero(sph["flags"] & capi.RT_SPHERE_MOVING)[0]
        st = np.nonzero(~sph["flags"] & capi.RT_SPHERE_MOVING)[0][: max(1, n // 10)]
        idx = np.concatenate([mv, st])
        new = sph[idx].copy()
        m = len(mv)
        new["center1"][:m] = (new["center0"][:m] + rng.uniform(-2, 2, (m, 3))).astype(F32)
        # (the motion still spans the rays' times [0, 1]: a sphere is bounded between its two motion ends only)
        new["time0"][:m] = rng.uniform(-0.5, 0.0, m).astype(F32)
        new["time1"][:m] = rng.uniform(1.0, 1.5, m).astype(F32)
        new["center0"][m:] = (new["center0"][m:] + 0.3 * np.abs(new["radius"][m:])[:, None]).astype(F32)
        new["center1"][m:] = new["center0"][m:]
    elif kind == "ids":
        new["id"] = (n + 7 + rng.permutation(n)).astype(np.uint32)
    return idx, new


@pytest.mark.parametrize("kind", ["move1", "move10", "move100", "radius0.1", "radius50", "motion", "ids"])
@pytest.mark.parametrize("scene", list(SCENES))
def test_updated_scene_equals_fresh_scene(ctx, earth, scene, kind):
    desc = SCENES[scene](earth)
    sph = desc.spheres()
    idx, new = _edit(kind, sph, np.random.default_rng(zlib.crc32(f"{scene}/{kind}".encode())))
    extra = towards(np.asarray(new["center0"], np.float64), 4096, 3.0, seed=5)
    upd, fresh, _ = check_update(ctx, desc, idx, new, extra_rays=extra)
    assert upd.info().bvh_mode == fresh.info().bvh_mode
    if scene == "lbvh5000":
        assert {2, 3} <= set(_walks(upd))  # the 4-wide and quantised forms exist and were compared


# ------------------------------------------------------------------------------------------------------------ adversarial

@pytest.mark.parametrize("scene", ["c2_sah", "lbvh5000"])
def test_all_spheres_on_one_point(ctx, earth, scene):
    desc = SCENES[scene](earth)
    new = desc.spheres()
    new["center0"] = F32([0.5, 1.0, -0.5])
    new["center1"] = new["center0"]
    upd, fresh, _ = check_update(ctx, desc, np.arange(len(new)), new, extra_rays=towards([[0.5, 1.0, -0.5]], 4096, 4.0, seed=7))
    hits = upd.trace_primary(towards([[0.5, 1.0, -0.5]], 1024, 1500.0, seed=8), use_bvh=1)
    assert (hits["id"] != capi.RT_INVALID_ID).any()


@pytest.mark.parametrize("scene", ["c2_sah", "lbvh5000"])
def test_one_sphere_far_outside_the_root_box(ctx, earth, scene):
    desc = SCENES[scene](earth)
    sph = desc.spheres()
    k = len(sph) // 2
    new = sph[[k]].copy()
    new["center0"] = (new["center0"] + F32([1e4, 2e4, -1e4])).astype(F32)
    new["center1"] = (new["center1"] + F32([1e4, 2e4, -1e4])).astype(F32)
    upd, _, _ = check_update(ctx, desc, [k], new, extra_rays=towards(new["center0"], 2048, 5.0, seed=9))
    got = upd.trace_primary(towards(new["center0"], 256, 5.0, seed=10), use_bvh=1)
    assert (got["id"] == sph["id"][k]).any()  # the refit tree reaches it


def test_fifty_successive_edits(ctx, earth):
    desc = SCENES["lbvh5000"](earth)
    upd = rt.Scene(ctx, desc)
    cur = desc.spheres()
    rng = np.random.default_rng(50)
    for step in range(1, 51):
        idx, new = _move(cur, rng.choice([0.001, 0.05, 0.5]), rng)
        if step % 7 == 0:
            new["radius"] = (new["radius"] * F32(rng.uniform(0.5, 3.0))).astype(F32)
        upd.update(idx, new)
        cur[idx] = new
        if step % 10 == 0:
            now = edited(desc, np.arange(len(cur)), cur)
            fresh = rt.Scene(ctx, now)
            rays = np.concatenate([camera_rays(now.desc.camera, 4096, step), towards(cur["center0"], 4096, 2.0, seed=step)])
            assert_same_hits(upd, fresh, np.concatenate([rays, secondary_rays(fresh.trace_primary(rays, use_bvh=0), 4096, step)]))


@pytest.mark.parametrize("bvh", ["sah", "lbvh"])
def test_moved_caterpillar(ctx, bvh):
    base = caterpillar(50)
    desc = from_list(base, bvh)
    sph = desc.spheres()
    rng = np.random.default_rng(3)
    new = sph.copy()
    j = rng.uniform(-0.2, 0.2, (len(sph), 3)).astype(F32)
    new["center0"] = (new["center0"] + j).astype(F32)
    new["center1"] = (new["center1"] + j).astype(F32)
    rays = towards(new["center0"], 8192, 1.5, seed=4)
    upd, _, _ = check_update(ctx, desc, np.arange(len(sph)), new, extra_rays=rays)
    assert upd.info().bvh_depth == rt.Scene(ctx, desc).info().bvh_depth  # the topology stays


def test_exact_tie_resolves_to_the_lower_ordinal(ctx, earth):
    desc = SCENES["lbvh5000"](earth)
    sph = desc.spheres()
    static = np.nonzero(~sph["flags"] & capi.RT_SPHERE_MOVING)[0]
    i, j = int(static[100]), int(static[3000])
    new = sph[[i, j]].copy()
    new["center0"] = F32([3.0, 2.0, 1.0])
    new["center1"] = new["center0"]
    new["radius"] = F32(0.7)
    new["id"] = [900001, 900002]
    rays = towards([[3.0, 2.0, 1.0]], 4096, 2.0, seed=12)
    upd, _, _ = check_update(ctx, desc, [i, j], new, extra_rays=rays)
    for u in _walks(upd):
        got = upd.trace_primary(rays, use_bvh=u)["id"]
        assert (got == 900001).mean() > 0.9 and not (got == 900002).any(), u


def test_cluster_spread_beyond_the_quantised_range(ctx, earth, monkeypatch):
    """Before the edit the quantised nodes exist; after spreading 125 spheres over 4e8 units they cannot, use_bvh = 3 is
    refused, and the persistent-lane render (which then walks the 128-byte nodes) equals the fresh scene's."""
    desc = SCENES["lbvh5000"](earth)
    sph = desc.spheres()
    upd = rt.Scene(ctx, desc)
    assert 3 in _walks(upd)
    static = np.nonzero(~sph["flags"] & capi.RT_SPHERE_MOVING)[0][1:126]  # (not the ground)
    grid = np.array([c for c, _, _ in grid_scene(1.0e8, 5, 3.5e7)], F32)
    new = sph[static].copy()
    new["center0"] = grid
    new["center1"] = grid
    new["radius"] = F32(3.5e7)
    upd.update(static, new)
    fresh = rt.Scene(ctx, edited(desc, static, new))
    assert 3 not in _walks(upd) and 3 not in _walks(fresh)
    with pytest.raises(capi.RtError) as e:
        upd.trace_primary(_PROBE, use_bvh=3)
    assert e.value.status == capi.RT_ERR_INVALID_ARG
    assert_same_hits(upd, fresh, np.concatenate([camera_rays(desc.desc.camera, 4096, 13), towards(grid, 4096, 1.5e8, seed=14)]))
    monkeypatch.setenv("RT_WF_GRAIN", "pt")
    p = rt.default_params(width=64, height=36, spp=4, max_depth=6)
    got, st = upd.render_accum(p)
    want, st0 = fresh.render_accum(p)
    _assert_same_frames(got, want)
    assert st.rays == st0.rays


# ----------------------------------------------------------------------------------------------------------------- frames

def _assert_same_frames(got, want):
    assert np.array_equal(got[..., 3], want[..., 3])
    assert np.allclose(got, want, rtol=1e-5, atol=1e-5), float(np.abs(got - want).max())


PIPES = {  # name: (scene, RT_WF_GRAIN or None, pipeline)
    "pt": ("lbvh5000", "pt", capi.RT_PIPE_WAVEFRONT),
    "warp": ("lbvh5000", "warp", capi.RT_PIPE_WAVEFRONT),
    "cta": ("lbvh5000", "cta", capi.RT_PIPE_WAVEFRONT),
    "mega": ("lbvh5000", None, capi.RT_PIPE_MEGAKERNEL),
    "c2_default": ("c2_sah", None, capi.RT_PIPE_WAVEFRONT),
    "c1_default": ("c1_list", None, capi.RT_PIPE_WAVEFRONT),
}


@pytest.mark.parametrize("tail", ["default", "0"])
@pytest.mark.parametrize("pipe", list(PIPES))
def test_frames_equal_fresh_scene(ctx, earth, monkeypatch, pipe, tail):
    scene, grain, pipeline = PIPES[pipe]
    if tail == "0":
        if pipeline == capi.RT_PIPE_MEGAKERNEL or grain == "pt":
            pytest.skip("no tail kernel on this path")
        monkeypatch.setenv("RT_WF_TAIL_PATHS", "0")
    if grain:
        monkeypatch.setenv("RT_WF_GRAIN", grain)
    desc = SCENES[scene](earth)
    idx, new = _move(desc.spheres(), 0.1, np.random.default_rng(21))
    upd = rt.Scene(ctx, desc)
    upd.update(idx, new)
    fresh = rt.Scene(ctx, edited(desc, idx, new))
    p = rt.default_params(width=80, height=45, spp=4, max_depth=8, pipeline=pipeline)
    got, st = upd.render_accum(p)
    want, st0 = fresh.render_accum(p)
    _assert_same_frames(got, want)
    assert st.rays == st0.rays and st.paths == st0.paths


def test_emitter_sampling_after_material_and_sphere_edits(ctx, earth):
    desc = SCENES["c1_list"](earth)
    mats = _materials(desc)
    sph = desc.spheres()
    kinds = [m.kind for m in mats]
    emit = [k for k, m in enumerate(mats) if m.kind == capi.RT_MAT_EMITTER]
    lamb = [k for k, m in enumerate(mats) if m.kind == capi.RT_MAT_LAMBERTIAN]
    assert emit and lamb, kinds
    p = rt.default_params(width=80, height=40, spp=8, max_depth=6, flags=capi.RT_RENDER_EMITTER_SAMPLING)
    # a lambertian becomes an emitter, an emitter a metal
    to_emitter = capi.rt_material.from_buffer_copy(mats[lamb[0]])
    to_emitter.kind = capi.RT_MAT_EMITTER
    to_emitter.param = 3.0
    to_metal = capi.rt_material(capi.RT_MAT_METAL, -1, (0.8, 0.7, 0.6), 0.2)
    upd = rt.Scene(ctx, desc)
    upd.update(material_index=[lamb[0], emit[0]], materials=[to_emitter, to_metal])
    step1 = edited(desc, material_index=[lamb[0], emit[0]], materials=[to_emitter, to_metal])
    fresh = rt.Scene(ctx, step1)
    got, st = upd.render_accum(p)
    want, st0 = fresh.render_accum(p)
    _assert_same_frames(got, want)
    assert st.rays == st0.rays
    # a sphere edit that gives a non-emitting sphere the emitter material of step 1
    k = int(np.nonzero((sph["material"] != lamb[0]) & (sph["material"] != emit[0]))[0][0])
    new = sph[[k]].copy()
    new["material"] = lamb[0]
    upd.update([k], new)
    fresh2 = rt.Scene(ctx, edited(step1, [k], new))
    got, st = upd.render_accum(p)
    want, st0 = fresh2.render_accum(p)
    _assert_same_frames(got, want)
    assert st.rays == st0.rays
    assert not np.allclose(got, rt.Scene(ctx, step1).render_accum(p)[0], rtol=1e-3, atol=1e-3)


def test_camera_edit_through_every_render_entry(ctx, earth):
    desc = SCENES["c1_list"](earth)
    cam = rt.orbit_cameras(desc.desc.camera, 4, 120.0)[1]
    upd = rt.Scene(ctx, desc)
    upd.update(camera=cam)
    fresh = rt.Scene(ctx, edited(desc, camera=cam))
    p = rt.default_params(width=96, height=48, spp=8, max_depth=8)
    a, sa = upd.render(p)
    b, sb = fresh.render(p)
    assert np.allclose(a, b, rtol=1e-5, atol=1e-5) and sa.rays == sb.rays
    assert not np.allclose(a, rt.Scene(ctx, desc).render(p)[0], rtol=1e-3, atol=1e-3)  # the camera did move
    a, sa = upd.render_progressive(p, 3)
    b, sb = fresh.render_progressive(p, 3)
    assert np.allclose(a, b, rtol=1e-5, atol=1e-5) and sa.rays == sb.rays
    a, sa = upd.render_denoised(p)
    b, sb = fresh.render_denoised(p)
    assert np.allclose(a, b, rtol=1e-4, atol=1e-4) and sa.rays == sb.rays
    ap = rt.default_adaptive_params(min_spp=8, step_spp=8, max_spp=32)
    a, spa, sa, _ = upd.render_adaptive(p, ap)
    b, spb, sb, _ = fresh.render_adaptive(p, ap)
    same = spa == spb
    assert same.mean() > 0.999, float(same.mean())  # a stopping decision at the threshold may flip with the sums' last bits
    assert np.allclose(a[same], b[same], rtol=1e-5, atol=1e-5)


# ------------------------------------------------------------------------------------------------------- identity, order

@pytest.mark.parametrize("scene", ["c1_list", "c2_sah", "lbvh5000"])
def test_identity_update(ctx, earth, scene):
    desc = SCENES[scene](earth)
    sph = desc.spheres()
    before = rt.Scene(ctx, desc)
    upd = rt.Scene(ctx, desc)
    upd.update(np.arange(len(sph)), sph, list(range(desc.desc.n_materials)), _materials(desc), desc.desc.camera)
    rays = scene_rays(desc, before, 30)
    assert_same_hits(upd, before, rays)
    p = rt.default_params(width=64, height=36, spp=4, max_depth=6)
    got, st = upd.render_accum(p)
    want, st0 = before.render_accum(p)
    _assert_same_frames(got, want)
    assert st.rays == st0.rays


def test_render_enqueued_before_an_update_sees_the_old_scene(ctx, earth):
    import torch

    desc = SCENES["lbvh5000"](earth)
    p = rt.default_params(width=96, height=54, spp=8, max_depth=6)
    want, _ = rt.Scene(ctx, desc).render_accum(p)
    upd = rt.Scene(ctx, desc)
    acc = torch.zeros((p.height, p.width, 4), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    upd.render_accum_device(p, acc.data_ptr())
    idx, new = _move(desc.spheres(), 1.0, np.random.default_rng(40))
    new["radius"] = (new["radius"] * 4).astype(F32)
    upd.update(idx, new)
    ctx.synchronize()
    _assert_same_frames(acc.cpu().numpy(), want)
    got, _ = upd.render_accum(p)
    fresh, _ = rt.Scene(ctx, edited(desc, idx, new)).render_accum(p)
    _assert_same_frames(got, fresh)


# -------------------------------------------------------------------------------------------------------------- rejected

def test_rejected_edits_leave_the_scene_unchanged(ctx, earth):
    desc = SCENES["lbvh5000"](earth)
    sph = desc.spheres()
    mats = _materials(desc)
    sc = rt.Scene(ctx, desc)
    rays = scene_rays(desc, sc, 50)
    hits0 = sc.trace_primary(rays, use_bvh=3)
    p = rt.default_params(width=64, height=36, spp=4, max_depth=6)
    frame0, st0 = sc.render_accum(p)
    moving = int(np.nonzero(sph["flags"] & capi.RT_SPHERE_MOVING)[0][0])
    static = int(np.nonzero(~sph["flags"] & capi.RT_SPHERE_MOVING)[0][1])
    moved = sph[[static, static]].copy()
    moved["center0"] += F32(5.0)
    to_moving = sph[[static]].copy()
    to_moving["flags"] |= capi.RT_SPHERE_MOVING
    to_static = sph[[moving]].copy()
    to_static["flags"] &= np.uint32(0xFFFFFFFF ^ capi.RT_SPHERE_MOVING)
    nan = sph[[static]].copy()
    nan["center0"][0, 1] = np.nan
    bad_mat = sph[[static]].copy()
    bad_mat["material"] = len(mats)
    bad_kind = capi.rt_material.from_buffer_copy(mats[0])
    bad_kind.kind = 7
    bad_tex = capi.rt_material.from_buffer_copy(mats[0])
    bad_tex.kind, bad_tex.texture = capi.RT_MAT_LAMBERTIAN, int(desc.desc.n_textures)
    bad_cam = capi.rt_camera.from_buffer_copy(desc.desc.camera)
    bad_cam.vfov = float("inf")
    cases = {
        "index out of range": dict(sphere_index=[len(sph)], spheres=moved[:1]),
        "repeated index": dict(sphere_index=[static, static], spheres=moved),
        "static to moving": dict(sphere_index=[static], spheres=to_moving),
        "moving to static": dict(sphere_index=[moving], spheres=to_static),
        "non-finite centre": dict(sphere_index=[static], spheres=nan),
        "sphere material out of range": dict(sphere_index=[static], spheres=bad_mat),
        "material index out of range": dict(material_index=[len(mats)], materials=[mats[0]]),
        "repeated material": dict(material_index=[0, 0], materials=[mats[0], mats[0]]),
        "bad material kind": dict(material_index=[0], materials=[bad_kind]),
        "bad texture index": dict(material_index=[0], materials=[bad_tex]),
        "non-finite camera": dict(sphere_index=[static], spheres=moved[:1], camera=bad_cam),
    }
    for name, kw in cases.items():
        with pytest.raises(capi.RtError) as e:
            sc.update(**kw)
        assert e.value.status == capi.RT_ERR_INVALID_ARG, name
        assert np.array_equal(_bytes(sc.trace_primary(rays, use_bvh=3)), _bytes(hits0)), name
    other = rt.Context(0)
    edit, keep = capi.scene_edit([static], moved[:1])
    assert ctx.lib.rt_scene_update(other._h, sc._h, C.byref(edit), None) == capi.RT_ERR_INVALID_ARG
    assert b"context" in ctx.lib.rt_last_error()
    assert np.array_equal(_bytes(sc.trace_primary(rays, use_bvh=3)), _bytes(hits0))
    frame, st = sc.render_accum(p)
    _assert_same_frames(frame, frame0)
    assert st.rays == st0.rays
    assert sc.update() == 0.0  # the empty edit
    assert np.array_equal(_bytes(sc.trace_primary(rays, use_bvh=3)), _bytes(hits0))
    del keep


# ------------------------------------------------------------------------------------------------------------------ multi

def test_multi_update_equals_multi_set_scene(earth):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    desc = SCENES["c2_sah"](earth)
    idx, new = _move(desc.spheres(), 0.1, np.random.default_rng(60))
    cam = rt.orbit_cameras(desc.desc.camera, 4, 60.0)[1]
    p = rt.default_params(width=96, height=54, spp=8, max_depth=6)
    m = rt.Multi([0, 1])
    m.set_scene(desc)
    m.update_scene(idx, new, camera=cam)
    got, _, st, _ = m.render(p)
    m.set_scene(edited(desc, idx, new, camera=cam))
    want, _, st0, _ = m.render(p)
    m.close()
    assert np.allclose(got, want, rtol=1e-5, atol=1e-5) and st.rays == st0.rays
