"""Scene updates from device memory on the B200: rt_scene_update_device against rt_scene_update of the same records and
against rt_scene_create of the edited description.

Closest hits must be bit-identical to both for every use_bvh the scenes share, renders must have equal sample and ray counts
and sums equal up to the order of float additions.  Covers every scene and edit kind of test_gpu_scene_update.py, the
packing of motion vectors (rounded toward zero) and durations (rounded to nearest), the emitter list, rejected edits (the
same status and message as the host entry, the scene unchanged, pointers refused before any kernel reads them), stream
ordering against earlier renders and against records produced by torch on the context's stream, and repeated steps."""
import ctypes as C
import zlib

import numpy as np
import pytest

import raytracing_renderer_cuda_b200 as rt
from raytracing_renderer_cuda_b200 import capi
from tests.test_gpu_scene_update import (SCENES, _assert_same_frames, _bytes, _edit, _materials, _move, _walks, assert_same_hits,
                                         camera_rays, edited, scene_rays, secondary_rays, towards)

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

F32 = np.float32


@pytest.fixture(scope="module")
def ctx():
    return rt.Context(0)


def on_device(idx, sph, as_bytes=False):
    """The edit as CUDA tensors: int32 indices and float32 (n, 12) or uint8 (n, 48) records, ready on the device."""
    sph = np.ascontiguousarray(sph, dtype=capi.SPHERE_DTYPE)
    raw = sph.view(np.uint8).reshape(len(sph), 48)
    i = torch.from_numpy(np.asarray(idx, np.int64).astype(np.int32)).cuda()
    r = torch.from_numpy(raw.copy()).cuda() if as_bytes else torch.from_numpy(raw.view(np.float32).copy()).cuda()
    torch.cuda.synchronize()
    return i, r


def device_update(ctx, desc, idx, sph, as_bytes=False):
    sc = rt.Scene(ctx, desc)
    ms = sc.update_device(*on_device(idx, sph, as_bytes))
    assert ms >= 0.0
    return sc


def assert_equal_scenes(a, b, rays):
    """Bit-identical hits of two scenes with the same tree for every walk."""
    assert _walks(a) == _walks(b)
    for u in _walks(a):
        got, want = _bytes(a.trace_primary(rays, use_bvh=u)), _bytes(b.trace_primary(rays, use_bvh=u))
        assert np.array_equal(got, want), (u, int((got != want).any(axis=1).sum()))


def assert_same_render(a, b, p):
    got, st = a.render_accum(p)
    want, st0 = b.render_accum(p)
    _assert_same_frames(got, want)
    assert st.rays == st0.rays and st.paths == st0.paths


# ------------------------------------------------------------------------------------------------ host path, fresh scene

@pytest.mark.parametrize("kind", ["move1", "move10", "move100", "radius0.1", "radius50", "motion", "ids"])
@pytest.mark.parametrize("scene", list(SCENES))
def test_device_update_equals_host_update_and_fresh_scene(ctx, earth, scene, kind):
    desc = SCENES[scene](earth)
    idx, new = _edit(kind, desc.spheres(), np.random.default_rng(zlib.crc32(f"{scene}/{kind}".encode())))
    dev = device_update(ctx, desc, idx, new, as_bytes=kind == "ids")
    host = rt.Scene(ctx, desc)
    host.update(idx, new)
    now = edited(desc, idx, new)
    fresh = rt.Scene(ctx, now)
    rays = np.concatenate([scene_rays(now, fresh, 3), towards(np.asarray(new["center0"], np.float64), 4096, 3.0, seed=5)])
    assert_same_hits(dev, fresh, rays)
    assert_equal_scenes(dev, host, rays)
    p = rt.default_params(width=64, height=36, spp=4, max_depth=6)
    assert_same_render(dev, host, p)
    assert_same_render(dev, fresh, p)


def _rz(exact, rn):
    """float32 round-toward-zero of `exact` (float64), given its round-to-nearest `rn`."""
    over = np.abs(rn.astype(np.float64)) > np.abs(exact)
    return np.where(over, np.nextafter(rn, F32(0)), rn).astype(F32)


def test_packing_rounds_like_the_host_packer(ctx, earth):
    """Moving spheres whose c1 - c0 and t1 - t0 differ rounded toward zero and rounded to nearest (the packers round the
    first toward zero, the second to nearest), probed at ray times next to time1, where both decide the centre."""
    desc = SCENES["lbvh5000"](earth)
    sph = desc.spheres()
    rng = np.random.default_rng(77)
    idx = np.nonzero(sph["flags"] & capi.RT_SPHERE_MOVING)[0][:200]
    new = sph[idx].copy()
    # (ends whose magnitudes differ by more than a factor of two: their difference is rarely exact in float32)
    c0 = (rng.choice([-1.0, 1.0], (len(idx), 3)) * rng.uniform(0.1, 1.0, (len(idx), 3))).astype(F32)
    c1 = (c0 * rng.uniform(2.5, 4.0, (len(idx), 3))).astype(F32)
    t0 = rng.uniform(-0.3, 0.1, len(idx)).astype(F32)
    t1 = rng.uniform(0.7, 1.1, len(idx)).astype(F32)
    new["center0"], new["center1"], new["time0"], new["time1"] = c0, c1, t0, t1
    d_exact = c1.astype(np.float64) - c0.astype(np.float64)
    assert (_rz(d_exact, c1 - c0) != c1 - c0).mean() > 0.2  # the two roundings differ for many of the motion vectors ...
    t_exact = t1.astype(np.float64) - t0.astype(np.float64)
    assert (_rz(t_exact, t1 - t0) != t1 - t0).mean() > 0.2  # ... and of the durations
    dev = device_update(ctx, desc, idx, new)
    host = rt.Scene(ctx, desc)
    host.update(idx, new)
    fresh = rt.Scene(ctx, edited(desc, idx, new))
    rays = towards(np.asarray(c1, np.float64), 16384, 1.5, seed=78)
    rays["time"] = np.minimum(rng.uniform(0.6, 1.0, len(rays)), 1.0).astype(F32)
    hit = host.trace_primary(rays, use_bvh=0)["id"]
    assert (hit != capi.RT_INVALID_ID).mean() > 0.5
    assert_equal_scenes(dev, host, rays)
    # the brute-force list does not depend on the tree: the records equal those rt_scene_create packs
    assert np.array_equal(_bytes(dev.trace_primary(rays, use_bvh=0)), _bytes(fresh.trace_primary(rays, use_bvh=0)))


# --------------------------------------------------------------------------------------------------------- emitter list

@pytest.mark.parametrize("scene", ["c1_list", "lbvh5000"])
def test_emitter_list_after_device_edits(ctx, earth, scene):
    desc = SCENES[scene](earth)
    mats = _materials(desc)
    sph = desc.spheres()
    emit = [k for k, m in enumerate(mats) if m.kind == capi.RT_MAT_EMITTER]
    other = [k for k, m in enumerate(mats) if m.kind != capi.RT_MAT_EMITTER]
    p = rt.default_params(width=80, height=40, spp=8, max_depth=6, flags=capi.RT_RENDER_EMITTER_SAMPLING)
    if not emit:  # give the scene an emitter material through the host entry first (materials stay with it)
        to_emitter = capi.rt_material.from_buffer_copy(mats[other[0]])
        to_emitter.kind, to_emitter.param = capi.RT_MAT_EMITTER, 4.0
        to_emitter.texture = max(to_emitter.texture, 0)
        desc = edited(desc, material_index=[other[0]], materials=[to_emitter])
        mats[other[0]] = to_emitter
        emit, other = [other[0]], other[1:]
    lit = np.nonzero(np.isin(sph["material"], emit))[0]
    dark = np.nonzero(~np.isin(sph["material"], emit))[0]
    cur = desc.spheres()
    sc = rt.Scene(ctx, desc)
    # step 1: two dark spheres become emitters; step 2: an emitter (if any) goes dark and a third sphere lights up
    steps = [dark[[0, len(dark) // 2]]] + ([np.array([lit[0], dark[-1]])] if len(lit) else [dark[[-1]]])
    for k, idx in enumerate(steps):
        new = cur[idx].copy()
        new["material"] = [other[0] if cur["material"][i] in emit else emit[0] for i in idx]
        sc.update_device(*on_device(idx, new))
        cur[idx] = new
        fresh = rt.Scene(ctx, edited(desc, np.arange(len(cur)), cur))
        assert_same_render(sc, fresh, p)


# ------------------------------------------------------------------------------------------------------------- rejected

def _host_error(ctx, desc, idx, sph):
    sc = rt.Scene(ctx, desc)
    with pytest.raises(capi.RtError) as e:
        sc.update(idx, sph)
    return e.value.status, str(e.value)


def test_rejected_edits_leave_the_scene_unchanged(ctx, earth):
    desc = SCENES["lbvh5000"](earth)
    sph = desc.spheres()
    mats = _materials(desc)
    sc = rt.Scene(ctx, desc)
    rays = scene_rays(desc, sc, 50)
    hits0 = _bytes(sc.trace_primary(rays, use_bvh=3))
    p = rt.default_params(width=64, height=36, spp=4, max_depth=6)
    frame0, st0 = sc.render_accum(p)
    moving = int(np.nonzero(sph["flags"] & capi.RT_SPHERE_MOVING)[0][0])
    static = np.nonzero(~sph["flags"] & capi.RT_SPHERE_MOVING)[0]
    s1 = int(static[1])
    moved = sph[[s1, s1]].copy()
    moved["center0"] += F32(5.0)
    to_moving = sph[[s1]].copy()
    to_moving["flags"] |= capi.RT_SPHERE_MOVING
    to_static = sph[[moving]].copy()
    to_static["flags"] &= np.uint32(0xFFFFFFFF ^ capi.RT_SPHERE_MOVING)
    nan = sph[[s1]].copy()
    nan["center0"][0, 1] = np.nan
    inf_t = sph[[s1]].copy()
    inf_t["time1"] = np.inf
    bad_mat = sph[[s1]].copy()
    bad_mat["material"] = len(mats)
    # a large edit with two bad records far apart, the earlier one breaking a later rule
    big_idx = static[2:2002].copy()
    big = sph[big_idx].copy()
    big["center0"] += F32(0.01)
    big["center1"] = big["center0"]
    big["radius"][1500] = np.nan            # position 1500: not finite (the fifth rule)
    big_idx[1700] = len(sph) + 3            # position 1700: out of range (the first rule)
    big_idx_rep = static[2:2002].copy()
    big_idx_rep[1900] = big_idx_rep[40]     # position 1900 repeats position 40 ...
    big_rep = sph[big_idx_rep].copy()
    big_rep["flags"][1950] |= capi.RT_SPHERE_MOVING  # ... and 1950 changes its kind: the repeat is reported
    cases = {
        "index out of range": ([len(sph)], moved[:1]),
        "repeated index": ([s1, s1], moved),
        "static to moving": ([s1], to_moving),
        "moving to static": ([moving], to_static),
        "non-finite centre": ([s1], nan),
        "non-finite time": ([s1], inf_t),
        "sphere material out of range": ([s1], bad_mat),
        "earlier position, later rule": (big_idx, big),
        "repeat before a kind change": (big_idx_rep, big_rep),
    }
    for name, (idx, new) in cases.items():
        want = _host_error(ctx, desc, idx, new)
        with pytest.raises(capi.RtError) as e:
            sc.update_device(*on_device(idx, new))
        assert (e.value.status, str(e.value)) == want, name
        assert np.array_equal(_bytes(sc.trace_primary(rays, use_bvh=3)), hits0), name
    assert "not finite" in _host_error(ctx, desc, big_idx, big)[1]
    assert "repeated" in _host_error(ctx, desc, big_idx_rep, big_rep)[1]

    lib = ctx.lib
    n = 2
    idx_np = np.array([s1, int(static[2])], np.uint32)
    rec_np = sph[idx_np].copy()
    i_dev, r_dev = on_device(idx_np, rec_np, as_bytes=True)
    # host memory, for either array: refused before any kernel reads it
    for ip, rp in ((idx_np.ctypes.data, r_dev.data_ptr()), (i_dev.data_ptr(), rec_np.ctypes.data)):
        assert lib.rt_scene_update_device(ctx._h, sc._h, C.c_void_p(ip), C.c_void_p(rp), n, None) == capi.RT_ERR_INVALID_ARG
        assert b"device" in lib.rt_last_error()
    # records 4 bytes off the 16-byte alignment (the buffer still holds n whole records from there)
    buf = torch.zeros(n * 48 + 16, dtype=torch.uint8, device="cuda")
    buf[4:4 + n * 48] = r_dev.view(-1)
    torch.cuda.synchronize()
    with pytest.raises(capi.RtError) as e:
        sc.update_device(i_dev, buf[4:4 + n * 48].view(n, 48))
    assert e.value.status == capi.RT_ERR_INVALID_ARG and "aligned" in str(e.value)
    # indices 2 bytes off the 4-byte alignment (n whole indices from there)
    ibuf = torch.zeros(4 * n + 8, dtype=torch.uint8, device="cuda")
    ibuf[2:2 + 4 * n] = i_dev.view(torch.uint8)
    torch.cuda.synchronize()
    assert lib.rt_scene_update_device(ctx._h, sc._h, C.c_void_p(ibuf.data_ptr() + 2), C.c_void_p(r_dev.data_ptr()), n, None) \
        == capi.RT_ERR_INVALID_ARG
    assert b"aligned" in lib.rt_last_error()
    other = rt.Context(0)
    assert lib.rt_scene_update_device(other._h, sc._h, C.c_void_p(i_dev.data_ptr()), C.c_void_p(r_dev.data_ptr()), n, None) \
        == capi.RT_ERR_INVALID_ARG
    assert b"context" in lib.rt_last_error()
    other.close()
    # the empty edit: a no-op, NULL pointers allowed
    ms = C.c_float(-1.0)
    assert lib.rt_scene_update_device(ctx._h, sc._h, None, None, 0, C.byref(ms)) == capi.RT_OK and ms.value == 0.0
    assert sc.update_device(*on_device(np.zeros(0, np.uint32), np.zeros(0, capi.SPHERE_DTYPE))) == 0.0

    assert np.array_equal(_bytes(sc.trace_primary(rays, use_bvh=3)), hits0)
    frame, st = sc.render_accum(p)
    _assert_same_frames(frame, frame0)
    assert st.rays == st0.rays
    # and the scene still takes a valid edit
    idx, new = _move(sph, 0.1, np.random.default_rng(51))
    sc.update_device(*on_device(idx, new))
    assert_same_hits(sc, rt.Scene(ctx, edited(desc, idx, new)), rays)


# ------------------------------------------------------------------------------------------------ small and empty scenes

def test_constant_bank_list_with_moving_spheres_before_static_ones(ctx):
    """A list scene small enough for the constant bank whose moving spheres come first in list order, so list ordinals and
    device indices (static spheres stored first) differ: both entries must write the constant-bank copy by device index."""
    from tests.test_gpu_bvh_adversarial import _doc

    spheres = [((0.2 * k, 0.1 * k, 1.0 + 0.3 * k), 0.25, (0.2 * k + 0.3, 0.1 * k, 1.0 + 0.3 * k) if k < 4 else None)
               for k in range(10)]
    desc = rt.SceneDesc.from_json(_doc(spheres, "none"))
    sph = desc.spheres()
    assert list(sph["flags"] & capi.RT_SPHERE_MOVING) == [1] * 4 + [0] * 6
    rng = np.random.default_rng(90)
    idx = np.array([0, 2, 5, 9])  # two moving, two static
    new = sph[idx].copy()
    j = rng.uniform(-0.2, 0.2, (len(idx), 3)).astype(F32)
    new["center0"] = (new["center0"] + j).astype(F32)
    new["center1"] = (new["center1"] + j).astype(F32)
    new["radius"] = (new["radius"] * F32(1.5)).astype(F32)
    dev = device_update(ctx, desc, idx, new)
    host = rt.Scene(ctx, desc)
    host.update(idx, new)
    now = edited(desc, idx, new)
    fresh = rt.Scene(ctx, now)
    assert fresh.info().n_nodes == 0 and _walks(dev) == [0]
    rays = np.concatenate([towards(np.asarray(new["center0"], np.float64), 4096, 1.5, seed=91),
                           towards(np.asarray(sph["center0"], np.float64), 4096, 1.5, seed=92)])
    want = _bytes(fresh.trace_primary(rays, use_bvh=0))
    assert (fresh.trace_primary(rays, use_bvh=0)["id"] != capi.RT_INVALID_ID).mean() > 0.3
    for sc in (dev, host):
        assert np.array_equal(_bytes(sc.trace_primary(rays, use_bvh=0)), want)
    p = rt.default_params(width=64, height=36, spp=4, max_depth=6)
    assert_same_render(dev, fresh, p)
    assert_same_render(host, fresh, p)


def test_updates_of_a_scene_without_spheres(ctx, earth):
    """A scene of materials only: a material edit through the host entry, with its device time requested, completes (its
    timing window ends with no device work after it); the device entry refuses every index (none is in range) and takes
    the empty edit."""
    base = SCENES["c1_list"](earth)
    d = capi.rt_scene_desc()
    C.memmove(C.byref(d), C.byref(base.desc), C.sizeof(d))
    d.n_spheres = 0
    desc = rt.SceneDesc(C.pointer(d), base._lib, keepalive=(base, d))
    sc = rt.Scene(ctx, desc)
    assert sc.info().n_spheres == 0
    mats = _materials(base)
    m = capi.rt_material.from_buffer_copy(mats[0])
    m.param = 2.5
    for _ in range(20):
        assert sc.update(material_index=[0], materials=[m]) >= 0.0
    with pytest.raises(capi.RtError) as e:
        sc.update_device(*on_device([0], base.spheres()[:1]))
    assert e.value.status == capi.RT_ERR_INVALID_ARG and "out of range" in str(e.value)
    assert sc.update_device(*on_device(np.zeros(0, np.uint32), np.zeros(0, capi.SPHERE_DTYPE))) == 0.0


# ------------------------------------------------------------------------------------------------------------- ordering

def test_render_enqueued_before_a_device_update_sees_the_old_scene(ctx, earth):
    desc = SCENES["lbvh5000"](earth)
    p = rt.default_params(width=96, height=54, spp=8, max_depth=6)
    want, _ = rt.Scene(ctx, desc).render_accum(p)
    idx, new = _move(desc.spheres(), 1.0, np.random.default_rng(40))
    new["radius"] = (new["radius"] * 4).astype(F32)
    i_dev, r_dev = on_device(idx, new)
    upd = rt.Scene(ctx, desc)
    acc = torch.zeros((p.height, p.width, 4), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    upd.render_accum_device(p, acc.data_ptr())
    upd.update_device(i_dev, r_dev)
    ctx.synchronize()
    _assert_same_frames(acc.cpu().numpy(), want)
    got, _ = upd.render_accum(p)
    fresh, _ = rt.Scene(ctx, edited(desc, idx, new)).render_accum(p)
    _assert_same_frames(got, fresh)


def test_records_from_torch_on_the_context_stream(earth):
    """With the context on torch's stream, records a torch op has just produced (not synchronised) are what the update
    reads; overwriting them after the call returns changes nothing."""
    desc = SCENES["lbvh5000"](earth)
    sph = desc.spheres()
    stream = torch.cuda.Stream()
    c = rt.Context(0)
    c.set_stream(stream.cuda_stream)
    dev = rt.Scene(c, desc)
    base = torch.from_numpy(np.ascontiguousarray(sph).view(np.uint8).reshape(len(sph), 48).view(np.float32).copy()).cuda()
    torch.cuda.synchronize()
    with torch.cuda.stream(stream):
        g = torch.Generator(device="cuda").manual_seed(9)
        jitter = (torch.rand((len(sph), 3), device="cuda", generator=g) * 2 - 1) * base[:, 3:4].abs() * 0.5
        rec = base.clone()
        rec[:, 0:3] += jitter
        rec[:, 4:7] += jitter
        idx = torch.arange(len(sph), device="cuda", dtype=torch.int32)
        dev.update_device(idx, rec)
        rec.fill_(float("nan"))
        idx.fill_(0)
    c.synchronize()
    moved = base.clone()
    moved[:, 0:3] += jitter
    moved[:, 4:7] += jitter
    new = moved.cpu().numpy().view(np.uint8).reshape(-1).view(capi.SPHERE_DTYPE).copy()
    host = rt.Scene(c, desc)
    host.update(np.arange(len(sph)), new)
    now = edited(desc, np.arange(len(sph)), new)
    fresh = rt.Scene(c, now)
    rays = np.concatenate([scene_rays(now, fresh, 60), towards(np.asarray(new["center0"], np.float64), 4096, 2.0, seed=61)])
    assert_equal_scenes(dev, host, rays)
    assert_same_hits(dev, fresh, rays)
    del dev, host, fresh
    c.close()


# --------------------------------------------------------------------------------------------------------- repeated steps

def test_fifty_successive_device_edits(ctx, earth):
    desc = SCENES["lbvh5000"](earth)
    dev = rt.Scene(ctx, desc)
    host = rt.Scene(ctx, desc)
    cur = desc.spheres()
    rng = np.random.default_rng(50)
    for step in range(1, 51):
        idx, new = _move(cur, rng.choice([0.001, 0.05, 0.5]), rng)
        if step % 7 == 0:
            new["radius"] = (new["radius"] * F32(rng.uniform(0.5, 3.0))).astype(F32)
        dev.update_device(*on_device(idx, new, as_bytes=step % 2 == 0))
        host.update(idx, new)
        cur[idx] = new
        if step % 10 == 0:
            now = edited(desc, np.arange(len(cur)), cur)
            fresh = rt.Scene(ctx, now)
            rays = np.concatenate([camera_rays(now.desc.camera, 4096, step), towards(cur["center0"], 4096, 2.0, seed=step)])
            rays = np.concatenate([rays, secondary_rays(fresh.trace_primary(rays, use_bvh=0), 4096, step)])
            assert_same_hits(dev, fresh, rays)
            assert_equal_scenes(dev, host, rays)
    rays = scene_rays(desc, dev, 70)
    before = _bytes(dev.trace_primary(rays, use_bvh=1))
    assert dev.update_device(*on_device(np.zeros(0, np.uint32), np.zeros(0, capi.SPHERE_DTYPE), as_bytes=True)) == 0.0
    assert np.array_equal(_bytes(dev.trace_primary(rays, use_bvh=1)), before)
