"""One shading step on the device (rt_shade_probe) against the oracle (orc_shade_probe) and the float64 restatements of
tests/test_shading.py, ray by ray and cell by cell: every material x texture kind the C ABI allows, with a minimum hit count
per cell so that no cell is skipped silently.

Rays are aimed at chosen surface points (origin = target + k n, direction = -n, plus jitter), so hits, t and the hit point
are bit-identical on both sides (asserted) and both shade the same float32 point.  Each texture value must lie within the
restatement's error bound of its float64 value; the bound holds the contraction nvcc applies and the oracle does not, and
the SFU error of __sinf / __sincosf / __powf where the kernels use them (assumed outside [-pi, pi]; the measured worst
error against the bound is recorded with record_parity).  A discrete difference — another checker leaf, a wood step of
c1 - c2, another texel, another reflect / refract choice, a metal ray absorbed on one side only — is allowed only where the
float64 quantity that decides it lies within its error bound of the threshold: a near-tie."""
import json

import numpy as np
import pytest

import raytracing_renderer_cuda_b200 as rt
from raytracing_renderer_cuda_b200 import capi
from tests.conftest import record_parity
from tests.oracle_api import camera_rays, secondary_rays
from tests.test_gpu_random_scenes import CASES, random_document
from tests.test_shading import (U, UZ, checker_chain, make_desc, probe_draws, rz32, schlick, schlick_err, tex_checker, tex_constant,
                                tex_image, tex_noise, tex_wood, texture_value, unit_ball)

pytestmark = pytest.mark.gpu

LAM, MET, DIE, EMI = capi.RT_MAT_LAMBERTIAN, capi.RT_MAT_METAL, capi.RT_MAT_DIELECTRIC, capi.RT_MAT_EMITTER
KIND = {0: "constant", 1: "checker", 2: "perlin", 3: "turbulence", 4: "marble", 5: "wood", 6: "image"}
MAT = {LAM: "lambertian", MET: "metal", DIE: "dielectric", EMI: "emitter"}


@pytest.fixture(scope="module")
def ctx():
    return rt.Context(0)


def params(seed=1000):
    return rt.default_params(seed=seed, tmin=1e-4)


def aim(centre, radius, n, k=0.5, jitter=0.0, rng=None, time=0.0, centre1=None):
    """Rays at the surface points centre + |radius| n (centre at the ray's time for a moving sphere), from k outside."""
    n = np.asarray(n, np.float64)
    n = n / np.linalg.norm(n, axis=1, keepdims=True)
    time = np.broadcast_to(np.asarray(time, np.float64), (len(n),))
    c = np.asarray(centre, np.float64)[None] + (0 if centre1 is None else time[:, None] * (np.asarray(centre1) - np.asarray(centre))[None])
    target = c + abs(radius) * n
    rays = np.zeros(len(n), capi.RAY_DTYPE)
    rays["origin"] = target + k * n
    d = -n
    if jitter:
        d = d + rng.normal(scale=jitter, size=d.shape)
    rays["direction"] = d
    rays["time"] = time
    return rays


def sphere_dirs(rng, m):
    n = rng.normal(size=(m, 3))
    return n / np.linalg.norm(n, axis=1, keepdims=True)


def check_step(desc, rays, got, orc, images=(), seed=1000, min_hits=50, label=""):
    """Every assertion of this file on one batch of probe records: `got` from the device, the oracle's from `orc`.
    Returns {cell: hits}; records the measured errors against their bounds per cell."""
    want = orc.shade_probe(rays, params(seed), arith=1)
    hits = orc.trace(rays, tmin=1e-4, arith=1)
    assert np.array_equal(got["id"], want["id"]) and np.array_equal(got["t"], want["t"]), label
    assert np.array_equal(hits["id"], want["id"])
    d = desc.desc
    sph = desc.spheres()
    by_id = {int(s["id"]): k for k, s in enumerate(sph)}
    textures = [d.textures[k] for k in range(d.n_textures)]
    mats = [d.materials[k] for k in range(d.n_materials)]
    imgs = [np.asarray(im, np.float32) for im in images]
    hit = np.nonzero(want["id"] != capi.RT_INVALID_ID)[0]
    mat_of = np.array([sph[by_id[int(i)]]["material"] for i in want["id"][hit]], np.int64)
    u1, u2, u3, u4 = (u[hit] for u in probe_draws(len(rays), seed))
    ball, berr = unit_ball(u1, u2, u3)
    p, n = hits["p"][hit], hits["n"][hit]
    g, w, r = got[hit], want[hit], rays[hit]
    bloom = np.float32(params().bloom)
    cells = {}
    for m in np.unique(mat_of):
        sel = np.nonzero(mat_of == m)[0]
        mt = mats[int(m)]
        gs, ws, rs = g[sel], w[sel], r[sel]
        cell = MAT[mt.kind] + ("" if mt.kind in (MET, DIE) else "/" + KIND[textures[mt.texture].kind])
        cells[cell] = cells.get(cell, 0) + len(sel)
        if mt.kind in (LAM, EMI):
            ref, err, tie = texture_value(textures, mt.texture, p[sel], n[sel], imgs)
            if mt.kind == LAM:
                val, wval = gs["attenuation"].astype(np.float64), ws["attenuation"].astype(np.float64)
                scale, extra = 1.0, 0.0
                assert (gs["continues"] == 1).all() and (ws["continues"] == 1).all(), (label, cell)
                assert np.array_equal(gs["scattered"]["origin"], ws["scattered"]["origin"]), (label, cell)
                assert np.array_equal(gs["scattered"]["time"], rs["time"]), (label, cell)  # lambertian keeps the ray's time
                dd = np.abs(gs["scattered"]["direction"] - ws["scattered"]["direction"]).max(axis=1)
                tol = berr[sel] + 8 * UZ * (np.abs(p[sel]).max(axis=1) + 3)  # target = p + n + ball, minus p
                assert (dd <= tol).all(), (label, cell, float((dd - tol).max()))
            else:
                scale = float(mt.param)
                val, wval = gs["emitted"].astype(np.float64) - bloom, ws["emitted"].astype(np.float64) - bloom
                extra = 4 * UZ * (np.abs(ref).max(axis=1) * scale + bloom)
                assert not gs["continues"].any() and not gs["attenuation"].any(), (label, cell)
                if textures[mt.texture].kind == capi.RT_TEX_CONSTANT:
                    assert np.array_equal(gs["emitted"], ws["emitted"]), (label, cell)  # constant emitters: bit-exact
            bound = err * scale + extra + 1e-30
            dev = np.abs(val - ref * scale).max(axis=1)
            orcd = np.abs(wval - ref * scale).max(axis=1)
            assert (dev[~tie] <= bound[~tie]).all(), (label, cell, float((dev - bound)[~tie].max()), p[sel][~tie][np.argmax((dev - bound)[~tie])])
            assert (orcd[~tie] <= bound[~tie]).all(), (label, cell, "oracle", float((orcd - bound)[~tie].max()))
            # (image_edge_rays aims at texel edges on purpose)
            assert tie.mean() < (0.5 if cell.endswith("image") else 0.1), (label, cell, float(tie.mean()))
            record_parity("shading_step", label=label, cell=cell, hits=len(sel), ties=int(tie.sum()),
                          worst_err=float(dev[~tie].max()) if (~tie).any() else 0.0,
                          worst_err_over_bound=float((dev[~tie] / np.maximum(bound[~tie], 1e-30)).max()) if (~tie).any() else 0.0)
            continue
        assert np.array_equal(gs["attenuation"], ws["attenuation"]), (label, cell)  # albedo / tint, as stored
        assert np.array_equal(gs["attenuation"], np.tile(np.float32(mt.albedo[:]), (len(sel), 1))), (label, cell)
        assert not gs["scattered"]["time"].any(), (label, cell)  # metal and dielectric reset the time to 0
        both = (gs["continues"] == 1) & (ws["continues"] == 1)
        assert np.array_equal(gs["scattered"]["origin"][both], ws["scattered"]["origin"][both]), (label, cell)
        gd, wd = gs["scattered"]["direction"].astype(np.float64), ws["scattered"]["direction"].astype(np.float64)
        if mt.kind == MET:
            rough = float(np.float32(mt.param))
            if rough == 0.0:  # the ball sample is multiplied by 0: the reflection itself, bit for bit
                assert np.array_equal(gs["continues"], ws["continues"]) and np.array_equal(gd[both], wd[both]), (label, cell)
                continue
            tol = rough * berr[sel] + 8 * UZ * (2 + rough)
            dd = np.abs(gd - wd).max(axis=1)
            assert (dd[both] <= tol[both]).all(), (label, cell, float((dd - tol)[both].max()))
            # absorbed (dot(out, n) <= 0) on one side only: only where float64 dot(out, n) is within its bound of 0
            flip = gs["continues"] != ws["continues"]
            out64 = wd + 0 * gd
            dn = np.abs((out64 * n[sel]).sum(axis=1))
            assert (dn[flip] <= (tol + 4 * UZ * np.abs(out64).sum(axis=1))[flip]).all(), (label, cell)
            record_parity("shading_step", label=label, cell=f"{cell} {rough}", hits=len(sel), absorbed=int((ws["continues"] == 0).sum()),
                          flips=int(flip.sum()), worst_err_over_bound=float((dd[both] / tol[both]).max()) if both.any() else 0.0)
            continue
        # dielectric: always continues; a reflect / refract flip only where Schlick is within the __powf bound of the draw
        assert (gs["continues"] == 1).all() and (ws["continues"] == 1).all(), (label, cell)
        flip = ~np.all(gd == wd, axis=1)
        # the cosine exactly as both sides compute it in float32 (it is singular at the critical angle, so a float64 cosine
        # would misplace the tie there): dot products rounded toward zero and summed to nearest, |d| = sqrt_rz(dot(d, d))
        pr = rz32(rs["direction"].astype(np.float64) * n[sel].astype(np.float64))
        ddn = (pr[:, 0] + pr[:, 1]) + pr[:, 2]
        sq = rz32(rs["direction"].astype(np.float64) ** 2)
        length = rz32(np.sqrt(((sq[:, 0] + sq[:, 1]) + sq[:, 2]).astype(np.float64)))
        ri = np.float32(mt.param)
        c = ddn / length
        with np.errstate(invalid="ignore"):
            leave = rz32(np.sqrt((np.float32(1) - (ri * ri) * (np.float32(1) - c * c)).astype(np.float64)))
        cos = np.where(ddn > 0, leave, -c).astype(np.float64)
        prob = schlick(cos, float(ri))
        near = np.abs(prob - u4[sel]) <= schlick_err(cos, float(ri)) + 40 * UZ
        # along the normal the float32 cosine can round above 1 (entering: -dot / |d|; leaving: sqrt_rz of 1 - ri^2 (1 - c^2)
        # with c^2 above 1): __powf(1 - cosine, 5) of a negative base is NaN on the device (the reference's __powf too) and
        # the ray refracts, while the oracle's powf gives r0 - 0
        over_one = cos > 1
        odd = np.nonzero(flip & ~near & ~over_one)[0]
        record_parity("shading_step", label=label, cell=f"{cell} {float(ri)}", hits=len(sel), flips=int(flip.sum()), near_ties=int(near.sum()),
                      cosine_above_one=int(over_one.sum()), leaving=int((ddn > 0).sum()), unexplained=int(len(odd)),
                      unexplained_rays=[dict(origin=rs[k]["origin"].tolist(), direction=rs[k]["direction"].tolist(), n=n[sel][k].tolist(), cos=float(cos[k]), prob=float(prob[k]),
                                             draw=float(u4[sel][k]), got=gd[k].tolist(), want=wd[k].tolist()) for k in odd[:4]])
        assert len(odd) == 0, (label, cell, float(ri), int(flip.sum()), len(odd))
    for cell, k in cells.items():
        assert k >= min_hits, (label, cell, k)
    return cells


# ------------------------------------------------------------------ scenes ----
def _images():
    """Sizes 1x1, 1x7, 7x1, 3x2 and 257x129, a distinct value in every texel (row 0 = top), so that a one-texel or a
    row-flip error cannot pass."""
    out = []
    for h, w in ((1, 1), (1, 7), (7, 1), (3, 2), (129, 257)):
        j, i = np.mgrid[0:h, 0:w]
        out.append(np.stack([(i + 1) / (w + 1), (j + 1) / (h + 1), (j * w + i + 1) / (w * h + 1)], -1).astype(np.float32))
    return out


def kinds_scene():
    """One sphere per material x texture kind (radius 100 for the lattice kinds: a hit point spans 800 Perlin cells at
    density 4, on both sides of 0), metal at roughness 0, 0.5, 1 and 3 (the C ABI does not clamp), dielectrics of ri 0.7,
    1, 1.5, 2.4, a tinted one and a hollow one (negative radius), emitters of intensity 0, 1 and 3, moving spheres."""
    images = _images()
    texs = [tex_constant((0.2, 0.5, 0.8)), tex_noise(capi.RT_TEX_NOISE_PERLIN, 4.0), tex_noise(capi.RT_TEX_NOISE_TURBULANCE, 2.5),
            tex_noise(capi.RT_TEX_NOISE_MARBLE, 0.1), tex_wood((0.9, 0.6, 0.2), (0.2, 0.1, 0.05), 0.15, 60.0),
            tex_checker(1, 0), tex_checker(5, 4), tex_noise(capi.RT_TEX_NOISE_MARBLE, 37.0), tex_wood((0.1, 0.8, 0.3), (0.7, 0.7, 0.9), 50, 5)]
    texs += [tex_image(k) for k in range(len(images))]
    leafs = [0, 1, 2, 3, 4, 6, 7, 8] + [9 + k for k in range(len(images))]
    mats, spheres = [], []
    big = {1, 2, 4}  # Perlin, turbulence and the wide wood: radius 100

    def add(mat, radius, centre1=False):
        # the radius-100 spheres on a row 310 apart, the small ones on a row above them near x = 0 (the checker's __sinf
        # bound grows with |10 p|, and so would the share of near-ties)
        k = len(spheres)
        nbig = sum(abs(s[1]) > 50 for s in spheres)
        c = (-620.0 + 310.0 * nbig, 5.0, 0.0) if abs(radius) > 50 else (-120.0 + 8.0 * (k - nbig), 120.0, 0.0)
        mats.append(mat)
        spheres.append((c, radius, len(mats) - 1) + (((c[0] + 3.0, c[1] + 0.5, -2.0),) if centre1 else ()))

    for t in leafs:
        add(capi.rt_material(LAM, t, (0, 0, 0), 0), 100.0 if t in big else 3.0)
    for t, inten in zip(leafs, [0.0, 1.0, 3.0] * 6):
        add(capi.rt_material(EMI, t, (0, 0, 0), inten), 100.0 if t in big else 3.0)
    for rough in (0.0, 0.5, 1.0, 3.0):
        add(capi.rt_material(MET, -1, (0.9, 0.7, 0.4), rough), 3.0)
    for ri in (0.7, 1.0, 1.5, 2.4):
        add(capi.rt_material(DIE, -1, (1, 1, 1), ri), 3.0)
    add(capi.rt_material(DIE, -1, (0.8, 0.9, 0.6), 1.5), 3.0)   # tinted
    add(capi.rt_material(DIE, -1, (1, 1, 1), 1.5), -3.0)        # hollow: the normal points in
    add(capi.rt_material(LAM, 1, (0, 0, 0), 0), 3.0, True)      # moving: Perlin at the moving hit point
    add(capi.rt_material(LAM, 6, (0, 0, 0), 0), 3.0, True)      # moving: a checker of a checker
    add(capi.rt_material(MET, -1, (0.5, 0.5, 0.5), 0.3), 3.0, True)
    add(capi.rt_material(DIE, -1, (1, 1, 1), 1.5), 3.0, True)
    return make_desc(spheres, mats, texs, images), spheres, images


def kinds_rays(spheres, m=1500, seed=0):
    r = np.random.default_rng(seed)
    out = []
    for c, rad, _, *c1 in spheres:
        moving = bool(c1)
        t = r.uniform(0, 1, m) if moving else 0.0
        n = sphere_dirs(r, m)
        out.append(aim(c, rad, n, k=0.5, jitter=0.02, rng=r, time=t, centre1=c1[0] if moving else None))
        if not moving:
            # the poles (|n.y| = 1; asinf may see |n.y| a hair above 1), the seam (n.x < 0, n.z = +-0) and grazing rays
            poles = aim(c, rad, np.array([[0, 1, 0], [0, -1, 0]] * 4, np.float64), k=1.0)
            seam = aim(c, rad, np.array([[-1, 0, 0], [-1, 0.3, 0], [-1, -0.6, 0]], np.float64), k=1.0)
            seam_neg = seam.copy()
            seam_neg["origin"][:, 2] = -0.0
            seam_neg["direction"][:, 2] = -0.0
            g = sphere_dirs(r, m // 5)
            graze = aim(c, rad, g, k=0.01)
            tang = np.cross(g, r.normal(size=g.shape))
            graze["direction"] = -g * 0.02 + tang / np.linalg.norm(tang, axis=1, keepdims=True)
            inside = np.zeros(m // 3, capi.RAY_DTYPE)  # from inside: leaving a dielectric, total internal reflection
            inside["origin"] = np.asarray(c) + 0.3 * abs(rad) * sphere_dirs(r, m // 3)
            inside["direction"] = sphere_dirs(r, m // 3)
            out += [poles, seam, seam_neg, graze, inside]
    return np.concatenate(out)


def image_edge_rays(spheres, images, seed=1):
    """Rays at texel boundaries of every image sphere: u = i / W and 1 - v = (j + 0.001) / H, nudged by +-2e-6."""
    r = np.random.default_rng(seed)
    out = []
    for (c, rad, mi), im in zip(spheres[8:13], images):
        h, w = im.shape[:2]
        us = np.concatenate([np.arange(w + 1) / w + e for e in (-2e-6, 0, 2e-6)])
        vs = np.concatenate([1 - (np.arange(h + 1) + 0.001) / h + e for e in (-2e-6, 0, 2e-6)])
        us, vs = np.clip(us, 0, 1), np.clip(vs, 1e-4, 1 - 1e-4)
        uu, vv = (a.ravel() for a in np.meshgrid(us, vs))
        keep = r.permutation(len(uu))[:3000]
        phi, theta = (1 - uu[keep]) * 2 * np.pi - np.pi, vv[keep] * np.pi - np.pi / 2
        n = np.stack([np.cos(theta) * np.cos(phi), np.sin(theta), np.cos(theta) * np.sin(phi)], 1)
        out.append(aim(c, rad, n, k=0.5))
    return np.concatenate(out)


# ------------------------------------------------------------------ tests ----
@pytest.mark.parametrize("use_bvh", [0, 1])
def test_every_material_and_texture_kind(ctx, oracle, use_bvh):
    desc, spheres, images = kinds_scene()
    desc.desc.bvh_mode = capi.RT_BVH_HOST_SAH if use_bvh else capi.RT_BVH_NONE
    rays = np.concatenate([kinds_rays(spheres), image_edge_rays(spheres, images)])
    got = rt.Scene(ctx, desc).shade_probe(rays, params(), use_bvh=bool(use_bvh))
    cells = check_step(desc, rays, got, oracle.scene(desc), images, min_hits=200, label=f"kinds bvh{use_bvh}")
    want_cells = {f"{m}/{k}" for m in ("lambertian", "emitter") for k in KIND.values() if k != "checker"}
    want_cells |= {"lambertian/checker", "emitter/checker", "metal", "dielectric"}
    assert want_cells <= set(cells), want_cells - set(cells)


@pytest.mark.parametrize("use_bvh", [0, 1])
def test_checker_chains_of_one_to_eight_levels(ctx, oracle, use_bvh):
    """Chains of 1..8 checker levels over a Perlin and a constant leaf (and over marble and wood): each resolves like the
    oracle; another leaf only where the float64 sines product is within the __sinf bound of 0."""
    texs = [tex_noise(capi.RT_TEX_NOISE_PERLIN, 3.0), tex_constant((0.9, 0.1, 0.3)), tex_noise(capi.RT_TEX_NOISE_MARBLE, 5.0),
            tex_wood((0.9, 0.6, 0.2), (0.2, 0.1, 0.05), 0.5, 20.0)]
    tops, mats = [], []
    for levels in range(1, 9):
        for ev, od in ((0, 1), (2, 3)):
            chain = checker_chain(levels, ev, od, first=len(texs))
            texs += chain
            tops.append(len(texs) - 1)
            mats.append(capi.rt_material(LAM, len(texs) - 1, (0, 0, 0), 0))
    spheres = [((-300.0 + 40.0 * k, 2.0, -1.0), 12.0, k) for k in range(len(mats))]
    desc = make_desc(spheres, mats, texs)
    desc.desc.bvh_mode = capi.RT_BVH_HOST_SAH if use_bvh else capi.RT_BVH_NONE
    r = np.random.default_rng(11)
    rays = np.concatenate([aim(c, rad, sphere_dirs(r, 2000), jitter=0.01, rng=r) for c, rad, _ in spheres])
    got = rt.Scene(ctx, desc).shade_probe(rays, params(), use_bvh=bool(use_bvh))
    check_step(desc, rays, got, oracle.scene(desc), min_hits=1000, label=f"checker chains bvh{use_bvh}")


def _refused(ctx, desc, status, needle):
    with pytest.raises(capi.RtError) as e:
        rt.Scene(ctx, desc)
    assert e.value.status == status and needle in str(e.value), str(e.value)


def test_checker_chains_deeper_than_the_device_resolves_and_cycles_are_refused(ctx):
    """Without the check, a 9-level chain was accepted and shaded white (the resolve loop's guard); now rt_scene_create
    declines it with RT_ERR_UNSUPPORTED, and a cycle with RT_ERR_INVALID_ARG, both naming the texture — used or not."""
    sph = [((0, 0, 0), 1.0, 0)]
    leaf = tex_constant((0.2, 0.4, 0.6))
    ok = make_desc(sph, [capi.rt_material(LAM, 8, (0, 0, 0), 0)], [leaf] + checker_chain(8, 0, 0, first=1))
    rt.Scene(ctx, ok)  # 8 levels: accepted
    deep = make_desc(sph, [capi.rt_material(LAM, 9, (0, 0, 0), 0)], [leaf] + checker_chain(9, 0, 0, first=1))
    _refused(ctx, deep, capi.RT_ERR_UNSUPPORTED, "texture 9 nests 9 checker levels")
    unused = make_desc(sph, [capi.rt_material(LAM, 0, (0, 0, 0), 0)], [leaf] + checker_chain(9, 0, 0, first=1))
    _refused(ctx, unused, capi.RT_ERR_UNSUPPORTED, "texture 9")
    # the message names the checker whose child closes the cycle on the walk from the lowest index
    for texs, k in (([leaf, tex_checker(1, 0)], 1), ([leaf, tex_checker(2, 0), tex_checker(0, 1)], 2),
                    ([leaf, tex_checker(0, 3), tex_checker(0, 0), tex_checker(2, 1)], 3)):
        _refused(ctx, make_desc(sph, [capi.rt_material(LAM, 0, (0, 0, 0), 0)], texs), capi.RT_ERR_INVALID_ARG,
                 f"checker texture {k} is its own descendant")
    # the JSON front-end can express the chain: "c1": checker(a, a), "c2": checker(c1, c1), ...
    textures = {"a": {"type": "constant", "color": [0.2, 0.4, 0.6]}, "c1": {"type": "checker", "even": "a", "odd": "a"}}
    for k in range(2, 10):
        textures[f"c{k}"] = {"type": "checker", "even": f"c{k - 1}", "odd": f"c{k - 1}"}
    doc = {"camera": {"lookfrom": [0, 0, 5], "lookat": [0, 0, 0], "up": [0, 1, 0], "vfov": 40, "aspect": 1.5},
           "textures": textures, "materials": {"m": {"type": "lambertian", "texture": "c9"}},
           "objects": [{"type": "sphere", "center": [0, 0, 0], "radius": 1, "material": "m"}]}
    with pytest.raises(capi.RtError) as e:
        rt.Scene(ctx, rt.SceneDesc.from_json(json.dumps(doc)))
    assert e.value.status == capi.RT_ERR_UNSUPPORTED and "nests 9 checker levels" in str(e.value), str(e.value)
    doc["materials"]["m"]["texture"] = "c8"
    del textures["c9"]
    rt.Scene(ctx, rt.SceneDesc.from_json(json.dumps(doc)))


@pytest.mark.parametrize("seed,n", CASES)
def test_random_documents_step_by_step(ctx, oracle, seed, n):
    """The random documents of test_gpu_random_scenes.py, ray by ray, with every per-cell assertion above."""
    d = rt.SceneDesc.from_json(random_document(seed, n))
    orc = oracle.scene(d)
    rays = camera_rays(d, 100_000, seed=7)
    first = orc.trace(rays, tmin=1e-4, arith=1)
    rays = np.concatenate([rays, secondary_rays(d, first, seed=8)[:100_000]])
    got = rt.Scene(ctx, d).shade_probe(rays, params(), use_bvh=True)
    check_step(d, rays, got, orc, min_hits=1 if n < 40 else 20, label=f"random {seed}")
