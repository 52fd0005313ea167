"""The four walks of a scene's tree — binary (use_bvh = 1), 4-wide (2), quantised 4-wide (3, what k_wf_step_pt walks) and,
in the renders, the speculative warp walk — against the brute-force list on trees built to break them: a caterpillar as
deep as the builder accepts, the outsized-sphere chain on top of a deep LBVH, thousands of exact ties, flat and collinear
scenes, coordinates far from the origin and extents that change the quantisation unit, and rays with zero direction
components, origins on box faces, tangents and several tmin.

Every case states what each builder does with it (accepts, or rejects with RT_ERR_UNSUPPORTED) and whether the quantised
nodes exist, so nothing is skipped silently.  Accepted trees must give (id, t, p, n) bit-identical to the list for every
ray; the list itself is checked against the oracle where that is affordable, and every hit against a float64 restatement
of the ray-sphere intersection.  The scenes keep the float32 quadratic well conditioned (no grazing hits from far away),
so no phantom hit needs to be excused."""
import json

import numpy as np
import pytest

import raytracing_renderer_cuda_b200 as rt
from raytracing_renderer_cuda_b200 import capi

pytestmark = pytest.mark.gpu

F32 = np.float32
MAX_DEPTH = 64  # RT_BVH_STACK_DEPTH: the deepest tree rt_scene_create accepts


@pytest.fixture(scope="module")
def ctx():
    return rt.Context(0)


# ---------------------------------------------------------------------------------------------------------------- scenes
# A scene is a list of (center0, radius, center1 or None); center1 makes a moving sphere over the shutter [0, 1].

def _f(x):
    return float(F32(x))  # exactly representable: the JSON number is the float32 value


def _doc(spheres, bvh, camera=None, emitters=False):
    """The scene document; with `emitters`, materials m1 and m3 emit (every other one is lambertian)."""
    colours = ((0.9, 0.2, 0.2), (0.2, 0.9, 0.2), (0.2, 0.2, 0.9), (0.8, 0.8, 0.3), (0.5, 0.5, 0.5))
    objs = []
    for k, (c0, r, c1) in enumerate(spheres):
        if c1 is None:
            objs.append({"type": "sphere", "center": [_f(v) for v in c0], "radius": _f(r), "material": f"m{k % 5}"})
        else:
            objs.append({"type": "moving_sphere", "center0": [_f(v) for v in c0], "center1": [_f(v) for v in c1], "time0": 0.0,
                         "time1": 1.0, "radius": _f(r), "material": f"m{k % 5}"})
    cam = camera or {"lookfrom": [0.1, 0.1, 0.1], "lookat": [1, 1, 1], "vfov": 60, "aspect": 1.5}
    return json.dumps({"camera": {"up": [0, 1, 0], "time0": 0, "time1": 1, **cam},
                       "textures": {f"t{k}": {"type": "constant", "color": list(c)} for k, c in enumerate(colours)},
                       "materials": {f"m{k}": {"type": "emitter" if emitters and k % 2 else "lambertian", "texture": f"t{k}"}
                                     for k in range(len(colours))},
                       "objects": objs, "bvh": bvh})


def _cell(j):
    """Spine point j of the caterpillar: on axis j mod 3 at (2^(20 - L) + 1/2) / 2^21, L = j // 3.  With the centroid bounds
    [0, 1] of the scene every such point sets one Morton bit of its own, and the half-cell offset keeps it robust against the
    rounding of the box centre; the codes fall strictly with j, so the Karras tree peels one spine point off per level."""
    c = [0.0, 0.0, 0.0]
    c[j % 3] = (2.0 ** (20 - j // 3) + 0.5) / 2.0 ** 21
    return c


def caterpillar(k, extra=0, moving=True):
    """Two spheres of radius 1 at every spine point (the second one hollow, radius -1, at odd j: same box and the same t,
    the other normal), `extra` more copies at the deepest point, an anchor at (1, 1, 1) that fixes the centroid bounds and,
    with `moving`, two spheres with a long motion on the far side of the anchor's Morton cell.  The LBVH is K levels deep
    (K + 1 or K + 2 with extra copies at the bottom, whose equal codes split by index); every box contains the region around
    the origin, so a ray from there enters all of them at tmin and the walk order is the slot order."""
    s = []
    for j in range(k):
        s += [(_cell(j), 1.0, None), (_cell(j), -1.0 if j % 2 else 1.0, None)]
    s += [(_cell(k - 1), 1.0, None)] * extra
    s.append(([1.0, 1.0, 1.0], 0.05, None))
    if moving:
        s += [([0.9, 0.6, 0.6], 0.05, [0.6, 0.9, 0.9]), ([0.6, 0.9, 0.6], 0.04, [0.9, 0.6, 0.95])]
    return s


def chain_scene(n_big, k=30, n_small=3000, seed=5):
    """`n_big` outsized spheres (radius 150, far above 32x the median radius 0.05) first in the list: the first 32 are hung
    above the LBVH as a chain (root -> (big_31, (... (big_0, LBVH)))), a 33rd stays in the LBVH.  Below, a caterpillar of
    depth k and a few thousand small spheres in the cube's far corner, so that chain + LBVH is 61-62 levels deep.  The big
    spheres sit around (200, 200, 200): a ray from near the origin enters their boxes late, so the 4-wide walk goes down the
    LBVH first and keeps two chain leaves per 4-wide chain node on its stack while it does."""
    rng = np.random.default_rng(seed)
    s = [([200.0 + 3 * (b % 5), 200.0 - 2 * (b % 7), 200.0 + (b % 3)], 150.0 + b, None) for b in range(min(n_big, 32))]
    if n_big > 32:  # the 33rd: outsized too, but centred in the cube so that it leaves the LBVH's Morton frame alone
        s.append(([0.75, 0.75, 0.75], 150.0, None))
    s += caterpillar(k, moving=False)
    s += [(list(map(float, p)), 0.05, None) for p in rng.uniform(0.75, 0.95, (n_small, 3)).astype(F32)]
    return s


def tie_scene(seed=7):
    """5000 spheres with the same centre and radius (every third one hollow: the same t, the other normal), 30 groups of 8
    duplicates at random positions, and 60 moving spheres with a motion of 3 units: k_topology splits equal Morton codes by
    index, the SAH binning sees zero centroid extent, and every walk must resolve the tie to the lowest list ordinal."""
    rng = np.random.default_rng(seed)
    s = [([0.0, 0.0, 0.0], -1.0 if k % 3 == 2 else 1.0, None) for k in range(5000)]
    for c in rng.uniform(-4, 4, (30, 3)):
        s += [(list(c), 0.3, None)] * 8
    for c in rng.uniform(-4, 4, (60, 3)):
        s.append((list(c), 0.2, list(c + rng.uniform(-3, 3, 3))))
    return s


def line_scene():
    """3000 overlapping spheres on the x axis: every Morton bit comes from one axis."""
    return [([0.05 * k, 0.0, 0.0], 0.08, None) for k in range(3000)]


def plane_scene():
    """A 64 x 64 grid of spheres in the plane y = 0: Morton bits from two axes, zero extent in the third."""
    return [([float(x), 0.0, float(z)], 0.45, None) for x in range(64) for z in range(64)]


def cluster_scene(offset, n=2000, seed=11):
    """Random spheres of radius 1-3 in a 100-unit cube centred on `offset` (1e5, 1e6: coordinates whose ulp is 1/128 and
    1/16, box padding of several units)."""
    rng = np.random.default_rng(seed)
    c = rng.uniform(-50, 50, (n, 3)) + np.array(offset)
    r = rng.uniform(1, 3, n)
    return [(list(c[k]), float(r[k]), None) for k in range(n)]


def grid_scene(spacing, m, radius):
    """m^3 spheres on a cubic grid about the origin: extent (m - 1) * spacing."""
    g = (np.arange(m) - (m - 1) / 2) * spacing
    return [([float(x), float(y), float(z)], radius, None) for x in g for y in g for z in g]


# ------------------------------------------------------------------------------------------------------------------ rays

def _rays(o, d, time=None):
    r = np.zeros(len(o), capi.RAY_DTYPE)
    r["origin"] = np.asarray(o, F32)
    r["direction"] = np.asarray(d, F32)
    r["time"] = np.asarray(time, F32) if time is not None else 0.5
    return r


def inside_rays(n, lo, hi, seed, dmin=0.05):
    """Origins uniform in [lo, hi]^3, directions with positive components in [dmin, 1]."""
    rng = np.random.default_rng(seed)
    return _rays(rng.uniform(lo, hi, (n, 3)), rng.uniform(dmin, 1.0, (n, 3)), rng.random(n))


def axis_rays(n, lo, hi, seed):
    """Origins uniform in [lo, hi]^3, directions along +-x, +-y, +-z whose other two components are +0.0 or -0.0 (the
    +-2^100 path of trav_begin)."""
    rng = np.random.default_rng(seed)
    d = np.zeros((n, 3), F32)
    axis = rng.integers(0, 3, n)
    d[np.arange(n), axis] = rng.choice([-1.0, 1.0], n) * rng.uniform(0.5, 2.0, n)
    zero = np.where(rng.random((n, 3)) < 0.5, F32(0.0), F32(-0.0))
    d = np.where(d == 0, zero, d)
    return _rays(rng.uniform(lo, hi, (n, 3)), d, rng.random(n))


def towards_rays(n, spheres, dist, seed, spread=0.8):
    """From `dist` away, aimed at random spheres (pass through within spread * r of the centre, so the hit is well
    conditioned)."""
    rng = np.random.default_rng(seed)
    idx = rng.integers(0, len(spheres), n)
    c = np.array([spheres[k][0] for k in idx], np.float64)
    r = np.abs(np.array([spheres[k][1] for k in idx], np.float64))
    u = rng.normal(size=(n, 3))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    target = c + rng.uniform(-spread, spread, (n, 3)) * r[:, None] / np.sqrt(3)
    o = target + u * dist
    return _rays(o, target - o, rng.random(n))


def face_and_tangent_rays(spheres, n, seed):
    """Origins exactly on the planes c_k +- r (the unpadded faces of the spheres' boxes), directions through the box, and
    tangent rays (line at distance r from the centre, computed in float64 and rounded)."""
    rng = np.random.default_rng(seed)
    idx = rng.integers(0, len(spheres), n)
    c = np.array([spheres[k][0] for k in idx], F32)
    r = np.abs(np.array([spheres[k][1] for k in idx], F32))
    axis = rng.integers(0, 3, n)
    side = rng.choice([-1.0, 1.0], n).astype(F32)
    o = c + rng.uniform(-0.5, 0.5, (n, 3)).astype(F32) * r[:, None]
    o[np.arange(n), axis] = c[np.arange(n), axis] + side * r
    d = rng.normal(size=(n, 3)).astype(F32)
    d[np.arange(n), axis] = -side * np.abs(d[np.arange(n), axis])
    face = _rays(o, d)
    # tangents: a unit vector w perpendicular to the direction, origin = c + r w - 3 r dir
    dd = rng.normal(size=(n, 3))
    dd /= np.linalg.norm(dd, axis=1, keepdims=True)
    w = np.cross(dd, rng.normal(size=(n, 3)))
    w /= np.linalg.norm(w, axis=1, keepdims=True)
    to = c + r[:, None] * w - 3 * r[:, None] * dd
    return face, _rays(to, dd)


# -------------------------------------------------------------------------------------------------- float64 restatement

def _centres(sph, time):
    """float64 centres of every sphere at each ray's time: (rays, spheres, 3)."""
    c0 = np.array([s[0] for s in sph], np.float64)
    c1 = np.array([s[2] if s[2] is not None else s[0] for s in sph], np.float64)
    return c0[None] + time[:, None, None] * (c1 - c0)[None]


def check_geometry(sph, rays, hits, tmin, chunk=256):
    """Every reported hit lies on its sphere and is the nearest one in float64 within the float32 quadratic's error bound:
    a sphere the float64 ray clearly meets (squared miss distance below r^2 (1 - 1e-4)) at a root in [tmin, t) farther
    than that bound from t is a missed closer hit; a ray reported as a miss must clearly meet none.  The bound: b, oc and
    the centre carry a few float32 roundings (2^-20 relative), the discriminant b^2 - a c an absolute error E of 2^-20 of its
    terms, which moves sqrt(disc) by E / sqrt(disc) (by sqrt(E) at a tangent)."""
    # the float32 values the scene holds; coincident spheres have the same geometry: test each distinct (centre0, |r|, centre1) once
    sph = [(np.asarray(c0, F32).astype(np.float64), float(F32(r)), None if c1 is None else np.asarray(c1, F32).astype(np.float64))
           for c0, r, c1 in sph]
    key = np.array([list(s[0]) + [abs(s[1])] + list(s[2] if s[2] is not None else s[0]) + [s[2] is not None] for s in sph], np.float64)
    key, first_of, which = np.unique(key, axis=0, return_index=True, return_inverse=True)
    sph = [sph[k] for k in first_of]
    r = np.abs(np.array([s[1] for s in sph], np.float64))
    moving = np.array([s[2] is not None for s in sph])
    o = rays["origin"].astype(np.float64)
    d = rays["direction"].astype(np.float64)
    t_got = hits["t"].astype(np.float64)
    hit = hits["id"] != capi.RT_INVALID_ID
    ids = np.where(hit, which.reshape(-1)[np.where(hit, hits["id"], 0).astype(np.int64)], -1)
    u = 2.0 ** -20
    for b in range(0, len(rays), chunk):
        sl = slice(b, b + chunk)
        c = _centres(sph, rays["time"][sl].astype(np.float64)) if moving.any() else np.array([s[0] for s in sph], np.float64)[None]
        oc = o[sl, None, :] - c
        a = np.einsum("ij,ij->i", d[sl], d[sl])[:, None]
        bb = np.einsum("ijk,ik->ij", oc, d[sl])
        oc2 = np.einsum("ijk,ijk->ij", oc, oc)
        cc = oc2 - r[None] ** 2
        disc = bb * bb - a * cc
        h2 = oc2 - bb * bb / a  # squared distance from the centre to the line
        clear = h2 < r[None] ** 2 * (1 - 1e-4)
        sq = np.sqrt(np.maximum(disc, 0))
        near, far = (-bb - sq) / a, (-bb + sq) / a
        err = u * (bb * bb + a * oc2 + a * r[None] ** 2)
        sq_err = np.where(disc > err, err / np.sqrt(np.maximum(disc, err)), np.sqrt(err))
        pos = np.sqrt(np.einsum("ijk,ijk->ij", c, c) + np.einsum("ij,ij->i", o[sl], o[sl])[:, None])  # coordinate magnitude
        tol = (u * np.sqrt(a) * (np.sqrt(oc2) + r[None] + pos) + sq_err) / a + 1e-7
        first = np.where(near >= tmin, near, np.where(far >= tmin, far, np.inf))
        first = np.where(disc >= 0, first, np.inf)
        # the reported sphere: its float64 root equals t within the error
        hb = hit[sl]
        rows = np.nonzero(hb)[0]
        mine = ids[sl][hb]
        root_err = np.minimum(np.abs(near[rows, mine] - t_got[sl][hb]), np.abs(far[rows, mine] - t_got[sl][hb]))
        assert (disc[rows, mine] >= -err[rows, mine]).all(), "a reported hit on a sphere the ray misses"
        assert (root_err <= tol[rows, mine]).all(), float((root_err - tol[rows, mine]).max())
        # nothing clearly closer
        limit = np.where(hb, t_got[sl], np.inf)[:, None] - tol
        closer = clear & (first < limit) & (first < np.inf) & (first >= tmin + tol)
        assert not closer.any(), (b + np.nonzero(closer.any(axis=1))[0][:5], np.nonzero(closer)[1][:5])


# -------------------------------------------------------------------------------------------------------------- the walk

def _build(ctx, sph, bvh, expect):
    """Scene from the JSON front-end; `expect` is True (accepted) or False (RT_ERR_UNSUPPORTED with a message)."""
    d = rt.SceneDesc.from_json(_doc(sph, bvh))
    if expect:
        return rt.Scene(ctx, d)
    with pytest.raises(capi.RtError) as e:
        rt.Scene(ctx, d)
    assert e.value.status == capi.RT_ERR_UNSUPPORTED and "depth" in str(e.value), str(e.value)
    return None


def _walks_equal_list(ctx, sph, ray_sets, builders, quant, oracle=None, tmins=(1e-5,), geometry=True):
    """builders: {"sah": accepted?, "lbvh": accepted?}; quant: whether the quantised nodes exist (use_bvh = 3).
    Returns the accepted scenes."""
    lst = _build(ctx, sph, "none", True)
    scenes = {}
    for name, ok in builders.items():
        sc = _build(ctx, sph, name, ok)
        if sc is None:
            continue
        assert sc.info().bvh_depth <= MAX_DEPTH
        scenes[name] = sc
        if not quant:
            with pytest.raises(capi.RtError) as e:
                sc.trace_primary(ray_sets[0][1][:4], use_bvh=3)
            assert e.value.status == capi.RT_ERR_INVALID_ARG and "quantised" in str(e.value)
    assert scenes, "no builder accepted the scene"
    for label, rays, check in ray_sets:
        for tmin in tmins:
            want = lst.trace_primary(rays, tmin=tmin, use_bvh=0)
            if oracle is not None:
                orc = oracle.scene(rt.SceneDesc.from_json(_doc(sph, "none"))).trace(rays, tmin=tmin, arith=1)
                for f in ("id", "t", "p", "n"):  # (u, v: the oracle's libm atan2/asin against the device's, not compared here)
                    assert np.array_equal(orc[f], want[f]), (label, tmin, f, int((orc["id"] != want["id"]).sum()))
            if geometry and check:
                check_geometry(sph, rays, want, tmin)
            bad = {}  # rays whose (id, t, p, n, u, v) differ from the list's, per builder and walk
            for name, sc in scenes.items():
                for use_bvh in (1, 2, 3) if quant else (1, 2):
                    got = sc.trace_primary(rays, tmin=tmin, use_bvh=use_bvh)
                    bad[f"{name}/{use_bvh}"] = int((got.view(np.uint8).reshape(len(got), -1) != want.view(np.uint8).reshape(len(want), -1)).any(axis=1).sum())
            assert not any(bad.values()), f"rays {label}, tmin {tmin}: mismatches {bad}"
    return scenes


# ------------------------------------------------------------------------------------------------------------------ cases

@pytest.mark.parametrize("k,extra,depth,lbvh_ok", [
    (50, 0, 50, True),   # worst 4-wide stack 75: more than 64 entries
    (63, 2, 64, True),   # the deepest tree accepted: the binary walk needs exactly 64 entries, the 4-wide walks 96
    (63, 3, 65, False),  # one level too deep
])
def test_deep_caterpillar(ctx, oracle, k, extra, depth, lbvh_ok):
    sph = caterpillar(k, extra)
    if lbvh_ok:  # the precondition: the tree is as deep as designed
        sc = _build(ctx, sph, "lbvh", True)
        assert sc.info().bvh_mode == capi.RT_BVH_GPU_LBVH and sc.info().bvh_depth == depth
    # balanced directions from near the origin: the closest hit is the far side of one of the deepest spheres
    rays = [("deep", inside_rays(20_000, 0.0, 0.1, seed=k, dmin=0.4), True), ("inside", inside_rays(10_000, 0.0, 0.3, seed=k + 1), True),
            ("axis", axis_rays(4000, 0.0, 0.3, seed=k + 2), True)]
    scenes = _walks_equal_list(ctx, sph, rays, {"sah": True, "lbvh": lbvh_ok}, quant=True, oracle=oracle, tmins=(1e-5, 1e-3, 0.0))
    assert scenes["sah"].info().bvh_depth <= 20  # the SAH tree of the same spheres is shallow


@pytest.mark.parametrize("n_big", [31, 32, 33])
def test_outsized_sphere_chain_over_a_deep_lbvh(ctx, n_big):
    sph = chain_scene(n_big)
    sc = _build(ctx, sph, "lbvh", True)
    assert sc.info().bvh_depth == (61 if n_big == 31 else 62)  # 31 or 32 chain nodes + the LBVH's 30 levels
    rays = [("deep", inside_rays(10_000, 0.0, 0.1, seed=n_big, dmin=0.4), True), ("axis", axis_rays(2000, 0.0, 0.2, seed=n_big), True)]
    _walks_equal_list(ctx, sph, rays, {"sah": True, "lbvh": True}, quant=True)


def test_exact_ties_resolve_to_the_lowest_ordinal(ctx):
    sph = tie_scene()
    assert len(sph) >= 4096  # the persistent-lane kernel's scene size
    shell = inside_rays(10_000, -0.5, 0.5, seed=3, dmin=-1.0)  # from inside the 5000 coincident spheres
    outside = towards_rays(20_000, sph, 8.0, seed=4)
    face, tangent = face_and_tangent_rays(sph[5000:], 4000, seed=5)
    rays = [("shell", shell, True), ("outside", outside, True), ("face", face, True), ("tangent", tangent, False),
            ("axis", axis_rays(4000, -4.0, 4.0, seed=6), True)]
    scenes = _walks_equal_list(ctx, sph, rays, {"sah": True, "lbvh": True}, quant=True, tmins=(1e-5, 1e-3, 0.0))
    # the coincident shell: whichever walk, the winner is ordinal 0; each group of duplicates: its first member
    got = scenes["lbvh"].trace_primary(np.concatenate([shell, outside]), use_bvh=3)
    ids = got["id"][got["id"] != capi.RT_INVALID_ID].astype(np.int64)
    assert (ids[ids < 5000] == 0).all() and (ids < 5000).any()
    grp = ids[(ids >= 5000) & (ids < 5240)]
    assert len(grp) and ((grp - 5000) % 8 == 0).all()


@pytest.mark.parametrize("kind", ["line", "plane"])
def test_flat_and_collinear_scenes(ctx, kind):
    sph = line_scene() if kind == "line" else plane_scene()
    face, tangent = face_and_tangent_rays(sph, 4000, seed=9)
    rng = np.random.default_rng(8)
    if kind == "line":  # along the line itself (both zero components exact) and from beside it
        along = _rays(np.c_[rng.uniform(-2, 160, 4000), np.zeros(4000), np.zeros(4000)], np.tile([1.0, 0.0, -0.0], (4000, 1)))
        lo, hi = (-1.0, -0.3, -0.3), (151.0, 0.3, 0.3)
    else:  # straight down onto the plane, and from just above it
        along = _rays(np.c_[rng.uniform(-1, 64, 4000), np.full(4000, 3.0), rng.uniform(-1, 64, 4000)], np.tile([-0.0, -1.0, 0.0], (4000, 1)))
        lo, hi = (-1.0, 0.2, -1.0), (64.0, 0.6, 64.0)
    o = rng.uniform(lo, hi, (10_000, 3))
    beside = _rays(o, rng.normal(size=(10_000, 3)))
    rays = [("towards", towards_rays(10_000, sph, 6.0, seed=10), True), ("along", along, True), ("beside", beside, True),
            ("face", face, True), ("tangent", tangent, False), ("axis", axis_rays(4000, -1.0, 64.0, seed=12), True)]
    _walks_equal_list(ctx, sph, rays, {"sah": True, "lbvh": True}, quant=True)


@pytest.mark.parametrize("offset", [1e5, 1e6])
def test_cluster_far_from_the_origin(ctx, offset):
    sph = cluster_scene((offset, -offset, offset))
    rays = [("towards", towards_rays(20_000, sph, 40.0, seed=13), True),
            ("axis", axis_rays(4000, np.array([offset - 50, -offset - 50, offset - 50]), np.array([offset + 50, -offset + 50, offset + 50]), seed=14), True)]
    _walks_equal_list(ctx, sph, rays, {"sah": True, "lbvh": True}, quant=True)


def test_quantisation_unit_overflow_on_axis_aligned_rays(ctx):
    """Extent 3.3e6: the root's quantisation unit is 2^14, so for a ray with a zero direction component S = 2^(e + 15) *
    2^100 overflows to inf in trav_inner_q and the bound of that axis is NaN.  fmax/fmin drop a NaN operand, so the axis
    is ignored: more visits, never fewer."""
    sph = grid_scene(3.0e5, 12, 1.1e5)
    g = 3.0e5 * 5.5
    rays = [("axis", axis_rays(20_000, -g, g, seed=15), True), ("towards", towards_rays(10_000, sph, 4.0e5, seed=16), True)]
    _walks_equal_list(ctx, sph, rays, {"sah": True, "lbvh": True}, quant=True)


def test_extent_beyond_the_quantised_range(ctx):
    """Extent 4e8: a unit past 2^20 is needed, k_quantize4 refuses, use_bvh = 3 is refused and the 128-byte 4-wide nodes
    (what k_wf_step_pt then walks) must still be exact."""
    sph = grid_scene(1.0e8, 5, 3.5e7)
    g = 2.5e8
    rays = [("axis", axis_rays(10_000, -g, g, seed=17), True), ("towards", towards_rays(10_000, sph, 1.5e8, seed=18), True)]
    _walks_equal_list(ctx, sph, rays, {"sah": True, "lbvh": True}, quant=False)


# ---------------------------------------------------------------------------------------------------------------- render

@pytest.mark.parametrize("name", ["caterpillar", "ties"])
def test_render_kernels_agree_on_adversarial_trees(ctx, monkeypatch, name):
    """k_wf_step_pt (quantised 4-wide walk), k_wf_step_warp (speculative binary walk) and k_wf_step_cta on the tree, and the
    megakernel on a brute-force copy of the scene, trace the same paths: equal ray and sample counts, sums equal up to the
    order of float additions.  Materials m1 and m3 emit, so the colour of a pixel depends on which sphere its camera ray hits
    first (with lambertian surfaces alone, paths that start inside these nested spheres never reach the sky)."""
    if name == "caterpillar":
        sph, bvh = caterpillar(50), "lbvh"
        cam = {"lookfrom": [0.1, 0.12, 0.08], "lookat": [1, 1, 1], "vfov": 70, "aspect": 1.5}
    else:
        sph, bvh = tie_scene(), "lbvh"
        cam = {"lookfrom": [0.3, 0.2, 0.4], "lookat": [3, 1, -2], "vfov": 90, "aspect": 1.5}
    w, h, spp = 96, 64, 4
    ref_sc = rt.Scene(ctx, rt.SceneDesc.from_json(_doc(sph, "none", cam, emitters=True)))
    want, st0 = ref_sc.render_accum(rt.default_params(width=w, height=h, spp=spp, max_depth=4, pipeline=capi.RT_PIPE_MEGAKERNEL))
    sc = rt.Scene(ctx, rt.SceneDesc.from_json(_doc(sph, bvh, cam, emitters=True)))
    assert np.array_equal(want[..., 3], np.full((h, w), spp, F32)) and (want[..., :3] > 0).mean() > 0.5  # light reaches the camera
    for grain in ("pt", "warp", "cta"):
        monkeypatch.setenv("RT_WF_GRAIN", grain)
        got, st = sc.render_accum(rt.default_params(width=w, height=h, spp=spp, max_depth=4, pipeline=capi.RT_PIPE_WAVEFRONT))
        assert np.array_equal(got[..., 3], want[..., 3]), grain
        diff = np.abs(got[..., :3] - want[..., :3]).max(axis=2)
        assert st.rays == st0.rays and np.allclose(got, want, rtol=1e-5, atol=1e-5), (grain, int(st.rays), int(st0.rays),
                                                                                      int((diff > 1e-5).sum()))
