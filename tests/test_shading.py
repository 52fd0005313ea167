"""The shading step in float64: textures (Perlin lattice, turbulence, marble, wood, checker resolution, image look-up),
optics (reflect, refract, Schlick), sphere (u, v), Philox4x32-10 and the direct samplers, restated with numpy from the
reference's formulas.  Each restatement returns its value together with a forward error bound: the most any float32
evaluation of the same expression, with every operation rounded once or with a multiply fused into the following add, can
be away from it.  The oracle (oracle/liboracle.so, no contraction) and the CUDA kernels (nvcc contracts) are both such
evaluations, so each must lie within that bound of the float64 value, and within twice the bound of each other.

The SFU intrinsics of the kernels (__sinf, __sincosf, __powf) add their own error.  Inside [-pi, pi] __sinf is documented
to 2^-21.41 absolute; outside, its argument is first scaled by a rounded 1/(2 pi), so the bound used here, SFU_SIN, grows
by 2^-22 per unit of |x|.  That growth and the __powf bound are assumed, not derived; tests/test_gpu_shading.py records what
the device measures against them.

This file checks the restatements against the oracle's unit hooks on the CPU; tests/test_gpu_shading.py uses them to
judge the device ray by ray, and to tell a genuine fault from a near-tie (a checker sign, a wood floor, a texel edge, a
reflect/refract draw) that one ulp may decide either way."""
from __future__ import annotations

import ctypes as C

import numpy as np
import pytest

from raytracing_renderer_cuda_b200 import capi

U = 2.0 ** -24   # float32 round-to-nearest unit roundoff
UZ = 2.0 ** -23  # round toward zero: the reference's vec3 operators (vec3.h), both sides
MASK = np.uint64(0xFFFFFFFF)

# Ken Perlin's 2002 permutation (perlin_noise.h:24-37)
PERM = np.array([int(x) for x in """151 160 137 91 90 15 131 13 201 95 96 53 194 233 7 225 140 36 103 30 69 142 8 99 37 240 21 10 23
190 6 148 247 120 234 75 0 26 197 62 94 252 219 203 117 35 11 32 57 177 33 88 237 149 56 87 174 20 125 136 171 168 68 175 74
165 71 134 139 48 27 166 77 146 158 231 83 111 229 122 60 211 133 230 220 105 92 41 55 46 245 40 244 102 143 54 65 25 63 161 1
216 80 73 209 76 132 187 208 89 18 169 200 196 135 130 116 188 159 86 164 100 109 198 173 186 3 64 52 217 226 250 124 123 5 202
38 147 118 126 255 82 85 212 207 206 59 227 47 16 58 17 182 189 28 42 223 183 170 213 119 248 152 2 44 154 163 70 221 153 101
155 167 43 172 9 129 22 39 253 19 98 108 110 79 113 224 232 178 185 112 104 218 246 97 228 251 34 242 193 238 210 144 12 191
179 162 241 81 51 145 235 249 14 239 107 49 192 214 31 181 199 106 157 184 84 204 176 115 121 50 45 127 4 150 254 138 236 205
93 222 114 67 29 24 72 243 141 128 195 78 66 215 61 156 180""".split()], np.int64)
assert len(PERM) == 256 and sorted(PERM) == list(range(256))


def sfu_sin(x):
    """Assumed absolute error of __sinf / __sincosf at argument x (see the module docstring)."""
    return 2.0 ** -21.41 + 2.0 ** -22 * np.abs(x)


POWF_REL = 2.0 ** -19  # assumed relative error of __powf(x, 5) = exp2(5 log2 x) on (0, 1]


class E:
    """A float64 value and a bound on how far a float32 evaluation of the same expression can be from it."""

    def __init__(self, v, e=0.0):
        self.v = np.asarray(v, np.float64)
        self.e = np.broadcast_to(np.asarray(e, np.float64), self.v.shape) if np.ndim(e) else np.full(self.v.shape, float(e))

    def _r(self, v, e, unit):
        return E(v, e + unit * (np.abs(v) + e))

    def add(self, o, unit=U):
        o = o if isinstance(o, E) else E(o)
        return self._r(self.v + o.v, self.e + o.e, unit)

    def sub(self, o, unit=U):
        o = o if isinstance(o, E) else E(o)
        return self._r(self.v - o.v, self.e + o.e, unit)

    def mul(self, o, unit=U):
        o = o if isinstance(o, E) else E(o)
        return self._r(self.v * o.v, np.abs(self.v) * o.e + np.abs(o.v) * self.e + self.e * o.e, unit)

    def div(self, o, unit=U):
        o = o if isinstance(o, E) else E(o)
        q = self.v / o.v
        return self._r(q, (self.e + np.abs(q) * o.e) / np.maximum(np.abs(o.v) - o.e, 1e-300), unit)


# ------------------------------------------------------------------ Perlin (perlin_noise.h:46-153) ----
def _ease(t):  # t * t * t * (t * (t * 6 - 15) + 10)
    t = E(t)
    return t.mul(t).mul(t).mul(t.mul(t.mul(6.0).sub(15.0)).add(10.0))


def _grad(h, x, y, z):  # exact float32 inputs; one rounding
    h = h & 15
    u = np.where(h < 8, x, y)
    v = np.where(h < 4, y, np.where((h == 12) | (h == 14), x, z))
    return E(np.where(h & 1, -u, u)).add(np.where(h & 2, -v, v))


def _lerp(t, a, b):  # a + t * (b - a)
    return a.add(t.mul(b.sub(a)))


def perlin(p):
    """perlin_noise::noise of float32 points p (N, 3) -> E.  floor, the & 255 wrap and xf = p - floor(p), xf - 1 are the
    float32 operations both implementations do (one rounding each, no multiply to fuse), so they are done in float32."""
    p = np.asarray(p, np.float32).reshape(-1, 3)
    fl = np.floor(p)
    idx = fl.astype(np.int64) & 255
    f = (p - fl).astype(np.float32)
    f1 = (f - np.float32(1)).astype(np.float32)
    xi, yi, zi = idx.T
    x, y, z = (f[:, k].astype(np.float64) for k in range(3))
    x1, y1, z1 = (f1[:, k].astype(np.float64) for k in range(3))
    u, v, w = _ease(x), _ease(y), _ease(z)
    P = lambda i: PERM[i & 255]
    A, B = P(xi) + yi, P(xi + 1) + yi
    AA, AB, BA, BB = P(A) + zi, P(A + 1) + zi, P(B) + zi, P(B + 1) + zi
    res = _lerp(w, _lerp(v, _lerp(u, _grad(P(AA), x, y, z), _grad(P(BA), x1, y, z)),
                         _lerp(u, _grad(P(AB), x, y1, z), _grad(P(BB), x1, y1, z))),
                _lerp(v, _lerp(u, _grad(P(AA + 1), x, y, z1), _grad(P(BA + 1), x1, y, z1)),
                      _lerp(u, _grad(P(AB + 1), x, y1, z1), _grad(P(BB + 1), x1, y1, z1))))
    r = res.add(1.0)
    return E(r.v / 2, r.e / 2)


def turbulence(p):
    """6 octaves, lacunarity 2, gain 0.5 (perlin_noise.h:142-153); p * 2^k and * 0.5^k are exact."""
    p = np.asarray(p, np.float32).reshape(-1, 3)
    s = E(np.zeros(len(p)))
    for k in range(6):
        r = perlin((p * np.float32(2.0 ** k)).astype(np.float32))
        a = E(r.v * 2, r.e * 2).sub(1.0)
        s = s.add(E(np.abs(a.v) * 0.5 ** k, a.e * 0.5 ** k))
    return s


def rz32(x):
    """float64 -> float32 rounded toward zero (the product of two float32 is exact in float64)."""
    x = np.asarray(x, np.float64)
    r = x.astype(np.float32)
    over = np.abs(r.astype(np.float64)) > np.abs(x)
    return np.where(over, np.nextafter(r, np.float32(0)), r).astype(np.float32)


def rz_div32(a, b):
    """float32 / float32 rounded toward zero: the float64 quotient, corrected by its exact residual."""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    q = (a.astype(np.float64) / b.astype(np.float64)).astype(np.float32)
    big = np.abs(q.astype(np.float64) * b.astype(np.float64)) > np.abs(a.astype(np.float64))  # rounded away from zero
    return np.where(big, np.nextafter(q, np.float32(0)), q).astype(np.float32)


# ------------------------------------------------------------------ textures (texture.h) ----
MARBLE_C1 = np.array([0.925, 0.816, 0.78], np.float32).astype(np.float64)
MARBLE_C2 = np.array([0.349 / 2, 0.431 / 2, 0.498 / 2], np.float32).astype(np.float64)


def checker_sines(p, sfu=True):
    """sin(10 x) sin(10 y) sin(10 z) in float64 of the float32 arguments both sides form, and the bound within which a
    float32 product of __sinf (sfu) or libm sinf values may have the other sign (a near-tie)."""
    a = (np.float32(10) * np.asarray(p, np.float32)).astype(np.float32).astype(np.float64)
    s = np.sin(a)
    return s.prod(axis=1), (sfu_sin(a) if sfu else np.full(a.shape, 2 * U)).sum(axis=1) + 2.0 ** -22


def resolve(textures, ix, p, sfu=True):
    """Leaf texture index of texture ix at every point, following checker_texture::value (texture.h:41-48): every level
    sees the same sines, so a chain takes the even or the odd child all the way.  Also returns the near-tie mask."""
    prod, tie_b = checker_sines(p, sfu)
    odd = prod < 0
    leaf = np.full(len(p), ix, np.int64)
    tie = np.zeros(len(p), bool)
    for _ in range(len(textures) + 1):
        chk = np.array([textures[int(k)].kind == capi.RT_TEX_CHECKER for k in leaf])
        if not chk.any():
            break
        tie |= chk & (np.abs(prod) <= tie_b)
        nxt = np.array([textures[int(k)].odd if o else textures[int(k)].even for k, o in zip(leaf, odd)])
        leaf = np.where(chk, nxt, leaf)
    return leaf, tie


def sphere_uv(n):
    """get_sphere_uv (sphere.h:61-83) in float64 of float32 normals, and the float32 u, v both sides then hold."""
    n = np.asarray(n, np.float32).astype(np.float64)
    with np.errstate(invalid="ignore"):
        phi, theta = np.arctan2(n[:, 2], n[:, 0]), np.arcsin(n[:, 1])
    return 1 - (phi + np.pi) / (2 * np.pi), (theta + np.pi / 2) / np.pi


UV_ERR = 2.0 ** -22  # |u|, |v| error of atan2f / asinf (<= 3 ulp of pi) through the affine maps, plus u, v's float rounding


def image_texel(u, v, w, h):
    """image_texture::value's texel (texture.h:118-132) of float64 (u, v), and whether u*W or (1-v)*H - 0.001 lies within
    the (u, v) error of an integer (a texel edge either side may take).  A NaN v (asinf of |n.y| a hair above 1) converts
    to row 0 on both sides."""
    x, y = u * w, (1 - v) * h - 0.001
    with np.errstate(invalid="ignore"):
        i = np.clip(np.nan_to_num(np.floor(x), nan=0), 0, w - 1).astype(np.int64)
        j = np.clip(np.nan_to_num(np.floor(y), nan=0), 0, h - 1).astype(np.int64)
        tie = (np.abs(x - np.round(x)) <= (UV_ERR + U) * w + 1e-9) | (np.abs(y - np.round(y)) <= (UV_ERR + U) * h + 1e-9)
    return i, j, tie & ~np.isnan(y)


def leaf_value(t, p, n, images=None, sfu=True):
    """A non-checker texture's value (N, 3) at float32 points p / normals n -> (value, error bound, near-tie mask).
    sfu=True adds the device's __sinf error (marble), else a libm sinf's."""
    p = np.asarray(p, np.float32).reshape(-1, 3)
    N = len(p)
    tie = np.zeros(N, bool)
    if t.kind == capi.RT_TEX_CONSTANT:
        return np.tile(np.array(t.color1[:], np.float32).astype(np.float64), (N, 1)), np.zeros(N), tie
    if t.kind == capi.RT_TEX_NOISE_PERLIN:  # perlin(p * density), the product rounded toward zero on both sides
        r = perlin(rz32(p.astype(np.float64) * np.float64(np.float32(t.density))))
        return np.repeat(r.v[:, None], 3, 1), r.e, tie
    if t.kind == capi.RT_TEX_NOISE_TURBULANCE:  # 0.5 * turb(p * density): the half is exact
        r = turbulence(rz32(p.astype(np.float64) * np.float64(np.float32(t.density))))
        return np.repeat(r.v[:, None] / 2, 3, 1), r.e / 2, tie
    if t.kind == capi.RT_TEX_NOISE_MARBLE:  # 0.5 (1 + sin(p.z density + 7 turb(p))), color1 value + color2 (1 - value)
        arg = E(p[:, 2]).mul(float(np.float32(t.density))).add(turbulence(p).mul(7.0))
        s_err = arg.e + (sfu_sin(arg.v) if sfu else 2 * U)
        val = 0.5 * (1 + np.sin(arg.v))
        ve = 0.5 * s_err + 2 * U
        out = MARBLE_C1 * val[:, None] + MARBLE_C2 * (1 - val[:, None])
        err = ve * np.abs(MARBLE_C1 - MARBLE_C2).max() + 4 * UZ
        return out, err, tie
    if t.kind == capi.RT_TEX_WOOD:  # nn = hardness * perlin(p / density); nn -= floor(nn); c1 nn + c2 (1 - nn)
        r = perlin(rz_div32(p, np.float32(t.density)))
        nn = E(r.v).mul(float(np.float32(t.hardness)))
        nn.e = nn.e + abs(float(np.float32(t.hardness))) * r.e
        fr = nn.v - np.floor(nn.v)
        tie = np.abs(nn.v - np.round(nn.v)) <= nn.e + U * np.abs(nn.v)
        c1, c2 = (np.array(c[:], np.float32).astype(np.float64) for c in (t.color1, t.color2))
        out = c1 * fr[:, None] + c2 * (1 - fr[:, None])
        err = (nn.e + U * (np.abs(nn.v) + 1)) * (np.abs(c1) + np.abs(c2)).max() + 4 * UZ * (np.abs(c1) + np.abs(c2)).max()
        return out, err, tie
    if t.kind == capi.RT_TEX_IMAGE:
        img = images[t.image]
        u, v = sphere_uv(n)
        i, j, tie = image_texel(u, v, img.shape[1], img.shape[0])
        return img[j, i].astype(np.float64), np.zeros(N), tie
    return np.ones((N, 3)), np.zeros(N), tie


def texture_value(textures, ix, p, n, images=None, sfu=True):
    """texture ix at float32 points p (N, 3) / normals n -> (value (N, 3), error bound (N,), near-tie mask (N,))."""
    p = np.asarray(p, np.float32).reshape(-1, 3)
    n = np.asarray(n, np.float32).reshape(-1, 3)
    leaf, tie = resolve(textures, ix, p, sfu)
    val, err = np.zeros((len(p), 3)), np.zeros(len(p))
    for k in np.unique(leaf):
        sel = leaf == k
        v, e, t = leaf_value(textures[int(k)], p[sel], n[sel], images, sfu)
        val[sel], err[sel] = v, e
        tie[sel] |= t
    return val, err, tie


# ------------------------------------------------------------------ random numbers (csrc/rt_device.cuh) ----
def philox4x32_10(c0, c1, c2, c3, k0, k1):
    c = [np.asarray(x, np.uint64) & MASK for x in (c0, c1, c2, c3)]
    k0, k1 = np.uint64(k0) & MASK, np.uint64(k1) & MASK
    c = list(np.broadcast_arrays(*c))
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c[0], np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & MASK, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & MASK]
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & MASK, (k1 + np.uint64(0xBB67AE85)) & MASK
    return [x.astype(np.uint32) for x in c]


def rng_block(seed, pixel, sample, bounce, blk):
    return philox4x32_10(pixel, sample, (bounce << 8) | blk, 0x52544232, seed, 0x42323030)


def u01(x):
    """fmaf(float(x), 2^-32, 2^-33): (0, 1]; the fused sum is exact in float64."""
    f = np.asarray(x, np.uint32).astype(np.float64).astype(np.float32).astype(np.float64)
    return (f * 2.0 ** -32 + 2.0 ** -33).astype(np.float32)


def probe_draws(n, seed):
    """The four uniforms of block 0 of rt_shade_probe / orc_shade_probe's step for rays 0..n-1 (pixel = ray index,
    sample 0, bounce 1)."""
    return [u01(x) for x in rng_block(seed, np.arange(n, dtype=np.uint64), 0, 1, 0)]


def unit_ball(u1, u2, u3):
    """sample_unit_ball in float64 and its bound: z = 1 - 2 u1, radius cbrt(u3), angle 2 pi u2 (a float32 product on both
    sides).  The bound holds __sincosf's error at that angle."""
    z = np.float32(1) - np.float32(2) * u1.astype(np.float64)
    z = z.astype(np.float32).astype(np.float64)
    rxy = np.sqrt(np.maximum(0, 1 - z * z))
    ang = (np.float32(6.283185307179586) * u2).astype(np.float32).astype(np.float64)
    rad = np.minimum(np.cbrt(u3.astype(np.float64)), float(np.float32(0.99999994)))
    b = np.stack([rad * rxy * np.cos(ang), rad * rxy * np.sin(ang), rad * z], 1)
    return b, sfu_sin(ang) + 8 * U


def schlick(cosine, ri):
    """utils::shlick in float64 of the float32 cosine."""
    r0 = ((1 - ri) / (1 + ri)) ** 2
    return r0 + (1 - r0) * (1 - cosine) ** 5


def schlick_err(cosine, ri):
    """How far the device's Schlick can be from float64: __powf's relative error plus the roundings of r0 and the sum."""
    r0 = ((1 - ri) / (1 + ri)) ** 2
    return (1 - r0) * (1 - cosine) ** 5 * POWF_REL + 8 * UZ


# ------------------------------------------------------------------ scenes ----
def make_desc(spheres, materials, textures, images=(), camera=None):
    """A raw rt_scene_desc (the C ABI: nothing is clamped, as the façade clamps metal roughness) held by capi.SceneDesc.
    spheres: (centre, radius, material[, centre1]) — a centre1 makes a moving sphere over [0, 1]; ids are list positions."""
    S = capi.rt_sphere * max(len(spheres), 1)
    sph = S(*[capi.rt_sphere(s[0], s[1], s[3] if len(s) > 3 else s[0], 0, 1, s[2], k, capi.RT_SPHERE_MOVING if len(s) > 3 else 0)
              for k, s in enumerate(spheres)])
    mats = (capi.rt_material * max(len(materials), 1))(*materials)
    texs = (capi.rt_texture * max(len(textures), 1))(*textures)
    imgs = [np.ascontiguousarray(im, np.float32) for im in images]
    ims = (capi.rt_image * max(len(imgs), 1))(*[capi.rt_image(im.ctypes.data_as(C.POINTER(C.c_float)), im.shape[1], im.shape[0])
                                                for im in imgs])
    d = capi.rt_scene_desc()
    d.spheres, d.n_spheres, d.materials, d.n_materials = sph, len(spheres), mats, len(materials)
    d.textures, d.n_textures, d.images, d.n_images = texs, len(textures), ims, len(imgs)
    d.camera = camera or capi.rt_camera((0, 0, 5), (0, 0, 0), (0, 1, 0), 40, 1.5, 0, 5, 0, 1)
    d.bvh_mode = capi.RT_BVH_NONE
    return capi.SceneDesc(C.pointer(d), None, keepalive=(sph, mats, texs, imgs, ims, d))


def tex_constant(c):
    return capi.rt_texture(capi.RT_TEX_CONSTANT, -1, -1, -1, tuple(c), (0, 0, 0), 0, 0)


def tex_checker(even, odd):
    return capi.rt_texture(capi.RT_TEX_CHECKER, even, odd, -1, (0, 0, 0), (0, 0, 0), 0, 0)


def tex_noise(kind, density):
    return capi.rt_texture(kind, -1, -1, -1, (0, 0, 0), (0, 0, 0), density, 0)


def tex_wood(c1, c2, density, hardness):
    return capi.rt_texture(capi.RT_TEX_WOOD, -1, -1, -1, tuple(c1), tuple(c2), density, hardness)


def tex_image(i):
    return capi.rt_texture(capi.RT_TEX_IMAGE, -1, -1, i, (0, 0, 0), (0, 0, 0), 0, 0)


def checker_chain(levels, leaf_even, leaf_odd, first=0):
    """Textures first.. of a chain of `levels` checkers: level 1 picks leaf_even / leaf_odd, level k picks level k-1 for
    both children.  Returns the list; the top of the chain is its last entry."""
    out = [tex_checker(leaf_even, leaf_odd)]
    for k in range(1, levels):
        out.append(tex_checker(first + k - 1, first + k - 1))
    return out


def lattice_points():
    """Lattice points the Perlin code goes wrong on: negative coordinates, beyond +-256 cells (the & 255 wrap), exact
    integers and half-integers, values a hair below an integer, and large magnitudes."""
    r = np.random.default_rng(3)
    pts = [r.uniform(-3, 3, (400, 3)), r.uniform(-700, 700, (400, 3)), r.integers(-600, 600, (100, 3)).astype(np.float64),
           r.integers(-600, 600, (100, 3)) + 0.5, r.integers(-300, 300, (100, 3)) - 2.0 ** -20, r.uniform(-1, 1, (100, 3)) * 2.0 ** -30,
           np.array([[-256, 256, -512], [255.99998, -0.0, 0.0], [-1e4, 2e4, -3e4]])]
    return np.concatenate(pts).astype(np.float32)


# ------------------------------------------------------------------ tests ----
def test_perlin_and_turbulence_match_the_oracle(oracle):
    pts = lattice_points()
    for fn, hook in ((perlin, oracle.perlin_noise), (turbulence, oracle.turbulence)):
        r = fn(pts)
        got = np.array([hook(q) for q in pts], np.float64)
        assert (np.abs(got - r.v) <= r.e).all(), (fn.__name__, float((np.abs(got - r.v) - r.e).max()))
        # an a-priori bound: it peaks (~1e-4) where x - floor(x) rounds up to 1, and stays far below a wrong term's error
        assert np.median(r.e) < 2.0 ** -18 and r.e.max() < 2.0 ** -13
    # the lattice wraps every 256 cells, on both sides of 0
    q = np.array([[0.25, 0.625, 0.125]], np.float32)
    for s in (256, -256, 512, -768):
        assert oracle.perlin_noise(q[0] + s) == oracle.perlin_noise(q[0])
        assert perlin(q + s).v[0] == pytest.approx(perlin(q).v[0], abs=2e-5)


@pytest.mark.parametrize("density", [0.1, 0.7, 4.0, 13.0, 50.0])
def test_texture_values_match_the_oracle(oracle, density):
    """Every non-image leaf kind and a checker of two of them, at densities 0.1-50, through orc_texture_value."""
    texs = [tex_noise(capi.RT_TEX_NOISE_PERLIN, density), tex_noise(capi.RT_TEX_NOISE_TURBULANCE, density),
            tex_noise(capi.RT_TEX_NOISE_MARBLE, density), tex_wood((0.9, 0.5, 0.1), (0.1, 0.2, 0.7), density, 37.0),
            tex_constant((0.2, 0.4, 0.6)), tex_checker(0, 3)]
    d = make_desc([((0, 0, 0), 1.0, 0)], [capi.rt_material(capi.RT_MAT_LAMBERTIAN, 0, (0, 0, 0), 0)], texs)
    sc = oracle.scene(d)
    pts = lattice_points()[:: 3] / np.float32(max(density, 1.0))
    n = np.tile(np.float32([0, 1, 0]), (len(pts), 1))
    for ix in range(len(texs)):
        want, err, tie = texture_value(texs, ix, pts, n, sfu=False)
        got = np.array([sc.texture_value(ix, 0.0, 0.0, q) for q in pts], np.float64)
        bad = (np.abs(got - want).max(axis=1) > err + 1e-12) & ~tie
        assert not bad.any(), (ix, float((np.abs(got - want).max(axis=1) - err)[bad].max()), pts[bad][:3])
        assert tie.mean() < 0.12, (ix, float(tie.mean()))  # the 100 points within 2^-30 of 0 lie on the checker's planes


@pytest.mark.parametrize("levels", list(range(0, 12)))
def test_oracle_resolves_checker_chains_as_deep_as_the_device(oracle, levels):
    """Up to RT_MAX_CHECKER_DEPTH = 8 checker levels resolve to the leaf; one more is past the loop's guard and gives the
    guard's white, as on the device — rt_scene_create refuses such a description, so neither renders it."""
    texs = [tex_constant((0.2, 0.4, 0.6))] + (checker_chain(levels, 0, 0, first=1) if levels else [])
    d = make_desc([((0, 0, 0), 1.0, 0)], [capi.rt_material(capi.RT_MAT_LAMBERTIAN, len(texs) - 1, (0, 0, 0), 0)], texs)
    got = oracle.scene(d).texture_value(len(texs) - 1, 0.0, 0.0, (0.13, 0.27, -0.61))
    want = (0.2, 0.4, 0.6) if levels <= 8 else (1.0, 1.0, 1.0)
    assert np.array_equal(got, np.float32(want)), (levels, got)


def test_oracle_stops_on_a_checker_cycle(oracle):
    """A cycle (even = itself) ends at the guard instead of looping: white, like the device."""
    texs = [tex_constant((0.2, 0.4, 0.6)), tex_checker(1, 0)]
    d = make_desc([((0, 0, 0), 1.0, 0)], [capi.rt_material(capi.RT_MAT_LAMBERTIAN, 1, (0, 0, 0), 0)], texs)
    sc = oracle.scene(d)
    assert np.array_equal(sc.texture_value(1, 0.0, 0.0, (0.05, 0.05, 0.05)), np.float32([1, 1, 1]))  # sines > 0: even = self
    assert np.array_equal(sc.texture_value(1, 0.0, 0.0, (-0.05, 0.05, 0.05)), np.float32([0.2, 0.4, 0.6]))  # odd: the leaf


def test_sphere_uv_matches_the_oracle(oracle):
    r = np.random.default_rng(5)
    n = r.normal(size=(3000, 3))
    n /= np.linalg.norm(n, axis=1, keepdims=True)
    n = np.concatenate([n, [[0, 1, 0], [0, -1, 0], [-1, 0, 0], [-1, 0, -0.0], [1, 0, 0], [0, 0, 1], [0, 0, -1]]]).astype(np.float32)
    u, v = sphere_uv(n)
    got = np.array([oracle.sphere_uv(q) for q in n])
    assert np.abs(got[:, 0] - u).max() <= UV_ERR and np.abs(got[:, 1] - v).max() <= UV_ERR
    # the seam: n.z = -0 gives u = 1 (last column), n.z = +0 a u a hair below 0 (first column): atan2f(+-0, -1) = +-float(pi)
    assert got[-4, 0] == 1.0 and -1e-7 < got[-5, 0] <= 0.0


def test_optics_match_the_oracle(oracle):
    r = np.random.default_rng(6)
    for _ in range(300):
        v = r.normal(size=3).astype(np.float32)
        n = r.normal(size=3)
        n = (n / np.linalg.norm(n)).astype(np.float32)
        v64, n64 = v.astype(np.float64), n.astype(np.float64)
        refl = v64 - 2 * (v64 @ n64) * n64
        assert np.abs(oracle.reflect(v, n) - refl).max() <= 8 * UZ * (np.abs(v64).max() + 2 * abs(v64 @ n64)) + 1e-30
        mu = float(np.float32(r.choice([0.7, 1.0, 1 / 1.5, 1.5, 2.4, 1 / 2.4])))
        i = v64 / np.linalg.norm(v64)
        cin = i @ n64
        delta = 1 - mu * mu * (1 - cin * cin)
        ok, out = oracle.refract(v, n, mu)
        if abs(delta) > 1e-5:
            assert ok == (delta > 0)
            if ok:
                want = mu * (i - n64 * cin) - n64 * np.sqrt(delta)
                assert np.abs(out - want).max() <= 1e-5 / np.sqrt(delta)
        c = float(np.float32(r.uniform(0, 1)))
        for ri in (0.7, 1.0, 1.5, 2.4):
            ri = float(np.float32(ri))
            assert abs(oracle.shlick(c, ri) - schlick(c, ri)) <= 8 * UZ + 4 * U


def test_philox_draws_reproduce_the_oracles_scattered_rays(oracle):
    """The host knows every probe ray's uniforms: metal directions (reflection + roughness * ball) and dielectric
    reflect / refract choices of orc_shade_probe follow from the restated Philox4x32-10, u01 and ball sampler."""
    texs = [tex_constant((0.5, 0.5, 0.5))]
    mats = [capi.rt_material(capi.RT_MAT_METAL, -1, (0.9, 0.8, 0.7), 0.7), capi.rt_material(capi.RT_MAT_DIELECTRIC, -1, (1, 1, 1), 1.5)]
    d = make_desc([((0, 0, 0), 1.0, 0), ((10, 0, 0), 1.0, 1)], mats, texs)
    r = np.random.default_rng(8)
    n = r.normal(size=(4000, 3))
    n[:, 1] = np.abs(n[:, 1])
    n /= np.linalg.norm(n, axis=1, keepdims=True)
    which = np.arange(4000) % 2
    centre = np.stack([10.0 * which, 0 * which, 0 * which], 1)
    rays = np.zeros(4000, capi.RAY_DTYPE)
    rays["origin"] = centre + 3 * n
    rays["direction"] = -n + r.normal(scale=0.3, size=(4000, 3))
    seed = 1000
    p = capi.rt_render_params()
    p.seed, p.tmin, p.bloom, p.max_depth = seed, 1e-5, 0.1, 50
    sc = oracle.scene(d)
    out = sc.shade_probe(rays, p)
    hits = sc.trace(rays)
    u1, u2, u3, u4 = probe_draws(len(rays), seed)
    met = (hits["id"] == 0)
    ball, berr = unit_ball(u1, u2, u3)
    dn = rays["direction"].astype(np.float64)
    dn /= np.linalg.norm(dn, axis=1, keepdims=True)
    hn = hits["n"].astype(np.float64)
    refl = dn - 2 * (dn * hn).sum(1, keepdims=True) * hn
    want = refl + 0.7 * ball
    got = out["scattered"]["direction"].astype(np.float64)
    cont = out["continues"] == 1
    assert (np.abs(got - want).max(axis=1)[met & cont] <= 0.7 * (2 * U * 8) + 16 * UZ).all()  # libm sin/cos: ~2 ulp
    dots = (want * hn).sum(1)
    assert (cont[met] == (dots[met] > 0))[np.abs(dots[met]) > 1e-5].all()
    # dielectric: reflected iff the draw is below Schlick (when refraction is possible)
    diel = hits["id"] == 1
    dd = rays["direction"].astype(np.float64)
    ddn = (dd * hn).sum(1)
    ent = ddn < 0
    cosine = -ddn / np.linalg.norm(dd, axis=1)
    prob = schlick(cosine, 1.5)
    reflected = np.abs(got - (dd - 2 * ddn[:, None] * hn)).max(axis=1) <= 1e-5 * np.abs(dd).max(axis=1) + 1e-6
    sel = diel & ent & (np.abs(u4 - prob) > 1e-5)
    assert sel.sum() > 800
    assert np.array_equal(reflected[sel], (u4 < prob)[sel])
