"""Perlin noise and NoiseTexture::value of the oracle against an independent restatement written from the reference's source
(utils/perlin.rs:41-97, texture.rs:191-196) in plain Python floats - same operations in the same order, so the comparison is
exact up to libm's sin.  The reference holds no vectors for the noise; this pins the oracle's table lookups (perm_x ^ perm_y ^
perm_z with the wrap-around of negative lattice coordinates), the Hermite weights, the 7-octave turbulence and the marble formula.
Lattice points are an analytic known answer: every corner offset but one has weight 0 and that one's dot product is with the
zero vector, so noise == 0 exactly."""
import ctypes as C
import math

import numpy as np


class _Perlin(C.Structure):
    _fields_ = [("randvec", (C.c_double * 3) * 256), ("perm_x", C.c_uint32 * 256), ("perm_y", C.c_uint32 * 256), ("perm_z", C.c_uint32 * 256)]


def _as_i64(x):
    """Rust's `f64 as i64`: NaN -> 0, saturating at -2^63 and 2^63 - 1."""
    if math.isnan(x):
        return 0
    if x >= 2.0 ** 63:
        return 2 ** 63 - 1
    if x <= -2.0 ** 63:
        return -2 ** 63
    return int(x)


def _noise(t, p):  # perlin.rs:41-60
    fl = [float("nan") if math.isnan(x) else (x if math.isinf(x) else float(math.floor(x))) for x in p]
    i, j, k = (_as_i64(x) for x in fl)  # (i + di) & 255 below: the low byte of the wrapping i64 sum
    u, v, w = (p[a] - fl[a] for a in range(3))
    uu, vv, ww = (x * x * (3.0 - 2.0 * x) for x in (u, v, w))  # perlin.rs:74
    accum = 0.0
    for di in range(2):
        for dj in range(2):
            for dk in range(2):
                g = t.randvec[t.perm_x[(i + di) & 255] ^ t.perm_y[(j + dj) & 255] ^ t.perm_z[(k + dk) & 255]]
                wv = (u - di, v - dj, w - dk)
                dot = g[0] * wv[0] + g[1] * wv[1] + g[2] * wv[2]
                accum += (di * uu + (1 - di) * (1.0 - uu)) * (dj * vv + (1 - dj) * (1.0 - vv)) * (dk * ww + (1 - dk) * (1.0 - ww)) * dot
    return accum


def _turb(t, p, depth):  # perlin.rs:62-72
    accum, q, weight = 0.0, list(p), 1.0
    for _ in range(depth):
        accum += weight * _noise(t, q)
        q = [2.0 * x for x in q]
        weight = 0.5 * weight
    return abs(accum)


def test_noise_texture_matches_a_plain_restatement(rt, orc):
    b = rt.Builder(17)
    scale = 1.75
    tex = b.noise(scale)
    hs = b.finish(b.list([b.sphere([0, 0, 0], 1.0, b.lambertian(tex))]), width=8, spp=1)
    d = hs.desc.contents
    assert d.n_perlins == 1
    tab = C.cast(d.perlins, C.POINTER(_Perlin)).contents
    # the tables are what Perlin::default() builds: unit vectors and three permutations of 0..255
    for g in tab.randvec:
        assert abs(math.sqrt(g[0] * g[0] + g[1] * g[1] + g[2] * g[2]) - 1.0) < 1e-12
    for perm in (tab.perm_x, tab.perm_y, tab.perm_z):
        assert sorted(perm) == list(range(256))
    osc = orc.OracleScene(hs)
    tex = C.c_uint32.from_address(d.materials + 176 * int(hs.objects()[0]["material"]) + 4).value  # the texture's index after flattening
    rng = np.random.default_rng(5)
    pts = [list(rng.uniform(-300.0, 300.0, 3)) for _ in range(400)]
    pts += [[0.5, -0.5, 2.5], [-1e-9, 255.999, -256.0], [1e5 + 0.25, -1e5 - 0.75, 3.125], [-0.0, 0.0, 0.0]]
    pts += saturation_points(rng)
    worst = 0.0
    for p in pts:
        want = 0.5 * (1.0 + math.sin(scale * p[2] + 10.0 * _turb(tab, p, 7)))  # texture.rs:193-194
        got = osc.texture_value(tex, 0.0, 0.0, p)
        assert got[0] == got[1] == got[2] or math.isnan(got[0])
        assert math.isnan(got[0]) == math.isnan(want), (p, got[0], want)
        if not math.isnan(want):
            worst = max(worst, abs(got[0] - want))
    assert worst <= 4e-16, worst  # one ulp of a value in [0, 1]: libm's sin is the only operation that may differ
    # lattice points: noise is exactly zero, so turbulence is zero and the marble value is 0.5 (1 + sin(scale z))
    for p in ([3.0, -7.0, 12.0], [-255.0, 256.0, 0.0], [1024.0, 2.0, -5.0]):
        assert _noise(tab, p) == 0.0
        got = osc.texture_value(tex, 0.0, 0.0, p)
        assert got[0] == 0.5 * (1.0 + math.sin(scale * p[2]))


# where `as i64` saturates: floor(p) at and around 2^63 (the largest double below it is 2^63 - 1024), infinities and NaN
SATURATION = [9.1e18, 9.2e18, 9.21e18, 9.22e18, float(np.nextafter(2.0 ** 63, 0.0)), 2.0 ** 63, 1e19]
SATURATION = SATURATION + [-x for x in SATURATION] + [float("inf"), float("-inf"), float("nan")]


def saturation_points(rng):
    """Each saturation value on each axis, the other two axes fractional."""
    out = []
    for x in SATURATION:
        for a in range(3):
            for _ in range(2):
                p = list(rng.uniform(-50.0, 50.0, 3))
                p[a] = x
                out.append(p)
    return out


def test_noise_saturates_like_rust_as_i64(rt, orc):
    """The lattice index of a coordinate at or beyond 2^63 is i64::MAX (i64::MIN below -2^63), not the value the last exact
    conversion gives, and NaN is index 0.  A known answer of the marble texture at p = (9.21e18, 0.5, 0.3)."""
    b = rt.Builder(17)
    tex = b.noise(1.0)
    hs = b.finish(b.list([b.sphere([0, 0, 0], 1.0, b.lambertian(tex))]), width=8, spp=1)
    d = hs.desc.contents
    tab = C.cast(d.perlins, C.POINTER(_Perlin)).contents
    osc = orc.OracleScene(hs)
    tex = C.c_uint32.from_address(d.materials + 176 * int(hs.objects()[0]["material"]) + 4).value
    assert _as_i64(9.21e18) == 9210000000000000000 and _as_i64(2.0 ** 63) == 2 ** 63 - 1 and _as_i64(-1e19) == -2 ** 63
    p = [9.21e18, 0.5, 0.3]
    want = 0.5 * (1.0 + math.sin(p[2] + 10.0 * _turb(tab, p, 7)))
    got = osc.texture_value(tex, 0.0, 0.0, p)
    assert abs(got[0] - want) <= 4e-16 and abs(want - 0.8738799519358917) <= 4e-16, (got[0], want)
