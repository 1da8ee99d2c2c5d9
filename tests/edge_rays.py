"""Rays placed exactly on, and a few binary64 ulps either side of, the edges where a box test can go wrong (tests/test_slab_edges.py).

A geometry is a plain description - spheres (centre, radius, centre_vec) and planars (kind, Q, u, v) - so that the ray families can be
derived from it and the same description can be built into any container.  Every family is seeded; nothing here touches a device.
"""
import numpy as np

SPECIAL_D = np.array([0.0, -0.0, 5e-324, -5e-324, 1e-310, 1e-30 * (1 + 2.0 ** -52), 1e-30 * (1 - 2.0 ** -52), -1e-30 * (1 + 2.0 ** -52),
                      -1e-30 * (1 - 2.0 ** -52)])


def nudge(x, k):
    """x moved by k binary64 ulps, elementwise (|k| <= 3)."""
    x = np.array(x, dtype=np.float64, copy=True)
    k = np.broadcast_to(k, x.shape)
    for step in range(1, 4):
        x = np.where(k >= step, np.nextafter(x, np.inf), x)
        x = np.where(k <= -step, np.nextafter(x, -np.inf), x)
    return x


def unit(v):
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


def perpendicular(d, rng):
    """A random unit vector perpendicular to each row of d."""
    return unit(np.cross(d, rng.normal(size=d.shape)))


class Geometry:
    def __init__(self, spheres=(), planars=()):
        self.spheres = list(spheres)  # (c, r, cv)
        self.planars = list(planars)  # (kind "quad" | "tri", q, u, v)

    def build(self, b, mat):
        ids = []
        for c, r, cv in self.spheres:
            ids.append(b.sphere_moving(c, c + cv, r, mat) if np.any(cv != 0) else b.sphere(c, r, mat))
        for kind, q, u, v in self.planars:
            ids.append((b.quad if kind == "quad" else b.triangle)(q, u, v, mat))
        return ids


def spheres(rng, n=8, offset=0.0, moving=False):
    """Centres U(-3, 3), radii U(0.1, 1): not dyadic, so c +- r is rounded."""
    return [(rng.uniform(-3, 3, 3) + offset, float(rng.uniform(0.1, 1.0)), rng.uniform(-2, 2, 3) if moving else np.zeros(3)) for _ in range(n)]


def planars(rng, n=6, offset=0.0):
    """Random quads and triangles, and axis-aligned quads (a binary32 box of zero thickness on one axis) including the six faces of a box."""
    out = []
    for i in range(n):
        out.append(("quad" if i % 2 == 0 else "tri", rng.uniform(-3, 3, 3) + offset, rng.uniform(-1.5, 1.5, 3), rng.uniform(-1.5, 1.5, 3)))
    for a in range(3):
        u, v = np.zeros(3), np.zeros(3)
        u[(a + 1) % 3], v[(a + 2) % 3] = rng.uniform(0.5, 2.0), rng.uniform(0.5, 2.0)
        out.append(("quad", rng.uniform(-3, 3, 3) + offset, u, v))
    lo, hi = rng.uniform(-3, -0.5, 3) + offset, rng.uniform(0.5, 3, 3) + offset
    ext = hi - lo
    for a in range(3):
        u, v = np.zeros(3), np.zeros(3)
        u[(a + 1) % 3], v[(a + 2) % 3] = ext[(a + 1) % 3], ext[(a + 2) % 3]
        for side in (lo, hi):
            q = lo.copy()
            q[a] = side[a]
            out.append(("quad", q, u, v))
    return out


def centres_at(geom, time):
    return [(c + time * cv, r) for c, r, cv in geom.spheres]


def sphere_tangent_axis(geom, rng, n, time=0.0):
    """Rays along +-x / y / z tangent to a sphere: the tangent coordinate is c +- r, then 0..3 ulps either side; the third coordinate
    is off the centre plane by at most 1e-6 r."""
    cs = centres_at(geom, time)
    o, d = np.zeros((n, 3)), np.zeros((n, 3))
    for i in range(n):
        c, r = cs[rng.integers(len(cs))]
        a = rng.integers(3)
        b_ = (a + 1 + rng.integers(2)) % 3
        c_ = 3 - a - b_
        s = rng.choice([-1.0, 1.0])
        o[i, b_] = nudge(c[b_] + rng.choice([-1.0, 1.0]) * r, rng.integers(-3, 4))
        o[i, c_] = c[c_] + rng.uniform(-1e-6, 1e-6) * r
        o[i, a] = c[a] - s * (r + rng.uniform(1, 4))
        d[i, a] = s
    return o, d


def sphere_tangent_oblique(geom, rng, n, time=0.0):
    """Rays in the tangent plane of a sphere, the origin nudged by 0..3 ulps per component and up to 1e-6 r off the tangent point."""
    cs = centres_at(geom, time)
    pick = rng.integers(len(cs), size=n)
    c = np.array([cs[k][0] for k in pick])
    r = np.array([cs[k][1] for k in pick])[:, None]
    d = unit(rng.normal(size=(n, 3)))
    nrm = perpendicular(d, rng)
    side = unit(np.cross(d, nrm))
    p = c + r * nrm + side * r * rng.uniform(-1e-6, 1e-6, (n, 1))
    o = nudge(p - rng.uniform(1, 5, (n, 1)) * d, rng.integers(-3, 4, (n, 3)))
    return o, d


def planar_edges(geom, rng, n):
    """Rays through the edges and corners of quads and triangles: alpha, beta in {0, 1} and alpha + beta = 1 (the inclusive edges of
    quad.rs / triangle.rs), the origin nudged by 0..3 ulps per component."""
    P = geom.planars
    o, d = np.zeros((n, 3)), np.zeros((n, 3))
    for i in range(n):
        kind, q, u, v = P[rng.integers(len(P))]
        w = rng.uniform()
        if kind == "tri":
            ab = [(0, 0), (1, 0), (0, 1), (w, 0), (0, w), (w, 1 - w)][rng.integers(6)]
        else:
            ab = [(0, 0), (1, 0), (0, 1), (1, 1), (w, 0), (0, w), (w, 1), (1, w)][rng.integers(8)]
        p = q + ab[0] * u + ab[1] * v
        nrm = unit(np.cross(u, v))
        di = unit(rng.normal(size=3))
        if abs(di @ nrm) < 0.2:
            di = unit(di + 0.5 * nrm)
        o[i] = nudge(p - rng.uniform(1, 5) * di, rng.integers(-3, 4, 3))
        d[i] = di
    return o, d


def in_face_plane(geom, rng, n):
    """Rays lying in the plane of an axis-aligned quad, that component of d exactly 0, aimed at points around its edges."""
    P = [(q, u, v) for kind, q, u, v in geom.planars if kind == "quad" and np.count_nonzero(u) == 1 and np.count_nonzero(v) == 1]
    o, d = np.zeros((n, 3)), np.zeros((n, 3))
    for i in range(n):
        q, u, v = P[rng.integers(len(P))]
        a = int(np.flatnonzero((u == 0) & (v == 0))[0])
        tgt = q + rng.uniform(-0.1, 1.1) * u + rng.uniform(-0.1, 1.1) * v
        di = rng.normal(size=3)
        di[a] = 0.0
        di = unit(di)
        di[a] = 0.0
        o[i] = tgt - rng.uniform(1, 5) * di
        o[i, a] = q[a]
        d[i] = di
    return o, d


def with_special_component(o, d, rng):
    """The smallest component of every direction replaced by 0, a subnormal or +-1e-30 (1 +- 2^-52), around the clamp of 1/d."""
    d = d.copy()
    k = np.argmin(np.abs(d), axis=1)
    d[np.arange(len(d)), k] = rng.choice(SPECIAL_D, len(d))
    return o, d


def quat_rotate(q, v):
    w, x = q[0], np.asarray(q[1:])
    t = 2.0 * np.cross(x, v)
    return v + w * t + np.cross(x, t)


def to_world(o, d, offset, quat, scale):
    """Transform::transform of shapes.rs:74-78 applied to the local origin and direction (up to rounding)."""
    scale = np.asarray(scale, np.float64)
    return quat_rotate(quat, o * scale) + offset, quat_rotate(quat, d * scale)
