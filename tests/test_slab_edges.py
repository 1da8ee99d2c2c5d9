"""Every ray query at the edges of the box test, against the brute-force oracle.

The primitive tests of every query are the reference's own binary64 arithmetic; the box test in front of them (make_rayf / slab in
csrc/traverse.cuh) is binary32 with a rounding-error slack, on boxes rounded outwards at build time.  Ids and t equal the oracle's bit
for bit only if that test never culls a box that holds a hit.  Random rays almost never come within an ulp of a box face, so the rays
here are built to: tangent to spheres, through the edges and corners of quads and triangles (axis-aligned ones among them, whose
binary32 box has no thickness), in the plane of a face with that direction component exactly 0, with direction components of 0,
subnormal or around the 1/d clamp, direction magnitudes of 1e-20 and 1e20, scenes translated to 1e6 .. 1e9, moving spheres at times
outside [0, 1], and Transforms (rays made in the local frame, then mapped to world space).

Each family is built in two containers:
- a flat `list`: the reference culls nothing there, so its container semantics (oracle mode 0) equal brute force (mode 1);
- a `bvh`: the reference's AABB::hit drops some hits that Sphere::hit / Quad::hit accept (a slab-edge cull) and its answer depends
  on the tree; the GPU returns the brute-force answer.  The CPU test classifies every mode 0 != mode 1 ray and fails on anything but
  such a cull.
The GPU equals mode 1 in both, on every tree variant and traversal knob set.
"""
import functools

import numpy as np
import pytest

import edge_rays as er
from scenes_util import compare_hits
from test_transmittance import assert_same_transmittance
from test_world_hit import assert_same_records
from transmittance_oracle import TransmittanceOracle
from world_hit_oracle import WorldHitOracle

TIMES = [-1.0, -2.0 ** -52, 0.0, 1.0, 1.0 + 2.0 ** -52, 2.0]
XFORMS = {"similarity": ([0.7, -1.3, 2.1], ([1, 2, 3], 37.0), [1.7, 1.7, 1.7]),
          "nonuniform": ([-0.4, 0.9, 0.3], ([0, 1, 1], 61.0), [2.0, 0.5, 1.3]),
          "mirror": ([0.2, 0.1, -0.6], ([1, 0, 1], 23.0), [1.3, -0.8, 1.1])}
FAMILIES = ["tangent_axis", "tangent_oblique", "planar_edges", "in_face_plane", "special_d", "tiny_d", "huge_d", "far_1e6", "far_1e7",
            "far_m3e8", "far_1e9_special", "moving_times", "xf_similarity", "xf_nonuniform", "xf_mirror"]
N = 3000
# d scaled by 1e20 puts the hits at t ~ 1e-20: those rays are traced on [1e-30, inf)
T_MIN = {"huge_d": 1e-30}

# mode 0 != mode 1 rays in the bvh container, per family (printed at the end of the module)
CULLS = {}


@pytest.fixture(scope="module", autouse=True)
def report():
    yield
    if CULLS:
        print("\nreference slab-edge culls (bvh container, mode 0 misses or finds a farther hit than brute force):")
        for k, (n, c) in sorted(CULLS.items()):
            print(f"  {k:18s} {c:6d} of {n}")


KNOBS = {"fifo64_refill1": {"RT2025_FIFO_SLOTS": "64", "RT2025_REFILL_MIN": "1"}, "no_fifo": {"RT2025_FIFO_SLOTS": "0"},
         "park": {"RT2025_PARK_LEAVES": "1"}}


@pytest.fixture(params=[(t, k) for t in ("by_size", "four_wide", "binary") for k in KNOBS], ids=lambda p: f"{p[0]}-{p[1]}")
def variant(request, monkeypatch):
    """The tree rt_scene_create picks by size, the four-wide collapse forced and the binary tree forced, each with the prepared-ray FIFOs
    refilled lane by lane, with direct refill (no FIFO) and with postponed leaves: every traversal variant the queries share."""
    tree, knobs = request.param
    if tree == "four_wide":
        monkeypatch.setenv("RT2025_WIDE_BVH", "1")
    elif tree == "binary":
        monkeypatch.setenv("RT2025_WIDE_BVH", "0")
    for k, v in KNOBS[knobs].items():
        monkeypatch.setenv(k, v)
    return request.param


def family(name):
    """-> (Geometry, o, d, time, transform or None): seeded, the same on every call."""
    rng = np.random.default_rng(FAMILIES.index(name) + 100)
    time = rng.uniform(0, 1, N)
    xf = None
    if name in ("tangent_axis", "tangent_oblique"):
        g = er.Geometry(er.spheres(rng))
        o, d = (er.sphere_tangent_axis if name == "tangent_axis" else er.sphere_tangent_oblique)(g, rng, N)
    elif name in ("planar_edges", "in_face_plane"):
        g = er.Geometry(planars=er.planars(rng))
        o, d = (er.planar_edges if name == "planar_edges" else er.in_face_plane)(g, rng, N)
    elif name == "moving_times":
        g = er.Geometry(er.spheres(rng, moving=True))
        time = np.repeat(TIMES, N // len(TIMES))
        parts = [(er.sphere_tangent_axis if k % 2 else er.sphere_tangent_oblique)(g, rng, N // len(TIMES), time=t) for k, t in enumerate(TIMES)]
        o, d = np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])
    else:
        offset = {"far_1e6": 1e6, "far_1e7": 1e7, "far_m3e8": -3e8, "far_1e9_special": 1e9}.get(name, 0.0)
        g = er.Geometry(er.spheres(rng, offset=offset), er.planars(rng, offset=offset))
        o1, d1 = er.sphere_tangent_oblique(g, rng, N // 2)
        o2, d2 = er.planar_edges(g, rng, N - N // 2)
        o, d = np.concatenate([o1, o2]), np.concatenate([d1, d2])
        if name in ("special_d", "far_1e9_special"):
            o, d = er.with_special_component(o, d, rng)
        elif name == "tiny_d":
            d = d * 1e-20
        elif name == "huge_d":
            d = d * 1e20
        elif name.startswith("xf_"):
            xf = XFORMS[name[3:]]
            offset_, (axis, deg), scale = xf
            q = quat_axis_angle(axis, deg)
            o, d = er.to_world(o, d, np.asarray(offset_), q, scale)
    return g, o, d, time, xf


def quat_axis_angle(axis, deg):
    a = np.asarray(axis, np.float64) / np.linalg.norm(axis)
    h = np.radians(deg) / 2
    return np.concatenate([[np.cos(h)], np.sin(h) * a])


def build(rt, g, container, xf=None):
    b = rt.Builder(3)
    prims = g.build(b, b.lambertian(b.solid(0.5, 0.5, 0.5)))
    inner = b.list(prims) if container == "list" else b.bvh(prims)
    if xf is not None:
        offset, (axis, deg), scale = xf
        inner = b.transform(inner, offset=offset, quat=b.quat_axis_angle(axis, deg), scale=scale)
    hs = b.finish(b.list([inner]))
    hs._builder = b
    return hs


@functools.lru_cache(maxsize=None)
def case(name, container):
    """The scene, its rays and the oracle's answers in both modes."""
    import orc
    rt = orc.rt
    g, o, d, time, xf = family(name)
    hs = build(rt, g, container, xf)
    rays = rt.make_rays(o, d, time)
    osc = orc.OracleScene(hs)
    t_min = T_MIN.get(name, 1e-8)
    return hs, rays, osc.closest_hit(rays, t_min=t_min, mode=1), osc.closest_hit(rays, t_min=t_min, mode=0), osc.ranks()


def assert_same_hits(rt, got, want):
    """compare_hits, where a sphere hit at a pole may carry v = NaN: Sphere::get_sphere_uv takes acos of a normal component that
    rounding puts just beyond +-1.  The NaN patterns must agree; the numbers elsewhere are compared as compare_hits does."""
    for f in ("u", "v"):
        assert np.array_equal(np.isnan(got[f]), np.isnan(want[f])), f"{f}: NaN patterns differ"
    got, want = got.copy(), want.copy()
    for f in ("u", "v"):
        got[f][np.isnan(got[f])] = 0.0
        want[f][np.isnan(want[f])] = 0.0
    compare_hits(rt, got, want)


def same_hits(a, b):
    return (a["prim_id"] == b["prim_id"]) & (a["inst_id"] == b["inst_id"]) & (a["t"].view(np.int64) == b["t"].view(np.int64))


@pytest.mark.parametrize("name", FAMILIES)
def test_flat_list_reference_equals_brute_force(rt, name):
    """In a flat list the reference tests every child: its answer is the brute-force one, ray for ray."""
    hs, rays, want1, want0, _ = case(name, "list")
    hit = want1["prim_id"] != rt.RT_NONE
    assert 0.1 < hit.mean(), "the family should graze geometry"
    assert same_hits(want0, want1).all()


@pytest.mark.parametrize("name", FAMILIES)
def test_bvh_reference_differs_only_by_slab_edge_culls(rt, name):
    """Inside a BVH the reference's AABB::hit may drop a hit that the primitive test accepts.  Every mode 0 != mode 1 ray must be such a
    cull: brute force finds a nearer hit, or the same t with a lower tie rank.  Anything else would be a bug in the oracle."""
    hs, rays, want1, want0, ranks = case(name, "bvh")
    diff = ~same_hits(want0, want1)
    h1 = want1["prim_id"] != rt.RT_NONE
    h0 = want0["prim_id"] != rt.RT_NONE
    rank = lambda w, m: ranks[w["prim_id"][m]]
    cull = diff & h1 & (~h0 | (want1["t"] < want0["t"]))
    tie = diff & h1 & h0 & (want1["t"] == want0["t"])
    cull[tie] |= rank(want1, tie) < rank(want0, tie)
    other = diff & ~cull
    CULLS[name] = (len(rays), int(cull.sum()))
    assert not other.any(), f"{int(other.sum())} rays where the reference's BVH answer is not a culled subset of brute force"


@pytest.mark.gpu
@pytest.mark.usefixtures("variant")
@pytest.mark.parametrize("container", ["list", "bvh"])
@pytest.mark.parametrize("name", FAMILIES)
def test_closest_hit_and_occlusion_equal_brute_force(gpu, rt, name, container):
    hs, rays, want, _, _ = case(name, container)
    t_min = T_MIN.get(name, 1e-8)
    sc = rt.Scene(hs)
    got, _ = sc.closest_hit(rays, t_min=t_min)
    assert_same_hits(rt, got, want)
    # occlusion with t_max_i at the hit t and its binary64 neighbours: the interval is closed, the t of the hit is the oracle's own
    hit = want["prim_id"] != rt.RT_NONE
    t_star = np.where(hit, want["t"], 1.0)
    for t_max in (t_star, np.nextafter(t_star, np.inf), np.nextafter(t_star, -np.inf)):
        occ, _ = sc.occluded(rays, t_min=t_min, t_max=t_max)
        assert np.array_equal(occ, hit & (want["t"] <= t_max)), f"{int((occ != (hit & (want['t'] <= t_max))).sum())} occlusion answers differ"
    sc.close()


def media_case(rt, moving):
    """Sphere-bounded media and a few surfaces, all in flat lists (the oracle's answer is then the exact one), and rays that are tangent
    to a boundary, cut a chord near the t1 + 1e-4 rule of ConstantMedium::hit, or start on the boundary.  moving: the boundaries and
    surfaces move, and the rays take the times of TIMES."""
    rng = np.random.default_rng(44 + moving)
    b = rt.Builder(5)
    g = er.Geometry(er.spheres(rng, n=4, moving=moving))
    surf = er.Geometry(er.spheres(rng, n=3, moving=moving), er.planars(rng, n=2))
    mats = b.lambertian(b.solid(0.5, 0.5, 0.5))
    media = [b.medium(s, dens, b.solid(1, 1, 1)) for s, dens in zip(g.build(b, b.empty()), (0.3, 2.0, 40.0, 1e3))]
    hs = b.finish(b.list(media + surf.build(b, mats)))
    hs._builder = b
    n = 4000
    time = np.repeat(TIMES, n // len(TIMES)) if moving else rng.uniform(0, 1, n)
    n = len(time)
    o, d = np.zeros((n, 3)), np.zeros((n, 3))
    for i in range(n):
        c, r = er.centres_at(g, time[i])[rng.integers(len(g.spheres))]
        di = er.unit(rng.normal(size=3))
        nrm = er.perpendicular(di[None], rng)[0]
        kind = i % 3
        if kind == 0:  # tangent
            h = r
        elif kind == 1:  # chord of 1e-4 (1 + small): the second boundary hit sits at the t1 + 1e-4 rule
            h = np.sqrt(r * r - (0.5e-4 * (1 + rng.uniform(-1e-6, 1e-6))) ** 2)
        else:  # starting on the boundary, heading in or out
            h = r * rng.uniform(-1, 1)
        p = c + h * nrm
        back = 0.0 if kind == 2 else rng.uniform(0.5, 3)
        if kind == 2:
            p = c + r * er.unit(rng.normal(size=3))
        o[i] = er.nudge(p - back * di, rng.integers(-3, 4, 3))
        d[i] = di
    return hs, rt.make_rays(o, d, time)


@pytest.mark.gpu
@pytest.mark.usefixtures("variant")
@pytest.mark.parametrize("moving", [False, True], ids=["static", "moving_times"])
def test_transmittance_and_world_hit_at_medium_edges(gpu, rt, moving):
    hs, rays = media_case(rt, moving)
    sc = rt.Scene(hs)
    t_max = np.where(np.arange(len(rays)) % 2 == 0, np.inf, np.random.default_rng(1).uniform(0.5, 6, len(rays)))
    want_T = TransmittanceOracle(hs).transmittance(rays, t_max=t_max)
    got_T, _ = sc.transmittance(rays, t_max=t_max)
    assert_same_transmittance(got_T, want_T)
    assert ((want_T > 0) & (want_T < 1)).mean() > 0.1
    want_W = WorldHitOracle(hs).world_hit(rays, t_max=t_max, seed=9, segment=2)
    got_W, _ = sc.world_hit(rays, t_max=t_max, seed=9, segment=2)
    assert_same_records(rt, hs, got_W, want_W)
    sc.close()


@pytest.mark.gpu
def test_out_of_range_times_inside_a_bvh(gpu, rt, orc):
    """A moving sphere in a BVH, rays straight down -z over its centre at time tau outside [0, 1]: the reference's box (bounded over
    [0, 1]) culls some of these, Sphere::hit does not; every query returns the hit."""
    b = rt.Builder(1)
    m = b.empty()
    hs = b.finish(b.list([b.bvh([b.sphere_moving([0, 0, 0], [4, 0, 0], 1.0, m), b.sphere([20, 20, 20], 0.5, m)])]))
    sc, osc = rt.Scene(hs), orc.OracleScene(hs)
    taus = np.array([-1.0, -0.5, -2.0 ** -52, 1 + 2.0 ** -52, 1.5, 2.0, 5.0])
    rays = rt.make_rays(np.column_stack([4 * taus, np.zeros_like(taus), np.full_like(taus, 6.0)]), np.tile([0, 0, -1.0], (len(taus), 1)), taus)
    want = osc.closest_hit(rays, mode=1)
    assert (want["prim_id"] != rt.RT_NONE).all() and np.all(want["t"] == 5.0)
    got, _ = sc.closest_hit(rays)
    assert_same_hits(rt, got, want)
    assert sc.occluded(rays)[0].all()
    assert not sc.transmittance(rays)[0].any()
    rec, _ = sc.world_hit(rays)
    assert np.array_equal(rec["prim_id"], want["prim_id"]) and np.array_equal(rec["t"], want["t"])


@pytest.mark.gpu
def test_device_lbvh_on_a_tangent_ray_soup(gpu, rt, orc):
    """About 60k spheres built into a device LBVH (one primitive per leaf), each the target of a tangent ray."""
    rng = np.random.default_rng(60)
    n = 60_000
    side = int(np.ceil(n ** (1 / 3)))
    idx = np.stack(np.unravel_index(np.arange(n), (side, side, side)), axis=1)
    g = er.Geometry([(idx[i] * 3.0 + rng.uniform(-0.5, 0.5, 3), float(rng.uniform(0.1, 1.0)), np.zeros(3)) for i in range(n)])
    hs = build(rt, g, "list")
    m = 30_000
    o1, d1 = er.sphere_tangent_oblique(g, rng, m // 2)
    o2, d2 = er.sphere_tangent_axis(g, rng, m - m // 2)
    rays = rt.make_rays(np.concatenate([o1, o2]), np.concatenate([d1, d2]), rng.uniform(0, 1, m))
    sc = rt.Scene(hs, flags=rt.RT_BUILD_DEVICE_LBVH)
    assert sc.info().n_nodes == n - 1
    want = orc.OracleScene(hs).closest_hit(rays, mode=1)
    assert (want["prim_id"] != rt.RT_NONE).mean() > 0.2
    got, _ = sc.closest_hit(rays)
    assert_same_hits(rt, got, want)
    hit = want["prim_id"] != rt.RT_NONE
    t_star = np.where(hit, want["t"], 1.0)
    assert np.array_equal(sc.occluded(rays, t_max=t_star)[0], hit)
    assert not sc.occluded(rays, t_max=np.nextafter(t_star, -np.inf))[0].any()
