"""rt_shade on records built by hand, against the oracle's shade_record (oracle/orc.py OracleScene.shade_record).

rt_shade uses a record as given (include/rt2025.h): p, normal, u, v, front_face and material; t, prim_id and reserved are not read,
nor anything of a miss but its kind.  Records of real geometry only reach unit normals that face the ray, a front_face that agrees
with them, u and v in [0, 1], finite p and the primitive's own material.  Here each family takes records of world.hit (the oracle's
reference of rt_world_hit, tests/world_hit_oracle.py) and sets one field to edge values:
- material: every index of the table (the inner materials of Mix, DiffuseLight and Remapped chains too) on surface and medium records;
- p: exactly on a quad light and on a sphere light, inside a sphere light and at its centre, far from it (an infinite sphere pdf),
  on checker lattice points and one ulp off, 1e300, +-inf, NaN, and where Perlin's `as i64` saturates (9.2e18, 2^63);
- normal: unit facing the ray and away, scaled by 1e-3 and 1e3, zero, subnormal, 1e200, +-inf, NaN, with inst_id RT_NONE, a real
  Transform id or an arbitrary value (only a flag);
- u, v: texel edges and their neighbours, +-0, -1e-300, 1e300, +-inf, NaN;  front_face: 0, 1, 2, 0xFFFFFFFF;
- the ray: miss directions along the axes, on the atan2 branch cut and at the poles, zero, subnormal, huge, infinite and NaN; zero and
  NaN directions on hits; times NaN, +-inf and -0.0; garbage origins;
- beta per channel 1, subnormal, 1e308, inf, NaN, -0.0, -1, 0; radiance on entry 0, -0.0, NaN, inf or random;
- draw addresses: seeds 0 and 2^64 - 1, segments 0, max_depth - 2 and max_depth - 1 with max_depth up to 4095.
Checks row by row with the rules of test_shade.test_against_the_oracle; unread fields filled with NaN and random bits change no bit.
"""
import ctypes as C

import numpy as np
import pytest

import test_segment_kat as tsk
from scenes_util import disney_scene, materials_scene, obj_mesh_scene
from test_device_kat import edge_coords
from test_segment_kat import REL, SCATTER_COSINE, SCATTER_DISNEY, SCATTER_RAY, SCATTER_SPHERE, compare, draw, expected_beta
from world_hit_oracle import WorldHitOracle

RT_NONE = 0xFFFFFFFF
MAT_NAMES = ["empty", "lambertian", "metal", "dielectric", "diffuse_light", "isotropic", "transparent", "mix", "portal", "disney", "remapped"]
MAT_DIFFUSE_LIGHT, MAT_MIX, MAT_REMAPPED = 4, 7, 10
RT_SLOT_MIXTURE = 4
INACTIVE_STATES = np.array([0, 2, 0xFC, 0xFE], np.uint8)


@pytest.fixture(scope="module", autouse=True)
def report():
    yield
    rows = sorted((k, v) for k, v in tsk.STATS.items() if k.startswith("records"))
    if rows:
        print("\n%-40s %10s %10s %12s" % ("output", "values", "bit-equal", "max rel"))
        for k, (n, eq, mx) in rows:
            print("%-40s %10d %10d %12.3e" % (k, n, eq, mx))


# ---------------------------------------------------------------- scenes
def kinds_room(rt, lights="four", background="solid"):
    """Every material kind in one room: Empty, Lambertian with each texture kind (solid, checker, image nearest / raw / linear,
    noise, gradient, missing image), Metal with fuzz 0 and 0.35, Dielectric, Isotropic (also as a medium), DiffuseLight with and
    without an inner material, Mix three deep with an image-alpha ratio, Portal, Transparent, Disney (solid and textured) and
    RemappedMaterial faces (with and without a normal map); a transformed quad; lights: a flat list of a quad and three spheres
    ("four"), the same nested ("nested") or none; the background of the given kind.  hs._points: points on and around the lights."""
    rng = np.random.default_rng(41)
    b = rt.Builder(41)
    img = rng.uniform(0, 1, (6, 9, 4)).astype(np.float32)
    alpha = rng.uniform(0, 1, (8, 8, 4)).astype(np.float32)
    alpha[..., 3] = rng.uniform(0, 1, (8, 8)) > 0.5
    nm = rng.uniform(0.35, 0.65, (5, 5, 4)).astype(np.float32)
    nm[..., 2] = rng.uniform(0.8, 1.0, (5, 5))
    checker = b.checker(0.5, b.solid(0.9, 0.9, 0.9), b.solid(0.2, 0.3, 0.4))  # lattice at multiples of 0.5: exact in binary64
    image = b.image(img)
    texs = [b.solid(0.7, 0.6, 0.5), checker, image, b.image(img, raw=True), b.image(img, linear_format=True), b.noise(1.0),
            b.gradient([1, 1, 1], [0.2, 0.4, 0.8]), b.image_missing()]
    white, red = b.lambertian(texs[0]), b.lambertian(b.solid(0.8, 0.2, 0.1))
    glass = b.dielectric(b.solid(0.95, 1.0, 0.9), 1.5)
    disney = b.disney((0.8, 0.5, 0.3), roughness=0.3, metallic=0.4, spec_trans=0.3, clearcoat=0.5, sheen=0.4)
    mats = [b.empty()] + [b.lambertian(t) for t in texs] + [
        b.metal([0.9, 0.8, 0.7], 0.0), b.metal([0.8, 0.8, 0.9], 0.35), glass, b.isotropic(checker),
        b.diffuse_light(b.solid(2.0, 1.5, 1.0)), b.diffuse_light(checker, inner=b.metal([0.8, 0.7, 0.6], 0.2)),
        b.mix(b.mix_image(b.mix(white, glass, 0.3), b.transparent(), b.image(alpha)), b.diffuse_light(b.solid(1, 1, 1), inner=red), 0.55),
        b.portal([0.9, 0.95, 1.0], [0.0, 0.0, -3.0], b.quat_axis_angle([0, 1, 0], 15.0)), b.transparent(), disney,
        b.disney((1, 1, 1), tex=image, roughness=0.6, spec_trans=0.5, diff_trans=0.3, thin=1.0)]
    objs = []
    for k, m in enumerate(mats):
        x, y = (k % 5) * 2.0 - 4.0, (k // 5) * 2.0 - 2.5
        objs.append(b.sphere([x, y, 0], 0.8, m) if k % 2 == 0 else b.quad([x - 0.8, y - 0.8, 0.2], [1.6, 0, 0], [0, 1.6, 0.2], m))
    for k, (inner, nmap) in enumerate(((white, b.image(nm, raw=True)), (disney, RT_NONE))):
        pos = [[4.5, -2.5 + 2 * k, 0.5], [6.0, -2.5 + 2 * k, 0.3], [5.0, -1.0 + 2 * k, 0.0]]
        nrm = [[0.1, 0.2, 1.0], [-0.1, 0.1, 1.0], [0.0, -0.2, 1.0]]
        objs.append(b.obj_face(inner, pos, [[0, 0], [1, 0], [0.3, 1]], [np.array(v) / np.linalg.norm(v) for v in nrm], nmap))
    objs.append(b.transform(b.quad([-1, -1, 0], [2, 0, 0], [0, 2, 0], b.metal([0.7, 0.9, 0.7], 0.1)), offset=[0.0, -1.5, -3.0],
                            quat=b.quat_axis_angle([1, 1, 0], 30.0), scale=[1.5, 1.2, 1.0]))
    objs.append(b.medium(b.sphere([-4.5, 3.0, 2.0], 0.9, b.empty()), 0.8, b.solid(0.6, 0.7, 0.8)))
    lamp = b.diffuse_light(b.solid(6, 6, 6))
    e = b.empty()
    quad_light = ([-1.5, 5.0, -1.5], [3.0, 0.0, 0.0], [0.0, 0.0, 3.0])
    spots = [([-3.0, 4.0, 1.0], 0.5), ([3.0, 4.0, 1.0], 0.25), ([0.0, 4.5, -2.0], 0.75)]
    things = [b.quad([-8, -3.5, -8], [16, 0, 0], [0, 0, 16], white), b.quad(*quad_light, lamp)] + [b.sphere(c, r, lamp) for c, r in spots]
    light_objs = [b.quad(*quad_light, e)] + [b.sphere(c, r, e) for c, r in spots]
    lt = {"four": lambda: b.list(light_objs), "nested": lambda: b.list([light_objs[0], b.list(light_objs[1:3]), light_objs[3]]),
          "none": lambda: rt.RT_NONE}[lights]()
    bg = {"solid": lambda: b.solid(0.4, 0.5, 0.7), "gradient": lambda: b.gradient([1, 1, 1], [0.3, 0.5, 0.9]),
          "image": lambda: b.image(rng.uniform(0, 2, (16, 32, 4)).astype(np.float32), linear_format=True),
          "checker": lambda: b.checker(0.3, b.solid(0.9, 0.9, 0.9), b.solid(0.2, 0.2, 0.2)), "noise": lambda: b.noise(1.5)}[background]()
    hs = b.finish(b.list([b.bvh(things + objs)]), lt, width=24, spp=1, max_depth=12, vfov=60, look_from=(0, 1, 11), look_at=(0, 0, 0),
                  background=bg)
    hs._builder = b
    q, u, v = (np.array(x) for x in quad_light)
    pts = [q + a * u + c * v for a in (0.0, 0.25, 0.5, 1.0) for c in (0.0, 0.5, 0.75)]  # exactly on the lamp (dyadic fractions)
    for c, r in spots:
        c = np.array(c)
        for ax in np.eye(3):
            pts += [c + r * ax, c - r * ax, c + 0.5 * r * ax]  # on the sphere (exact axis points) and inside it
        pts += [c, c + np.array([1e150, 0.0, 0.0]), c + np.array([0.0, -1e150, 1e150])]  # the centre; far away (1 - cos_theta_max == 0)
    for k in range(-3, 4):  # checker lattice points and one ulp off them
        x = k * 0.5
        pts += [np.array([x, 0.5, x]), np.array([np.nextafter(x, 9.0), 1.0, x]), np.array([x, np.nextafter(-1.0, -9.0), np.nextafter(x, -9.0)])]
    hs._points = pts
    return hs


SCENES = {
    "materials": materials_scene,
    "disney": lambda rt: disney_scene(rt, width=24),
    "obj_mesh": lambda rt: obj_mesh_scene(rt, width=24),
    "panic": lambda rt: tsk.panic_scene(rt, True),
    "room_four_solid": lambda rt: kinds_room(rt, "four", "solid"),
    "room_nested_gradient": lambda rt: kinds_room(rt, "nested", "gradient"),
    "room_none_image": lambda rt: kinds_room(rt, "none", "image"),
    "room_four_checker": lambda rt: kinds_room(rt, "four", "checker"),
    "room_nested_noise": lambda rt: kinds_room(rt, "nested", "noise"),
}


def material_table(hs):
    d = hs.desc.contents
    raw = np.frombuffer(C.string_at(d.materials, 176 * d.n_materials), np.uint32).reshape(d.n_materials, 44)
    return raw[:, 0].copy(), raw[:, 2].copy()  # kind, inner


def emitting(hs):
    """Per material index: does shade_hit add an emission for it (the kind below its RemappedMaterial chain is DiffuseLight or Mix)."""
    kind, inner = material_table(hs)
    out = np.zeros(len(kind), bool)
    for m in range(len(kind)):
        k = m
        while kind[k] == MAT_REMAPPED:
            k = inner[k]
        out[m] = kind[k] in (MAT_DIFFUSE_LIGHT, MAT_MIX)
    return out


# ---------------------------------------------------------------- record families
def base_records(rt, orc, name, hs, rng):
    """Rays into the scene (camera rays, rays from inside it, the panic scene's own rays) and the records world.hit gives them."""
    cam = hs.camera
    px = np.stack([rng.integers(0, cam.image_width, 400), rng.integers(0, cam.image_height, 400)], axis=1)
    rays = [orc.camera_rays(cam, 5, px, 0), tsk.make_rays(rng.uniform(-4, 4, (600, 3)), rng.normal(size=(600, 3)), rng.uniform(0, 1, 600))]
    if name == "panic":
        rays.append(tsk.panic_rays(rng, 400))
    rays = np.concatenate(rays)
    rec = WorldHitOracle(hs).world_hit(rays, t_min=1e-8, seed=11, segment=0).view(rt.rt_hit_record_dtype)
    return rays, rec


def families(rt, hs, rays0, rec0, rng):
    """One batch of every family: (records, rays, beta, radiance on entry, family label per row)."""
    n_mat = hs.desc.contents.n_materials
    hits = np.flatnonzero(rec0["kind"] != rt.RT_HIT_MISS)
    assert len(hits) > 100
    xforms = sorted(set(rec0["inst_id"][rec0["inst_id"] != RT_NONE].tolist())) or [0]
    recs, rays, labels = [], [], []

    def take(label, k, rows=hits):
        idx = rng.choice(rows, k)
        r, y = rec0[idx].copy(), rays0[idx].copy()
        recs.append(r), rays.append(y), labels.extend([label] * k)
        return r, y

    def any_material(r):
        r["material"] = rng.integers(0, n_mat, len(r))
        r["kind"] = rng.choice([rt.RT_HIT_SURFACE, rt.RT_HIT_MEDIUM], len(r), p=[0.8, 0.2])

    for m in range(n_mat):  # material: every index of the table on both hit kinds
        for kind in (rt.RT_HIT_SURFACE, rt.RT_HIT_MEDIUM):
            r, _ = take("material", 6)
            r["material"], r["kind"] = m, kind
    big = [9.1e18, 9.2e18, 9.21e18, 9.22e18, float(np.nextafter(2.0 ** 63, 0.0)), 2.0 ** 63, 1e19, 1e300]
    specials = big + [-x for x in big] + [np.inf, -np.inf, np.nan]
    pts = list(getattr(hs, "_points", []))
    for x in specials:
        for a in range(3):
            p = rng.uniform(-3, 3, 3)
            p[a] = x
            pts.append(p)
        pts.append(np.full(3, x))
    for p in pts:  # p
        r, _ = take("p", 8)
        r["p"] = p
        any_material(r)
    s = 5e-324
    normals = [None, "away", 1e-3, 1e3, [0.0, 0.0, 0.0], [s, 0.0, 0.0], [1e-310, -1e-310, s], 1e200, [np.inf, 0.0, 0.0],
               [-np.inf, 1.0, np.inf], [np.nan, 0.0, 0.0], [0.0, np.nan, np.nan]]
    for nv in normals:  # normal, with inst_id RT_NONE, a Transform's id or an arbitrary value
        for inst in (RT_NONE, xforms[0], xforms[-1], 0xDEADBEEF, 7):
            r, y = take("normal", 6)
            any_material(r)
            if nv is None or nv == "away":
                d = y["direction"] / np.linalg.norm(y["direction"], axis=1)[:, None]
                r["normal"] = -d if nv is None else d
            elif np.ndim(nv) == 0:
                r["normal"] = r["normal"] * nv
            else:
                r["normal"] = nv
            r["inst_id"] = inst
    coords = sorted(set(edge_coords(9, 6)) | {0.0, 1e300, np.inf, -np.inf}, key=lambda x: (x, np.signbit(x)))
    coords += [-0.0, -1e-300, np.nan]
    for x in coords:  # u, v
        for which in ("u", "v", "uv"):
            r, _ = take("uv", 2)
            any_material(r)
            for f in which:
                r[f] = x
    for ff in (0, 1, 2, 0xFFFFFFFF):  # front_face, on every material
        r, _ = take("front_face", n_mat)
        any_material(r)
        r["material"] = np.arange(n_mat)
        r["front_face"] = ff
    dirs = [[1, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0], [0, 0, 1], [0, 0, -1], [-1, 0, 0.0], [-1, 0, -0.0], [-1, 1e-300, -0.0],
            [1e-17, 1, 0], [0, -1, 1e-17], [0, 0, 0], [s, 0, 0], [0, -s, s], [1e300, -1e300, 1e300], [np.inf, 0, 0], [1, np.inf, -np.inf],
            [np.nan, 1, 0], [1e-160, 1e-160, 0]]
    for dv in dirs:  # ray: miss directions
        r, y = take("miss direction", 4, np.arange(len(rec0)))
        r["kind"] = rt.RT_HIT_MISS
        y["direction"] = dv
    for dv in ([0.0, 0.0, 0.0], [np.nan, 0.0, 1.0], [-0.0, s, 0.0]):  # ray: degenerate directions on every material
        r, y = take("hit direction", n_mat)
        any_material(r)
        r["material"] = np.arange(n_mat)
        y["direction"] = dv
    for tv in (np.nan, np.inf, -np.inf, -0.0):  # ray: time
        _, y = take("time", 40, np.arange(len(rec0)))
        y["time"] = tv
    for kind in (3, 7, 0xFFFFFFFF):  # malformed records: a kind beyond RT_HIT_MEDIUM, a material beyond the table
        r, _ = take("malformed", 20, np.arange(len(rec0)))
        r["kind"] = kind
    for m in (n_mat, n_mat + 5, RT_NONE):
        r, _ = take("malformed", 20)
        r["material"] = m
    for _ in range(3):  # beta (below) on hits and misses
        take("beta", 100, np.arange(len(rec0)))
    take("plain", 400, np.arange(len(rec0)))
    recs, rays, labels = np.concatenate(recs), np.concatenate(rays), np.array(labels)
    n = len(recs)
    garbage = rng.uniform(size=n) < 0.5  # origins are not read by shading
    rays["origin"][garbage] = rng.choice([np.nan, np.inf, -1e300, 3.0, 0.0], (int(garbage.sum()), 3))
    beta = np.ones((n, 3))
    bv = np.array([1.0, 5e-324, 1e308, np.inf, np.nan, -0.0, -1.0, 0.0])
    sel = labels == "beta"
    beta[sel] = rng.choice(bv, (int(sel.sum()), 3))
    beta[~sel] = rng.uniform(0.05, 2.0, (int((~sel).sum()), 3))
    rad0 = np.where(rng.uniform(size=(n, 3)) < 0.6, 0.0, rng.choice(np.array([0.0, -0.0, np.nan, np.inf, -np.inf, 1.5, -2.25, 1e-300]), (n, 3)))
    rad0[rng.uniform(size=n) < 0.2] = rng.normal(size=3)
    return recs, rays, beta, rad0, labels


def garble_unread(rt, recs, rng):
    """t, prim_id and reserved to NaN or random bits; every field of a miss but its kind too."""
    g = recs.copy()
    n = len(g)
    raw = g.view(np.uint8).reshape(n, 96)
    g["t"] = np.where(rng.uniform(size=n) < 0.5, np.nan, rng.normal(size=n) * 1e300)
    g["prim_id"] = rng.integers(0, 2 ** 32, n, dtype=np.uint64).astype(np.uint32)
    g["reserved"] = rng.integers(0, 2 ** 32, n, dtype=np.uint64).astype(np.uint32)
    miss = g["kind"] == rt.RT_HIT_MISS
    kind = g["kind"].copy()
    raw[miss] = rng.integers(0, 256, (int(miss.sum()), 96), dtype=np.uint8)
    g["kind"] = kind
    return g


ADDRESSES = [(0, 0, None), (2 ** 64 - 1, -2, None), (0x9E3779B97F4A7C15, -1, None), (0, 4093, 4095), (2 ** 64 - 1, 4094, 4095)]


def batches_for(rt, orc, name, hs):
    """(name, hs, camera, seed, segment, records, rays, beta, radiance, labels, state) of scene `name` at every draw address."""
    rng = np.random.default_rng(sum(map(ord, name)))
    rays0, rec0 = base_records(rt, orc, name, hs, rng)
    recs, rays, beta, rad0, labels = families(rt, hs, rays0, rec0, rng)
    n = len(recs)
    state = np.full(n, rt.RT_PATH_ALIVE, np.uint8)
    inactive = rng.uniform(size=n) < 0.1
    state[inactive] = rng.choice(INACTIVE_STATES, int(inactive.sum()))
    state[~inactive] |= rng.choice(np.array([0, 0xFC], np.uint8), int((~inactive).sum()))  # other bits are ignored
    for seed, seg, depth in ADDRESSES:
        cam = rt.rt_camera.from_buffer_copy(hs.camera)
        if depth is not None:
            cam.max_depth = depth
        segment = seg if seg >= 0 else cam.max_depth + seg
        yield name, hs, cam, seed, segment, recs, rays, beta, rad0, labels, state


def batches(rt, orc):
    """batches_for every scene."""
    for name in sorted(SCENES):
        yield from batches_for(rt, orc, name, SCENES[name](rt))


def oracle_expectation(rt, osc, hs, cam, seed, segment, recs, rays, beta, rad0):
    """The oracle's shade_record and what rt_shade must leave: radiance, alive, error bit, next throughput (the rules of
    test_shade.test_against_the_oracle; the emission is added for the materials shade_hit adds it for)."""
    n = len(recs)
    ids3 = np.column_stack([np.arange(n), np.zeros(n), np.full(n, segment)]).astype(np.uint32)
    st = osc.shade_record(rays, recs, np.full(n, seed, np.uint64), ids3, camera=cam)
    n_mat = hs.desc.contents.n_materials
    miss = recs["kind"] == rt.RT_HIT_MISS
    valid_hit = (recs["kind"] <= rt.RT_HIT_MEDIUM) & ~miss & (recs["material"] < n_mat)
    emit = valid_hit & emitting(hs)[np.minimum(recs["material"], n_mat - 1)]
    with np.errstate(all="ignore"):
        c = np.where((miss & ~st["error"])[:, None], beta * st["background"], np.where(emit[:, None], beta * st["emission"], 0.0))
        nan_c = np.isnan(c).any(axis=1)
        acc = np.where((c != 0.0) & ~nan_c[:, None], c, 0.0)
        rad = np.where(acc != 0.0, rad0 + acc, rad0)
    nb = expected_beta(st, beta)
    alive = st["goes_on"] & ~st["error"] & (segment + 1 < cam.max_depth) & (nb != 0.0).any(axis=1)
    return st, dict(radiance=rad, alive=alive, error=st["error"] | nan_c, nbeta=nb, nan_c=nan_c, miss=miss)


# ---------------------------------------------------------------- CPU: the oracle
def test_shade_record_equals_shade_step(rt, orc):
    """shade_record on the records world.hit gives is the oracle's ray_step, bit for bit, over the scenes of test_segment_kat."""
    keys = ("background", "emission", "kind", "attenuation", "albedo_x_pscatter", "pdf_val", "o", "d", "time", "goes_on", "generated", "error", "fuzzed")
    for name in sorted(tsk.SCENES):
        hs = tsk.SCENES[name](rt)
        rng = np.random.default_rng(sum(map(ord, name)))
        osc = orc.OracleScene(hs)
        cam = hs.camera
        px = np.stack([rng.integers(0, cam.image_width, 300), rng.integers(0, cam.image_height, 300)], axis=1)
        rays = np.concatenate([orc.camera_rays(cam, 3, px, 0), tsk.edge_rays(rng, 100)])
        n = len(rays)
        for seed, seg in ((7, 0), (2 ** 64 - 1, 5)):
            rec = WorldHitOracle(hs).world_hit(rays, seed=seed, segment=seg).view(rt.rt_hit_record_dtype)
            ids3 = np.column_stack([np.arange(n), np.zeros(n), np.full(n, seg)]).astype(np.uint32)
            seeds = np.full(n, seed, np.uint64)
            want = osc.shade_step(rays, seeds, ids3)
            got = osc.shade_record(rays, rec, seeds, ids3)
            assert np.array_equal(got["hit"], want["hit"]), name
            for k in keys:
                a, b = np.ascontiguousarray(got[k]), np.ascontiguousarray(want[k])
                assert a.tobytes() == b.tobytes(), (name, k)


def panic_transform_scene(rt):
    """A Metal quad under a world Transform with a subnormal x scale: normal / scale is infinite, so the Transform's normal cannot be
    normalised (shapes.rs:107 panics).  A ray along +y at x = 0 hits it."""
    b = rt.Builder(5)
    quad = b.quad([-0.5, 1.5, -0.5], [1.0, -1.0, 0.0], [0.0, 0.0, 1.0], b.metal([0.9, 0.9, 0.9], 0.0))
    world = b.list([b.transform(quad, offset=[0.0, 0.0, 0.0], quat=[1.0, 0.0, 0.0, 0.0], scale=[1e-310, 1.0, 1.0])])
    hs = b.finish(world, width=8, spp=1, max_depth=4, background=b.solid(0.5, 0.5, 0.5))
    hs._builder = b
    return hs


def test_transform_normal_panic_is_an_error(rt, orc):
    """Known answer: the hit is found, its normal is NaN, and the step is an error (a Metal alone would end the path silently:
    reflect of a NaN normal cannot be normalised, scatter returns None)."""
    hs = panic_transform_scene(rt)
    osc = orc.OracleScene(hs)
    rays = tsk.make_rays([[0.0, -3.0, 0.0]], [[0.0, 1.0, 0.0]], [0.5])
    h = osc.world_hit([0.0, -3.0, 0.0], [0.0, 1.0, 0.0])
    assert h is not None and h["inst_id"] != RT_NONE and np.isnan(h["normal"][0]) and h["t"] == 4.0
    st = osc.shade_step(rays, [3], [[0, 0, 0]])
    assert st["hit"][0] == 1 and st["error"][0] and not st["goes_on"][0]
    # the same through shade_record: the Transform flag is inst_id with a non-finite normal; without inst_id no error
    rec = WorldHitOracle(hs).world_hit(rays).view(rt.rt_hit_record_dtype)
    assert rec["kind"][0] == rt.RT_HIT_SURFACE and rec["inst_id"][0] != RT_NONE and np.isnan(rec["normal"][0, 0])
    assert osc.shade_record(rays, rec, [3], [[0, 0, 0]])["error"][0]
    rec["inst_id"] = RT_NONE
    st = osc.shade_record(rays, rec, [3], [[0, 0, 0]])
    assert not st["error"][0] and not st["goes_on"][0]


def outcome_counts(rt, orc):
    """Per outcome, the rows of every batch that reach it (the oracle side of test_records_vs_oracle)."""
    counts = {}

    def add(k, v):
        counts[k] = counts.get(k, 0) + int(np.count_nonzero(v))

    cache = {}
    for name, hs, cam, seed, segment, recs, rays, beta, rad0, labels, state in batches(rt, orc):
        if name not in cache:
            cache.clear()
            cache[name] = orc.OracleScene(hs)
        osc = cache[name]
        st, w = oracle_expectation(rt, osc, hs, cam, seed, segment, recs, rays, beta, rad0)
        on = (state & rt.RT_PATH_ALIVE) != 0
        kind_of, _ = material_table(hs)
        n_mat = len(kind_of)
        has_lights = hs.desc.contents.lights_root != RT_NONE
        malformed = (recs["kind"] > 2) | ((recs["kind"] != 0) & (recs["material"] >= n_mat))
        hit = ~w["miss"] & ~malformed
        nrm = recs["normal"]
        with np.errstate(all="ignore"):
            un = nrm / np.sqrt((nrm * nrm).sum(axis=1))[:, None]
            ud = rays["direction"] / np.sqrt((rays["direction"] ** 2).sum(axis=1))[:, None]
        bad_normal = ~np.isfinite(un).all(axis=1)
        bad_dir = ~np.isfinite(ud).all(axis=1)
        xform = hit & (recs["inst_id"] != RT_NONE) & ~np.isfinite(nrm).all(axis=1)
        err = st["error"] & on
        pick = np.array([draw(orc, seed, i, 0, segment, RT_SLOT_MIXTURE)[0] for i in range(len(recs))])
        pdfk = np.isin(st["kind"], [SCATTER_COSINE, SCATTER_SPHERE, SCATTER_DISNEY])
        lit = pdfk & (pick >= 0.5) & has_lights
        next_set = (st["d"] != 0).any(axis=1)
        for m in range(n_mat):
            sel = on & hit & (recs["material"] == m)
            kname = MAT_NAMES[kind_of[m]]
            add(f"{kname} alive", sel & w["alive"])
            add(f"{kname} dead", sel & ~w["alive"] & ~w["error"])
            add(f"{kname} error", sel & w["error"])
        add("rule: malformed record", err & malformed)
        add("rule: Transform normal", err & xform)
        add("rule: unit_vector of the direction", err & hit & ~xform & bad_dir & ~st["generated"])
        add("rule: ONB", err & hit & ~xform & ~bad_dir & bad_normal & pdfk & ~st["generated"] & ~lit)
        add("rule: Disney derr", err & hit & ~xform & ~bad_dir & ~bad_normal & (st["kind"] == SCATTER_DISNEY) & ~lit & ~st["generated"])
        add("rule: lights_random", err & hit & ~xform & lit & ~st["generated"])
        add("rule: NaN light pdf", err & st["generated"] & np.isnan(st["pdf_val"]))
        add("rule: value0 == value1 == 0", err & st["generated"] & next_set & (st["pdf_val"] == 0.0) & has_lights)
        add("rule: pdf_val == 0", err & st["generated"] & next_set & (st["pdf_val"] == 0.0) & (not has_lights))
        add("rule: background without a unit direction", err & w["miss"])
        add("rule: NaN contribution", on & w["nan_c"])
        add("Disney None (stop 2)", on & hit & (st["kind"] == SCATTER_DISNEY) & ~st["generated"] & ~st["error"])
        add("infinite light pdf: zero throughput, cut", on & st["generated"] & ~st["error"] & np.isinf(st["pdf_val"]) & ~w["alive"])
    return counts


def test_families_reach_every_outcome(rt, orc):
    """The oracle side of the record families: each material kind alive, dead and in error, Disney's None, every error rule and the
    zero-throughput cut of an infinite light pdf, each at least a few dozen times."""
    counts = outcome_counts(rt, orc)
    print("\n" + "\n".join("%-48s %8d" % kv for kv in sorted(counts.items())))
    need = [f"{k} {o}" for k in MAT_NAMES for o in ("alive", "dead", "error")]
    need.remove("diffuse_light alive")  # (kept: DiffuseLight with an inner material)
    # a NaN light pdf needs an empty light list (0 / 0), which the scene compiler refuses (hits.rs:73); with a non-empty one no
    # input reaches it (a sphere light's NaN cos_theta_max returns 1 / (4 pi))
    need += [k for k in counts if k.startswith("rule:") and k != "rule: NaN light pdf"]
    need += ["Disney None (stop 2)", "infinite light pdf: zero throughput, cut"]
    low = {k: counts.get(k, 0) for k in need if counts.get(k, 0) < 30}
    assert not low, low
    assert counts.get("diffuse_light alive", 0) >= 30, counts


# ---------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(SCENES))
def test_records_vs_oracle(gpu, rt, orc, name):
    hs0 = SCENES[name](rt)
    sc, osc = rt.Scene(hs0), orc.OracleScene(hs0)
    seen = 0
    for bname, hs, cam, seed, segment, recs, rays, beta, rad0, labels, state in batches_for(rt, orc, name, hs0):
        n = len(recs)
        st, w = oracle_expectation(rt, osc, hs, cam, seed, segment, recs, rays, beta, rad0)
        grng = np.random.default_rng(seed % 1000 + segment)
        inactive = (state & rt.RT_PATH_ALIVE) == 0
        r, b, rad, s = rays.copy(), beta.copy(), rad0.copy(), state.copy()
        junk = []
        for a in (r, b, rad):
            v = a.view(np.uint8).reshape(n, -1)
            v[inactive] = grng.integers(0, 256, v[inactive].shape, dtype=np.uint8)
            junk.append(v[inactive].copy())
        stats = sc.shade(recs, r, b, rad, s, seed=seed, segment=segment, camera=cam)
        # inactive rows: untouched byte for byte
        for a, j in zip((r, b, rad), junk):
            assert a.view(np.uint8).reshape(n, -1)[inactive].tobytes() == j.tobytes(), name
        assert np.array_equal(s[inactive], state[inactive])
        on = ~inactive
        alive, err = (s & rt.RT_PATH_ALIVE) != 0, (s & rt.RT_PATH_ERROR) != 0
        assert ((s[on] & ~np.uint8(3)) == 0).all()
        where = f"{name}, seed {seed}, segment {segment} of {cam.max_depth}"
        bad = np.flatnonzero(on & (alive != w["alive"]))
        assert not len(bad), f"{where}: alive differs in {len(bad)} rows, first {bad[0]} ({labels[bad[0]]}): device {alive[bad[0]]}, " \
                             f"record {recs[bad[0]]}, ray {rays[bad[0]]}, beta {beta[bad[0]]}, oracle kind {st['kind'][bad[0]]} error {st['error'][bad[0]]}"
        bad = np.flatnonzero(on & (err != w["error"]))
        assert not len(bad), f"{where}: error bit differs in {len(bad)} rows, first {bad[0]} ({labels[bad[0]]}): device {err[bad[0]]}, " \
                             f"record {recs[bad[0]]}, ray {rays[bad[0]]}, beta {beta[bad[0]]}"
        assert stats.errors == int(err[on].sum()) and stats.segments == n
        mag = lambda v: np.max(np.abs(np.nan_to_num(v, nan=0.0, posinf=0.0, neginf=0.0)), axis=1, keepdims=True)  # noqa: E731
        miss = on & w["miss"]
        compare("records: radiance (hit, malformed)", rad[on & ~miss], w["radiance"][on & ~miss])
        compare("records: radiance (miss)", rad[miss], w["radiance"][miss], rel=REL, scale=mag(w["radiance"][miss]))
        go = on & alive
        compare("records: next origin", r["origin"][go], st["o"][go])
        compare("records: next time", r["time"][go], st["time"][go])
        exact_d = go & (st["kind"] == SCATTER_RAY) & ~st["fuzzed"]
        compare("records: next direction (ray, no fuzz)", r["direction"][exact_d], st["d"][exact_d])
        compare("records: next direction", r["direction"][go & ~exact_d], st["d"][go & ~exact_d], rel=REL, scale=mag(st["d"][go & ~exact_d]))
        ray = go & (st["kind"] == SCATTER_RAY)
        compare("records: next throughput (ray)", b[ray], w["nbeta"][ray])
        compare("records: next throughput (pdf)", b[go & ~ray], w["nbeta"][go & ~ray], rel=REL, scale=mag(w["nbeta"][go & ~ray]))
        stay = on & ~alive  # a path that ends leaves its ray and throughput as they were
        assert r[stay].tobytes() == rays[stay].tobytes() and b[stay].tobytes() == beta[stay].tobytes(), where
        # a second call, and a call on records whose unread fields are garbage: the same bits
        for rr in (recs, garble_unread(rt, recs, grng)):
            r2, b2, rad2, s2 = rays.copy(), beta.copy(), rad0.copy(), state.copy()
            for a, a2 in ((r, r2), (b, b2), (rad, rad2)):
                a2.view(np.uint8).reshape(n, -1)[inactive] = a.view(np.uint8).reshape(n, -1)[inactive]
            sc.shade(rr, r2, b2, rad2, s2, seed=seed, segment=segment, camera=cam)
            assert r2.tobytes() == r.tobytes() and b2.tobytes() == b.tobytes() and rad2.tobytes() == rad.tobytes() and s2.tobytes() == s.tobytes(), where
        seen += int(on.sum())
    assert seen > 10000


def test_unread_fields_are_not_read_by_the_oracle(rt, orc):
    """The oracle's record mapping reads what the header says rt_shade reads: garbage in t, prim_id, reserved and in the fields of a
    miss changes no output."""
    name = "room_four_solid"
    hs = SCENES[name](rt)
    osc = orc.OracleScene(hs)
    _, _, cam, seed, segment, recs, rays, beta, rad0, _, _ = next(batches_for(rt, orc, name, hs))
    n = len(recs)
    ids3 = np.column_stack([np.arange(n), np.zeros(n), np.full(n, segment)]).astype(np.uint32)
    a = osc.shade_record(rays, recs, np.full(n, seed, np.uint64), ids3, camera=cam)
    b = osc.shade_record(rays, garble_unread(rt, recs, np.random.default_rng(3)), np.full(n, seed, np.uint64), ids3, camera=cam)
    for k in a:
        assert np.ascontiguousarray(a[k]).tobytes() == np.ascontiguousarray(b[k]).tobytes(), k


# ---------------------------------------------------------------- the batch limit comes first
@pytest.mark.gpu
def test_oversized_batches_are_refused_before_any_allocation(gpu, rt):
    """n = 2^32 - 15 with one-element buffers: RT_ERR_INVALID naming the batch size, before anything is allocated or copied (the
    buffers are never dereferenced)."""
    L = rt.product_lib()
    b = rt.Builder(1)
    hs = b.finish(b.list([b.sphere([0, 0, 0], 1.0, b.lambertian(b.solid(0.5, 0.5, 0.5)))]), width=8, spp=1)
    sc = rt.Scene(hs)
    cam = rt.rt_camera.from_buffer_copy(hs.camera)
    n = 2 ** 32 - 15
    ray = rt.make_rays([[0.0, 0.0, 5.0]], [[0.0, 0.0, -1.0]])
    rec = np.zeros(1, rt.rt_hit_record_dtype)
    one, tmax, st8 = np.zeros(96), np.full(1, np.inf), np.ones(1, np.uint8)
    p = lambda a: a.ctypes.data  # noqa: E731
    st = rt.rt_stats()
    calls = {
        "rt_closest_hit": lambda: L.rt_closest_hit(sc.h, p(ray), n, 1e-8, np.inf, 0, p(one), C.byref(st)),
        "rt_closest_hit_device": lambda: L.rt_closest_hit_device(sc.h, p(ray), n, 1e-8, np.inf, 0, p(one), None, C.byref(st)),
        "rt_occluded": lambda: L.rt_occluded(sc.h, p(ray), p(tmax), n, 1e-8, np.inf, 0, p(st8), C.byref(st)),
        "rt_occluded_device": lambda: L.rt_occluded_device(sc.h, p(ray), p(tmax), n, 1e-8, np.inf, 0, p(st8), None, C.byref(st)),
        "rt_transmittance": lambda: L.rt_transmittance(sc.h, p(ray), p(tmax), n, 1e-8, np.inf, 0, p(one), C.byref(st)),
        "rt_transmittance_device": lambda: L.rt_transmittance_device(sc.h, p(ray), p(tmax), n, 1e-8, np.inf, 0, p(one), None, C.byref(st)),
        "rt_world_hit": lambda: L.rt_world_hit(sc.h, p(ray), p(tmax), n, 1e-8, np.inf, 1, 0, 0, p(rec), C.byref(st)),
        "rt_world_hit_device": lambda: L.rt_world_hit_device(sc.h, p(ray), p(tmax), n, 1e-8, np.inf, 1, 0, 0, p(rec), None, C.byref(st)),
        "rt_shade": lambda: L.rt_shade(sc.h, C.byref(cam), p(rec), n, 1, 0, 0, p(ray), p(one), p(one), p(st8), C.byref(st)),
        "rt_shade_device": lambda: L.rt_shade_device(sc.h, C.byref(cam), p(rec), n, 1, 0, 0, p(ray), p(one), p(one), p(st8), None, C.byref(st)),
    }
    for fname, call in calls.items():
        assert call() == -1, fname  # RT_ERR_INVALID
        assert "2^32 - 16" in L.rt_last_error().decode(), (fname, L.rt_last_error())
    assert L.rt_shade(sc.h, C.byref(cam), p(rec), 2 ** 32 - 16, 1, cam.max_depth, 0, p(ray), p(one), p(one), p(st8), None) == -1
    assert "max_depth" in L.rt_last_error().decode()  # at the limit the other refusals still come first
