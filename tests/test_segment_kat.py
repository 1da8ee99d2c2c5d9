"""One path segment at a time against the oracle: every shade class and its lean twin, camera rays, and path ids at their limits.

The oracle's ray_color is one level (ray_step, oracle/orc.py OracleScene.shade_step) plus the recursion.  Real segments are drawn by
following paths through that step; each segment - the ray, the throughput, the addressed draws (seed; pixel, sample, segment), the
hit the oracle found - is then shaded on the device by the product's own segment code (csrc/shade_step.cuh through
tests/device_kat.cu): shade_one of the hit's compiled shade class, shade_one<SC_OTHER>, and the lean twins where the scene has them.

Checks per segment:
- the compiled class and every lean twin give exactly the bits of shade_one<SC_OTHER> (a difference is a routing or lean bug);
- against the oracle, expected values computed in numpy in the device's association order: contribution beta * emission (or beta *
  background), next throughput beta * attenuation or beta * (axp / pdf_val); alive, the error count and NaN patterns identical;
  next-ray origins and times bit-equal (no transcendental function reaches them), directions and throughputs within REL of their
  row's magnitude (random_unit_vector, random_cosine_direction, sphere lights and Disney go through sin, cos, acos, pow).
Path ids run up to the packing limits (pixel 2^28 - 1, sample 2^24 - 1, segment 4094) and max_depth up to 4095.
"""
import numpy as np
import pytest

import device_kat as dk
from scenes_util import disney_scene, materials_scene, obj_mesh_scene, random_graph_scene
from test_gpu_parity import _walk_scene, image_close
from test_shade_lean import lean_scene as shade_lean_scene
from test_walk_lean import lean_scene as walk_lean_scene

REL = 1e-13
RT_NONE = 0xFFFFFFFF
HIT_MISS, HIT_SURFACE, HIT_MEDIUM = 0, 1, 2
SC_MISS, SC_DIFFUSE, SC_TEXTURED, SC_ISOTROPIC, SC_METAL, SC_DIELECTRIC, SC_EMISSIVE, SC_DISNEY, SC_OTHER, SC_WALK = range(10)
CLASS_NAMES = ["miss", "diffuse", "textured", "isotropic", "metal", "dielectric", "emissive", "disney", "other"]
SCATTER_NONE, SCATTER_COSINE, SCATTER_SPHERE, SCATTER_RAY, SCATTER_DISNEY = range(5)
MEDIUM_THICK = 1
PIXEL_MAX, SAMPLE_MAX, SEGMENT_MAX = (1 << 28) - 1, (1 << 24) - 1, (1 << 12) - 1

STATS = {}   # output: [values compared, bit-equal, largest relative difference]
COUNTS = {}  # instantiation: segments it shaded


@pytest.fixture(scope="module", autouse=True)
def report():
    yield
    if STATS:
        print("\n%-34s %10s %10s %12s" % ("output", "values", "bit-equal", "max rel"))
        for k, (n, eq, mx) in sorted(STATS.items()):
            print("%-34s %10d %10d %12.3e" % (k, n, eq, mx))
    if COUNTS:
        print("\n%-34s %10s" % ("instantiation", "segments"))
        for k, n in sorted(COUNTS.items()):
            print("%-34s %10d" % (k, n))


def compare(name, got, want, rel=0.0, scale=None):
    """got == want bit for bit where rel == 0; else |got - want| <= rel * max(|want|, scale).  scale: per value (broadcast), the
    magnitude of the vector the value belongs to.  NaN and infinity patterns must agree exactly."""
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape
    sc = np.zeros_like(want) if scale is None else np.broadcast_to(np.asarray(scale, dtype=np.float64), want.shape)
    got, want, sc = got.ravel(), want.ravel(), sc.ravel()
    gn, wn = np.isnan(got), np.isnan(want)
    assert np.array_equal(gn, wn), f"{name}: NaN pattern differs at {np.flatnonzero(gn != wn)[:8]}"
    bits = (got.view(np.int64) == want.view(np.int64)) | (gn & wn)
    fin = np.isfinite(want) & ~bits
    assert np.array_equal(np.isinf(got), np.isinf(want)) and np.all(got[np.isinf(want)] == want[np.isinf(want)]), f"{name}: infinities differ"
    diff = np.abs(got[fin] - want[fin])
    s = np.maximum(np.maximum(np.abs(want[fin]), sc[fin]), np.finfo(np.float64).tiny)
    relerr = diff / s
    st = STATS.setdefault(name, [0, 0, 0.0])
    st[0] += got.size
    st[1] += int(bits.sum())
    st[2] = max(st[2], float(relerr.max()) if relerr.size else 0.0)
    bad = diff > rel * s
    if bad.any():
        k = np.flatnonzero(fin)[np.flatnonzero(bad)[0]]
        pytest.fail(f"{name}: {int(bad.sum())} of {got.size} values differ beyond the bound; first at flat index {k}: {got[k]!r} vs {want[k]!r}")


def same_bits(name, a, b, rows):
    """Every output of two device runs bit for bit (routing and lean twins)."""
    for key in ("o", "d", "time", "nbeta", "contribution"):
        x, y = np.ascontiguousarray(a[key][rows]), np.ascontiguousarray(b[key][rows])
        bad = x.view(np.int64) != y.view(np.int64)
        if bad.any():
            r = np.flatnonzero(bad.reshape(len(x), -1).any(axis=1))[0]
            pytest.fail(f"{name}: {key} differs from shade_one<SC_OTHER> in {int(bad.reshape(len(x), -1).any(axis=1).sum())} segments; "
                        f"first: {x[r]!r} vs {y[r]!r}")
    for key in ("alive", "errors"):
        assert np.array_equal(a[key][rows], b[key][rows]), f"{name}: {key} differs from shade_one<SC_OTHER>"


# ---------------------------------------------------------------- segments drawn from the oracle
def make_rays(o, d, time):
    rays = np.zeros(len(o), dtype=dk.RAY_DTYPE)
    rays["origin"], rays["direction"], rays["time"] = o, d, time
    return rays


def expected_beta(step, beta):
    """The next throughput in the device's association order: beta * attenuation, or beta * (axp / pdf_val) with x / s = (1 / s) x."""
    with np.errstate(all="ignore"):
        pdf = beta * ((1.0 / step["pdf_val"])[:, None] * step["albedo_x_pscatter"])
        return np.where((step["kind"] == SCATTER_RAY)[:, None], beta * step["attenuation"], pdf)


def walk_segments(orc, osc, hs, rng, n_paths, extra_rays=None, id_limits=True):
    """Segments of n_paths real paths, followed level by level through the oracle's step.  The first rays are camera rays (and
    extra_rays); a quarter of the paths is addressed at the packing limits - pixel 2^28 - 1 - k, sample 2^24 - 1, segments ending
    at 4094 - and every path ends at its own max_depth, so the last segments sit at max_depth - 2 and max_depth - 1."""
    cam = hs.camera
    px = np.stack([rng.integers(0, cam.image_width, n_paths), rng.integers(0, cam.image_height, n_paths)], axis=1)
    sidx = rng.integers(0, cam.sqrt_spp ** 2, n_paths)
    seeds = rng.integers(0, 2 ** 63, n_paths, dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, n_paths, dtype=np.uint64)
    rays = np.concatenate([orc.camera_rays(cam, int(seeds[k]), px[k:k + 1], int(sidx[k])) for k in range(n_paths)])
    pixel = (px[:, 1] * cam.image_width + px[:, 0]).astype(np.uint32)
    seg0 = np.zeros(n_paths, np.uint32)
    depth = np.full(n_paths, cam.max_depth, np.uint32)
    if extra_rays is not None:
        m = len(extra_rays)
        rays = np.concatenate([rays, extra_rays])
        pixel = np.concatenate([pixel, rng.integers(0, PIXEL_MAX, m).astype(np.uint32)])
        sidx = np.concatenate([sidx, rng.integers(0, SAMPLE_MAX, m)])
        seeds = np.concatenate([seeds, rng.integers(0, 2 ** 63, m, dtype=np.uint64)])
        seg0 = np.concatenate([seg0, np.zeros(m, np.uint32)])
        depth = np.concatenate([depth, np.full(m, cam.max_depth, np.uint32)])
    n = len(rays)
    sidx = sidx.astype(np.uint32)
    if id_limits:
        lim = rng.uniform(size=n) < 0.25
        pixel[lim] = PIXEL_MAX - rng.integers(0, 3, int(lim.sum())).astype(np.uint32)
        sidx[lim] = SAMPLE_MAX
        seg0[lim] = SEGMENT_MAX - depth[lim]  # the last segment of these paths is 4094 = max_depth - 1
        depth[lim] = SEGMENT_MAX
    # some paths end early: max_depth 1, 2 or 3 above their first segment
    short = rng.uniform(size=n) < 0.15
    depth[short] = seg0[short] + rng.integers(1, 4, int(short.sum())).astype(np.uint32)
    beta = np.ones((n, 3))
    segs = []
    seg = seg0.copy()
    live = np.arange(n)
    while len(live):
        ids3 = np.column_stack([pixel[live], sidx[live], seg[live]])
        step = osc.shade_step(rays[live], seeds[live], ids3)
        segs.append(dict(rays=rays[live].copy(), beta=beta[live].copy(), seeds=seeds[live].copy(), ids3=ids3, max_depth=depth[live].copy(), step=step))
        nb = expected_beta(step, beta[live])
        go = step["goes_on"] & ~step["error"] & (seg[live] + 1 < depth[live]) & (nb != 0.0).any(axis=1)
        nxt = live[go]
        rays[nxt] = make_rays(step["o"][go], step["d"][go], step["time"][go])
        beta[nxt] = nb[go]
        seg[nxt] += 1
        live = nxt
    out = {k: np.concatenate([s[k] for s in segs]) for k in ("rays", "beta", "seeds", "ids3", "max_depth")}
    out["step"] = {k: np.concatenate([s["step"][k] for s in segs]) for k in segs[0]["step"]}
    return out


def device_inputs(ds, segs):
    """The oracle's hit as the device's shade stage sees it: device primitive or medium index, hit kind, t; and the class byte."""
    st = segs["step"]
    n = len(st["hit"])
    prim = np.full(n, RT_NONE, np.uint32)
    kind = np.where(st["hit"] == 2, HIT_MEDIUM, np.where(st["hit"] == 1, HIT_SURFACE, HIT_MISS)).astype(np.uint32)
    surf, med = st["hit"] == 1, st["hit"] == 2
    prim[surf] = ds.prim_of_object[st["object"][surf]]
    assert (prim[surf] != RT_NONE).all()
    medium_of_object = {int(o): m for m, o in enumerate(ds.medium_object)}
    prim[med] = [medium_of_object[int(o)] for o in st["object"][med]]
    cls = np.full(n, SC_MISS, np.uint32)
    cls[surf] = ds.prim_class[prim[surf]]
    cls[med] = np.where(ds.medium_flags[prim[med]] & MEDIUM_THICK, SC_WALK, SC_ISOTROPIC)
    ids6 = np.column_stack([segs["ids3"], prim, kind, segs["max_depth"]]).astype(np.uint32)
    t = np.where(st["hit"] > 0, st["t"], np.inf)
    return ids6, t, cls


def check_against_oracle(name, got, segs, libm_background=False):
    """libm_background: the scene's background lookup goes through acos / atan2 (image) or sin (noise)."""
    st, beta = segs["step"], segs["beta"]
    seg, max_depth = segs["ids3"][:, 2], segs["max_depth"]
    with np.errstate(all="ignore"):
        c = beta * np.where((st["hit"] == 0)[:, None], st["background"], st["emission"])
    nan_c = np.isnan(c).any(axis=1)
    miss_error = (st["hit"] == 0) & st["error"]
    want_acc = np.where((c != 0.0) & ~nan_c[:, None] & ~miss_error[:, None], c, 0.0)
    want_err = (nan_c & ~miss_error).astype(np.int64) + st["error"].astype(np.int64)
    nb = expected_beta(st, beta)
    want_alive = st["goes_on"] & ~st["error"] & (seg + 1 < max_depth) & (nb != 0.0).any(axis=1)
    bad = np.flatnonzero(got["alive"] != want_alive)
    assert not len(bad), f"{name}: alive differs in {len(bad)} segments, first {bad[0]}: device {got['alive'][bad[0]]}, oracle hit {st['hit'][bad[0]]} " \
                         f"kind {st['kind'][bad[0]]} error {st['error'][bad[0]]} goes_on {st['goes_on'][bad[0]]}"
    bad = np.flatnonzero(got["errors"] != want_err)
    assert not len(bad), f"{name}: error count differs in {len(bad)} segments, first {bad[0]}: {got['errors'][bad[0]]} vs {want_err[bad[0]]}"
    mag = lambda v: np.max(np.abs(v), axis=1, keepdims=True)
    # emission (solid, checker and image-alpha Mix textures on planar uv) and solid / gradient / checker backgrounds: bit for bit
    libm = (st["hit"] == 0) & libm_background
    compare("contribution", got["contribution"][~libm], want_acc[~libm])
    compare("contribution (image / noise background)", got["contribution"][libm], want_acc[libm], rel=REL, scale=mag(want_acc[libm]))
    # a path that goes on: its next ray and throughput (the scatter kinds that generate one, also at the depth limit).  A
    # ScatterRecord::Ray multiplies beta by a constant colour or a solid texture and, but for a Metal's fuzz, builds its direction
    # with +, -, *, / and sqrt: bit for bit.  The pdf kinds' directions and axp / pdf_val go through sin, cos, acos or pow.
    on = st["goes_on"] & ~st["error"]
    ray = on & (st["kind"] == SCATTER_RAY)
    exact_d = ray & ~st["fuzzed"]
    pdf = on & (st["kind"] != SCATTER_RAY)
    compare("next origin", got["o"][on], st["o"][on])
    compare("next time", got["time"][on], st["time"][on])
    compare("next direction (ray, no fuzz)", got["d"][exact_d], st["d"][exact_d])
    compare("next direction (fuzz, pdf)", got["d"][on & ~exact_d], st["d"][on & ~exact_d], rel=REL, scale=mag(st["d"][on & ~exact_d]))
    compare("next throughput (ray)", got["nbeta"][ray], nb[ray])
    compare("next throughput (pdf)", got["nbeta"][pdf], nb[pdf], rel=REL, scale=mag(nb[pdf]))
    for k in (SCATTER_NONE, SCATTER_COSINE, SCATTER_SPHERE, SCATTER_RAY, SCATTER_DISNEY):
        COUNTS["oracle scatter kind %d" % k] = COUNTS.get("oracle scatter kind %d" % k, 0) + int(((st["kind"] == k) & (st["hit"] > 0)).sum())


def instantiations(ds, cls, ids6):
    """[(label, class, lean, rows)]: shade_one<SC_OTHER> on every segment, the compiled class of every segment (SC_WALK scatter
    points: SC_ISOTROPIC, as the generic k_walk shades them), and the lean twins where the scene has them."""
    out = [("shade_one<other>", SC_OTHER, 0, np.arange(len(cls)))]
    for c in range(SC_OTHER):
        rows = np.flatnonzero((cls == c) | ((c == SC_ISOTROPIC) & (cls == SC_WALK)))
        if not len(rows):
            continue
        out.append((f"shade_one<{CLASS_NAMES[c]}>", c, 0, rows))
        if c in (SC_DIFFUSE, SC_TEXTURED) and ds.shade_lean_mask >> c & 1:
            out.append((f"shade_one<{CLASS_NAMES[c]}, lean>", c, 1, rows))
        if c == SC_ISOTROPIC and ds.shade_lean_mask >> SC_ISOTROPIC & 1:
            out.append(("lean_isotropic_scatter(ShadeLean)", c, 1, rows[cls[rows] == SC_ISOTROPIC]))
        if c == SC_ISOTROPIC and ds.has_walk_lean:
            out.append(("lean_isotropic_scatter(WalkLean)", c, 2, rows[(cls[rows] == SC_WALK) & (ids6[rows, 3] == ds.walk_thick)]))
    return [x for x in out if len(x[3])]


def run_segments(ds, hs, segs, name, libm_background=False):
    """The device instantiations on every segment: routing (compiled class == SC_OTHER == lean twin, bit for bit), then the oracle.
    Returns {instantiation: [segments, segments that counted an error]}."""
    ids6, t, cls = device_inputs(ds, segs)
    rays, beta, seeds = segs["rays"], segs["beta"], segs["seeds"]
    cam = hs.camera
    other = ds.shade_step(cam, SC_OTHER, 0, rays, beta, t, ids6, seeds)
    check_against_oracle(name, other, segs, libm_background)
    seen = {}
    for label, c, lean, r in instantiations(ds, cls, ids6):
        got = other if c == SC_OTHER else ds.shade_step(cam, c, lean, rays[r], beta[r], t[r], ids6[r], seeds[r])
        ref = {k: v[r] for k, v in other.items()}
        if lean != 0 and c == SC_ISOTROPIC:
            # lean_isotropic_scatter writes nothing when it ends a path with an error; shade_one leaves the ray and beta
            same_bits(f"{name}: {label}", got, ref, got["alive"] | (got["errors"] == 0))
            assert np.array_equal(got["alive"], ref["alive"]) and np.array_equal(got["errors"], ref["errors"]), f"{name}: {label}"
        else:
            same_bits(f"{name}: {label}", got, ref, slice(None))
        seen[label] = [len(r), int((got["errors"] > 0).sum())]
        COUNTS[label] = COUNTS.get(label, 0) + len(r)
        COUNTS[label + " errors"] = COUNTS.get(label + " errors", 0) + seen[label][1]
    return seen


# ---------------------------------------------------------------- scenes
def flat_four_scene(rt, lights="four", background="solid", width=32, spp=16):
    """The edge families in one room: a flat list of exactly four lights (lights="four"), none (lights="none") or a nested list;
    Mix three deep and an image-alpha Mix, Portal, Transparent, a DiffuseLight around a material, a zero-albedo Lambertian, a glass
    ball (total internal reflection from inside) and a fuzz-0 mirror; the background of the given kind."""
    rng = np.random.default_rng(17)
    b = rt.Builder(17)
    white, red = b.lambertian(b.solid(0.8, 0.8, 0.8)), b.lambertian(b.solid(0.8, 0.2, 0.1))
    alpha = rng.uniform(0, 1, (8, 8, 4)).astype(np.float32)
    alpha[..., 3] = rng.uniform(0, 1, (8, 8)) > 0.5
    glass = b.dielectric(b.solid(1, 1, 1), 1.5)
    mirror = b.metal([0.9, 0.9, 0.9], 0.0)
    mix3 = b.mix(b.mix(b.mix(white, mirror, 0.3), glass, 0.6), b.mix(red, b.transparent(), 0.5), 0.45)
    mats = [mix3, b.mix_image(b.transparent(), red, b.image(alpha)),
            b.portal([0.9, 0.95, 1.0], [0.0, 0.0, -3.0], b.quat_axis_angle([0, 1, 0], 15.0)), b.transparent(),
            b.diffuse_light(b.solid(0.6, 0.5, 0.4), inner=b.metal([0.8, 0.7, 0.6], 0.2)), b.lambertian(b.solid(0, 0, 0)), glass, mirror,
            b.diffuse_light(b.solid(0.3, 0.3, 0.3), inner=b.mix(white, glass, 0.5))]
    objs = []
    for k, m in enumerate(mats):
        x, y = (k % 3) * 2.4 - 2.4, (k // 3) * 2.2 - 1.8
        objs.append(b.sphere([x, y, 0], 0.95, m) if k % 2 == 0 else b.quad([x - 0.9, y - 0.9, 0.2], [1.8, 0, 0], [0, 1.8, 0.3], m))
    lamp = b.diffuse_light(b.solid(7, 7, 7))
    e = b.empty()
    spots = [([-3.0, 4.0, 1.0], 0.3), ([3.0, 4.0, 1.0], 0.4), ([0.0, 4.5, -2.0], 0.25)]
    things = [b.quad([-8, -3.5, -8], [16, 0, 0], [0, 0, 16], white), b.quad([-1.5, 5, -1.5], [3, 0, 0], [0, 0, 3], lamp)]
    things += [b.sphere(c, r, lamp) for c, r in spots] + objs
    light_objs = [b.quad([-1.5, 5, -1.5], [3, 0, 0], [0, 0, 3], e)] + [b.sphere(c, r, e) for c, r in spots]
    if lights == "four":
        lt = b.list(light_objs)
    elif lights == "nested":
        lt = b.list([light_objs[0], b.list(light_objs[1:3]), light_objs[3]])
    else:
        lt = rt.RT_NONE
    bg = {"solid": lambda: b.solid(0.4, 0.5, 0.7), "gradient": lambda: b.gradient([1, 1, 1], [0.3, 0.5, 0.9]),
          "image": lambda: b.image(rng.uniform(0, 2, (16, 32, 4)).astype(np.float32), linear_format=True),
          "checker": lambda: b.checker(0.3, b.solid(0.9, 0.9, 0.9), b.solid(0.2, 0.2, 0.2)), "noise": lambda: b.noise(1.5)}[background]()
    hs = b.finish(b.list([b.bvh(things)]), lt, width=width, spp=spp, max_depth=12, vfov=50, look_from=(0, 1, 10), look_at=(0, 0, 0), background=bg)
    hs._builder = b
    return hs


def edge_rays(rng, n):
    """Rays from inside the glass ball (total internal reflection), rays grazing the spheres' surfaces, rays out of the room."""
    c = np.array([-2.4, 2.6, 0.0])  # the glass ball, k = 6
    u = rng.normal(size=(n, 3))
    u /= np.linalg.norm(u, axis=1)[:, None]
    inside = make_rays(c + 0.3 * u, rng.normal(size=(n, 3)), rng.uniform(0, 1, n))
    # grazing: tangent to the glass ball, offset by a few ulps of the radius
    t = np.cross(u, rng.normal(size=(n, 3)))
    t /= np.linalg.norm(t, axis=1)[:, None]
    r = 0.95 * (1.0 - rng.integers(-4, 4, n) * 2.0 ** -52)
    graze = make_rays(c + r[:, None] * u - 3.0 * t, t, rng.uniform(0, 1, n))
    out = make_rays(rng.uniform(-1, 1, (n, 3)), rng.normal(size=(n, 3)), rng.uniform(0, 1, n))
    return np.concatenate([inside, graze, out])


LIBM_BACKGROUND = {"edges_no_lights_image", "edges_four_noise"}  # the others' backgrounds are solid, gradient or checker
SCENES = {
    "random_graph_media": lambda rt: random_graph_scene(rt, 11, n_prims=72, with_media=True, width=32, spp=4, depth=8),
    "no_lights_media": lambda rt: random_graph_scene(rt, 5, n_prims=48, with_media=True, with_lights=False, width=24, spp=4, depth=8),
    "materials": materials_scene,
    "disney": lambda rt: disney_scene(rt),
    "obj_mesh": lambda rt: obj_mesh_scene(rt),
    "walk_surfaces_inside": lambda rt: _walk_scene(rt, "surfaces_inside"),
    "walk_moving_transformed": lambda rt: _walk_scene(rt, "moving_transformed"),
    "shade_lean_book2": lambda rt: shade_lean_scene(rt, "book2"),
    "shade_lean_checker_lamp": lambda rt: shade_lean_scene(rt, "checker_lamp"),
    "shade_lean_nested_lights": lambda rt: shade_lean_scene(rt, "nested_lights"),
    "walk_lean_two_lights": lambda rt: walk_lean_scene(rt, "two_lights"),
    "edges_four_lights": lambda rt: flat_four_scene(rt, "four", "solid"),
    "edges_nested_gradient": lambda rt: flat_four_scene(rt, "nested", "gradient"),
    "edges_no_lights_image": lambda rt: flat_four_scene(rt, "none", "image"),
    "edges_four_checker": lambda rt: flat_four_scene(rt, "four", "checker"),
    "edges_four_noise": lambda rt: flat_four_scene(rt, "four", "noise"),
}


def test_oracle_step_composes_to_the_render(rt, orc):
    """The oracle hook is ray_color's own step: composing the levels of every path reproduces orc.render bit for bit."""
    for name in ("random_graph_media", "materials", "edges_four_lights", "obj_mesh"):
        hs = SCENES[name](rt)
        cam = hs.camera
        cam.image_width, cam.image_height = 8, 8
        osc = orc.OracleScene(hs)
        ref, _ = osc.render(camera=cam, seed=3, sample_begin=5, sample_end=6)
        px = np.array([(i, j) for j in range(8) for i in range(8)])
        rays = orc.camera_rays(cam, 3, px, 5)
        ids = np.column_stack([px[:, 1] * 8 + px[:, 0], np.full(64, 5), np.zeros(64)]).astype(np.uint32)
        seeds = np.full(64, 3, np.uint64)
        levels, live = [], np.arange(64)
        while len(live) and len(levels) < cam.max_depth:
            st = osc.shade_step(rays[live], seeds[live], ids[live])
            levels.append((live, st))
            go = st["goes_on"] & ~st["error"]
            rays[live[go]] = make_rays(st["o"][go], st["d"][go], st["time"][go])
            ids[live[go], 2] += 1
            live = live[go]
        color, error = np.zeros((64, 3)), np.zeros(64, bool)
        for live, st in reversed(levels):  # ray_color from the deepest level up, in its association order
            L = color[live]
            with np.errstate(all="ignore"):
                go = st["goes_on"] & ~st["error"]
                scat = np.where((st["kind"] == SCATTER_RAY)[:, None], st["attenuation"] * L, (st["albedo_x_pscatter"] * L) * (1.0 / st["pdf_val"])[:, None])
                ret = np.where(go[:, None], st["emission"] + scat, np.where((st["kind"] == SCATTER_NONE)[:, None], st["emission"], st["emission"] + 0.0))
                ret = np.where((st["hit"] == 0)[:, None], st["background"], ret)
            error[live] |= st["error"] | (go & np.isnan(ret).any(axis=1))
            color[live] = np.where(st["error"][:, None], 0.0, ret)
        want = np.where(error[:, None], 0.0, 0.0 + color) * cam.pixel_sample_scale
        assert np.array_equal(want.reshape(8, 8, 3).view(np.int64), ref.view(np.int64)), name


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(SCENES))
def test_segments_vs_oracle_and_routing(gpu, rt, orc, name):
    hs = SCENES[name](rt)
    rng = np.random.default_rng(sum(map(ord, name)))
    osc, ds = orc.OracleScene(hs), dk.DeviceScene(hs)
    extra = edge_rays(rng, 1500) if name.startswith("edges") else None
    segs = walk_segments(orc, osc, hs, rng, 6000, extra)
    seen = run_segments(ds, hs, segs, name, name in LIBM_BACKGROUND)
    st = segs["step"]
    assert (st["hit"] == 0).any() and (st["hit"] == 1).any()
    if name.startswith("edges"):
        assert seen["shade_one<other>"][0] - sum(n for k, (n, _) in seen.items() if k != "shade_one<other>" and "lean" not in k) > 1000


@pytest.mark.gpu
def test_every_instantiation_saw_thousands_of_segments(gpu, rt, orc):
    """The segments test_segments_vs_oracle_and_routing draws, counted per instantiation (the same seeds, no shading)."""
    counts = {}
    for name in sorted(SCENES):
        hs = SCENES[name](rt)
        rng = np.random.default_rng(sum(map(ord, name)))
        osc, ds = orc.OracleScene(hs), dk.DeviceScene(hs)
        extra = edge_rays(rng, 1500) if name.startswith("edges") else None
        segs = walk_segments(orc, osc, hs, rng, 6000, extra)
        ids6, _, cls = device_inputs(ds, segs)
        for label, _, _, rows in instantiations(ds, cls, ids6):
            counts[label] = counts.get(label, 0) + len(rows)
    for c in CLASS_NAMES:
        assert counts.get(f"shade_one<{c}>", 0) >= 2000, (c, counts)
    for label in ("shade_one<diffuse, lean>", "shade_one<textured, lean>", "lean_isotropic_scatter(ShadeLean)", "lean_isotropic_scatter(WalkLean)"):
        assert counts.get(label, 0) >= 2000, (label, counts)


# ---------------------------------------------------------------- the panic and error rules
def panic_scene(rt, lean=True):
    """Every error rule of a segment, in one room.  lean: the light list is flat (the lean kernels' LeanLights), else nested (with a
    third light).
    - pdf.rs:105-109 (value0 == value1 == 0): shelves in the lamp's plane y = 4 - a Lambertian, a checker Lambertian, a Mix - where
      a direction sampled towards the lamp lies in the plane;
    - hits.rs:64 (a NaN light pdf): a sphere light of radius 1.2 around a thin fog, a thick medium and two small balls - from inside
      it the sphere's pdf is NaN (cos_theta_max = sqrt(1 - r^2 / d^2));
    - camera.rs:323 (NaN radiance): a light whose colour is NaN;
    - a zero direction: a Portal whose quaternion is zero sends the path on with direction 0, whose miss has no background."""
    b = rt.Builder(29)
    e = b.empty()
    white = b.lambertian(b.solid(0.7, 0.7, 0.7))
    checker = b.lambertian(b.checker(0.5, b.solid(0.3, 0.5, 0.9), b.solid(0.9, 0.5, 0.3)))
    shelf = lambda x, z, m: b.quad([x, 4, z], [3, 0, 0], [0, 0, 3], m)
    things = [shelf(-1.5, -1.5, b.diffuse_light(b.solid(12, 12, 12))), shelf(2, -1.5, white), shelf(-5, -1.5, checker),
              shelf(-1.5, 2, b.mix(white, checker, 0.5)), shelf(-1.5, -5, b.diffuse_light(b.solid(float("nan"), 1.0, 1.0))),
              b.quad([-8, -3, -8], [16, 0, 0], [0, 0, 16], white),
              b.quad([-2, -3, -6], [4, 0, 0], [0, 5, 0], b.portal([1, 1, 1], [0, 0, 0], [0, 0, 0, 0])),
              b.medium(b.sphere([0, 0, 0], 0.9, e), 0.3, b.solid(0.9, 0.9, 0.9)),
              b.medium(b.sphere([0, 0, 0], 0.4, e), 6.0, b.solid(0.3, 0.5, 0.9)),
              b.sphere([0.75, 0, 0], 0.2, white), b.sphere([-0.75, 0, 0], 0.2, checker)]
    lamp, ball = b.quad([-1.5, 4, -1.5], [3, 0, 0], [0, 0, 3], e), b.sphere([0, 0, 0], 1.2, e)
    lights = b.list([lamp, ball]) if lean else b.list([lamp, b.list([ball, b.sphere([3, 6, 3], 0.3, e)])])  # weights 1/2, 1/4, 1/4
    hs = b.finish(b.list(things), lights, width=24, spp=4, max_depth=10, vfov=60, look_from=(0, 8, 9), look_at=(0, 0, 0),
                  background=b.solid(0.4, 0.5, 0.7))
    hs._builder = b
    return hs


def panic_rays(rng, n):
    """Straight down onto the shelves (every hit exactly in the plane y = 4), from inside the light sphere, at the zero-quaternion
    portal, and rays with a zero direction."""
    down = make_rays(np.column_stack([rng.uniform(-5, 5, n), np.full(n, 5.0), rng.uniform(-5, 5, n)]), np.tile([0.0, -1.0, 0.0], (n, 1)),
                     rng.uniform(0, 1, n))
    u = rng.normal(size=(n, 3))
    u *= (1.1 * rng.uniform(0, 1, n) ** (1 / 3) / np.linalg.norm(u, axis=1))[:, None]
    inside = make_rays(u, rng.normal(size=(n, 3)), rng.uniform(0, 1, n))
    m = n // 4
    portal = make_rays(np.column_stack([rng.uniform(-1.5, 1.5, m), rng.uniform(-2.5, 1.5, m), np.full(m, 2.0)]), np.tile([0.0, 0.0, -1.0], (m, 1)),
                       rng.uniform(0, 1, m))
    zero = make_rays(rng.uniform(-3, 3, (m, 3)), np.zeros((m, 3)), rng.uniform(0, 1, m))
    return np.concatenate([down, inside, portal, zero])


def panic_segments(rt, orc, lean):
    hs = panic_scene(rt, lean)
    rng = np.random.default_rng(31 + lean)
    osc = orc.OracleScene(hs)
    return hs, osc, walk_segments(orc, osc, hs, rng, 2000, panic_rays(rng, 3000))


def test_panic_family_reaches_every_error_rule(rt, orc):
    """The oracle side of the panic family: each rule ends segments with an error."""
    for lean in (True, False):
        hs, _, segs = panic_segments(rt, orc, lean)
        st, rays = segs["step"], segs["rays"]
        err = st["error"]
        on_shelf = (st["hit"] == 1) & (segs["rays"]["direction"][:, 1] == -1.0) & (rays["origin"][:, 1] == 5.0)
        inside = np.linalg.norm(rays["origin"], axis=1) < 1.2
        zero = (rays["direction"] == 0.0).all(axis=1)
        assert err[on_shelf].sum() >= 100, "value0 == value1 == 0"
        assert err[inside & (st["hit"] > 0)].sum() >= 200, "NaN light pdf"
        assert err[zero].sum() >= 500 and (st["hit"][zero] == 0).all(), "zero direction"
        with np.errstate(invalid="ignore"):
            assert np.isnan(st["emission"]).any(axis=1).sum() >= 200, "NaN emission"


@pytest.mark.gpu
@pytest.mark.parametrize("lean", [True, False], ids=["flat_lights", "nested_lights"])
def test_panic_segments_vs_oracle_and_routing(gpu, rt, orc, lean):
    """Every instantiation, lean twins included, meets the error rules and ends the path exactly as shade_one<SC_OTHER> and the
    oracle do."""
    hs, _, segs = panic_segments(rt, orc, lean)
    ds = dk.DeviceScene(hs)
    if lean:
        assert ds.shade_lean_mask >> SC_DIFFUSE & 1 and ds.shade_lean_mask >> SC_TEXTURED & 1 and ds.shade_lean_mask >> SC_ISOTROPIC & 1
        assert ds.has_walk_lean
    else:
        assert (ds.shade_lean_mask & (1 << SC_DIFFUSE | 1 << SC_TEXTURED | 1 << SC_ISOTROPIC)) == 0 and not ds.has_walk_lean
    seen = run_segments(ds, hs, segs, "panic " + ("flat" if lean else "nested"))
    labels = ["shade_one<other>", "shade_one<miss>", "shade_one<diffuse>", "shade_one<textured>", "shade_one<isotropic>", "shade_one<emissive>"]
    if lean:
        labels += ["shade_one<diffuse, lean>", "shade_one<textured, lean>", "lean_isotropic_scatter(ShadeLean)", "lean_isotropic_scatter(WalkLean)"]
    for label in labels:
        assert seen.get(label, [0, 0])[1] >= 20, (label, seen)

def draw(orc, seed, pixel, sample, segment, slot):
    import ctypes as C
    ab = (C.c_double * 2)()
    orc.lib().orc_kat_draw(seed, pixel, sample, segment, slot, ab)
    return ab[0], ab[1]


def boundary_segments(rt, orc, rng, n_addr=24):
    """Segments whose decision draw sits within a few ulps of its threshold, on both sides: the Dielectric's reflect / refract coin
    against the Schlick reflectance (a bisection over the ray's offset from the ball's axis, down to adjacent binary64 offsets), and
    Mix picks against ratios set to the draw itself and its neighbours (one Mix per ratio)."""
    b = rt.Builder(23)
    addrs = [(int(rng.integers(0, 2 ** 63)), PIXEL_MAX - k % 2, SAMPLE_MAX - k % 3, int(rng.integers(0, SEGMENT_MAX))) for k in range(n_addr)]
    red, green = b.lambertian(b.solid(0.8, 0.2, 0.1)), b.lambertian(b.solid(0.1, 0.8, 0.2))
    mixes = []
    for a in addrs:
        xi = draw(orc, *a, 6)[0]  # RT_SLOT_MIX, nesting level 0
        for d in (-2, -1, 0, 1, 2):
            r = xi
            for _ in range(abs(d)):
                r = np.nextafter(r, 2.0 if d > 0 else -1.0)
            mixes.append((a, b.mix(red, green, float(r))))
    glass = b.dielectric(b.solid(0.9, 1.0, 0.95), 1.5)
    objs = [b.sphere([0.0, 0.0, 0.0], 1.0, glass)]
    for k, (_, m) in enumerate(mixes):
        objs.append(b.sphere([4.0 + 3.0 * (k % 10), 3.0 * (k // 10), 0.0], 1.0, m))
    hs = b.finish(b.list([b.bvh(objs)]), width=8, spp=1, max_depth=8, look_from=(0, 0, 10), background=b.solid(0.3, 0.3, 0.3))
    hs._builder = b
    osc = orc.OracleScene(hs)
    rays, seeds, ids = [], [], []
    for k, (a, _) in enumerate(mixes):  # straight at the Mix sphere's centre
        c = np.array([4.0 + 3.0 * (k % 10), 3.0 * (k // 10), 0.0])
        rays.append(make_rays(c[None, :] + [[0.0, 0.0, 5.0]], [[0.0, 0.0, -1.0]], [0.25]))
        seeds.append(a[0]), ids.append(a[1:])
    for a in addrs:  # the glass ball: reflectance(s) rises with the offset s; find where the coin flips
        xi = draw(orc, *a, 3)[0]  # RT_SLOT_MATERIAL
        if not 0.045 < xi < 0.95:
            continue

        def reflects(s):
            st = osc.shade_step(make_rays([[s, 0.0, 5.0]], [[0.0, 0.0, -1.0]], [0.5]), [a[0]], [a[1:]])
            return st["d"][0, 2] > 0.0 or st["d"][0, 0] > 0.0  # refraction bends towards the axis, a reflection away from it

        lo, hi = 0.0, 1.0 - 1e-12
        assert not reflects(lo) and reflects(hi)
        while np.nextafter(lo, 2.0) < hi:
            mid = 0.5 * (lo + hi)
            if mid <= lo or mid >= hi:
                break
            lo, hi = (lo, mid) if reflects(mid) else (mid, hi)
        for s0 in (lo, hi):
            for d in (-2, -1, 0, 1, 2):
                s = s0
                for _ in range(abs(d)):
                    s = np.nextafter(s, 2.0 if d > 0 else -1.0)
                rays.append(make_rays([[s, 0.0, 5.0]], [[0.0, 0.0, -1.0]], [0.5]))
                seeds.append(a[0]), ids.append(a[1:])
    rays = np.concatenate(rays)
    n = len(rays)
    ids3 = np.array(ids, np.uint32).reshape(n, 3)
    segs = dict(rays=rays, beta=np.ones((n, 3)), seeds=np.array(seeds, np.uint64), ids3=ids3,
                max_depth=np.minimum(ids3[:, 2].astype(np.uint64) + 2, SEGMENT_MAX).astype(np.uint32))
    segs["step"] = osc.shade_step(rays, segs["seeds"], ids3)
    return hs, segs


def test_boundary_segments_reach_both_sides(rt, orc):
    """The oracle side of the draw-boundary family: both decisions occur at every threshold."""
    hs, segs = boundary_segments(rt, orc, np.random.default_rng(5))
    st = segs["step"]
    assert (st["hit"] == 1).all() and not st["error"].any()
    glass = segs["rays"]["origin"][:, 0] < 2.0
    refl = (st["d"][:, 2] > 0.0) | (st["d"][:, 0] > segs["rays"]["origin"][:, 0] * 0.0)
    assert refl[glass].sum() >= 40 and (~refl[glass]).sum() >= 40
    mix = ~glass  # the Mix rows: which material the pick chose shows in the albedo (cosine pdf)
    assert (st["albedo_x_pscatter"][mix, 0] > st["albedo_x_pscatter"][mix, 1]).any() and (st["albedo_x_pscatter"][mix, 0] < st["albedo_x_pscatter"][mix, 1]).any()


@pytest.mark.gpu
def test_boundary_segments_vs_oracle(gpu, rt, orc):
    hs, segs = boundary_segments(rt, orc, np.random.default_rng(5))
    ds = dk.DeviceScene(hs)
    run_segments(ds, hs, segs, "draw boundaries")


# ---------------------------------------------------------------- camera rays
@pytest.mark.gpu
@pytest.mark.parametrize("defocus", [0.0, 0.9])
@pytest.mark.parametrize("sqrt_spp", [1, 31, 4095])
def test_camera_rays(gpu, rt, orc, defocus, sqrt_spp):
    b = rt.Builder(1)
    hs = b.finish(b.list([b.sphere([0, 0, 0], 1.0, b.lambertian(b.solid(0.5, 0.5, 0.5)))]), width=16384, aspect=16384 / 16383, spp=sqrt_spp ** 2,
                  vfov=40, look_from=(0.3, 1.1, 7), look_at=(0, 0, 0), defocus_angle=defocus, focus_dist=6.5)
    cam = hs.camera
    assert cam.image_width == 16384 and cam.image_height == 16383 and cam.sqrt_spp == sqrt_spp
    W, H, S = cam.image_width, cam.image_height, sqrt_spp * sqrt_spp
    rng = np.random.default_rng(sqrt_spp)
    ij = [(0, 0), (W - 1, 0), (0, H - 1), (W - 1, H - 1), (W // 2, H - 1), (W - 1, H // 2), (0, H // 2), (W // 2, 0)]
    ij += [tuple(x) for x in np.column_stack([rng.integers(0, W, 24), rng.integers(0, H, 24)])]
    samples = sorted({0, S - 1, S // 2, max(S - 2, 0)} | set(rng.integers(0, S, 4).tolist()))
    assert (H - 1) * W + W - 1 > (1 << 28) - 2 ** 15  # the corner pixel index is close to 2^28
    for seed in (0, 2 ** 64 - 1, 0x9E3779B97F4A7C15):
        for s in samples:
            want = orc.camera_rays(cam, seed, ij, s)
            got = dk.camera_ray(cam, seed, [p[0] for p in ij], [p[1] for p in ij], s)
            compare("camera ray origin", got["origin"], want["origin"], rel=REL if defocus else 0.0,
                    scale=np.max(np.abs(want["origin"]), axis=1, keepdims=True))
            compare("camera ray direction", got["direction"], want["direction"], rel=REL if defocus else 0.0,
                    scale=np.max(np.abs(want["direction"]), axis=1, keepdims=True))
            compare("camera ray time", got["time"], want["time"])


# ---------------------------------------------------------------- renders at the packing limits
@pytest.mark.gpu
def test_render_at_the_top_of_the_sample_field(gpu, rt, orc):
    """sqrt_spp 4095 on a 16 x 16 frame, the two strata just below 4095^2: sample indices within 8193 of 2^24."""
    for h in (flat_four_scene(rt, "four", "gradient", width=16, spp=4095 ** 2),
              random_graph_scene(rt, 11, n_prims=40, with_media=True, width=16, spp=4095 ** 2, depth=8)):
        assert h.camera.sqrt_spp == 4095
        lo, hi = (1 << 24) - 8193, (1 << 24) - 8191
        assert hi == 4095 ** 2
        img, st = rt.Scene(h).render(seed=12, sample_begin=lo, sample_end=hi)
        ref, ost = orc.OracleScene(h).render(seed=12, sample_begin=lo, sample_end=hi)
        assert st.paths == ost.paths == 2 * 16 * 16
        # the device ends a path whose throughput is zero (a zero albedo, a light sample below the surface); the oracle recurses on
        # to max_depth with a zero weight, so it counts at least as many segments and errors
        assert 0 < st.segments <= ost.segments and st.errors <= ost.errors
        image_close(img, ref, frac_bad=0.0)


def cavity_scene(rt, depth):
    """Two parallel mirror plates, each a DiffuseLight wrapped around a fuzzy Metal, with the camera between them: every segment adds
    the light's colour and draws the metal's fuzz, and almost every path bounces until max_depth."""
    b = rt.Builder(21)
    plate = b.diffuse_light(b.solid(0.001, 0.002, 0.003), inner=b.metal([1.0, 1.0, 1.0], 0.004))
    world = b.list([b.quad([-1e5, -1e5, -0.5], [2e5, 0, 0], [0, 2e5, 0], plate), b.quad([-1e5, -1e5, 0.5], [2e5, 0, 0], [0, 2e5, 0], plate)])
    hs = b.finish(world, width=8, spp=1, max_depth=depth, vfov=4, look_from=(0, 0, 0.25), look_at=(0, 0, -1), background=b.solid(0, 0, 0))
    hs._builder = b
    return hs


def test_oracle_reaches_the_depth_limit(rt, orc):
    """The oracle recurses 4095 levels on the main thread (threads=1, for this render only: OpenMP's worker threads have smaller
    stacks)."""
    hs = cavity_scene(rt, 4095)
    osc = orc.OracleScene(hs)
    ref, ost = osc.render(seed=4, threads=1)
    assert ost.paths == 64 and ost.errors == 0
    assert ost.segments > 64 * 4000


@pytest.mark.gpu
def test_render_at_the_depth_limit(gpu, rt, orc):
    hs = cavity_scene(rt, 4095)
    img, st = rt.Scene(hs).render(seed=4)
    osc = orc.OracleScene(hs)
    ref, ost = osc.render(seed=4, threads=1)
    assert st.paths == ost.paths == 64 and st.segments == ost.segments and st.errors == ost.errors == 0
    assert st.segments > 64 * 4000  # paths pass segment 4000
    image_close(img, ref, frac_bad=0.0)
