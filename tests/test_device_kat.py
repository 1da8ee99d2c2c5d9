"""The device shading functions, one call at a time, against the oracle.

Every function of csrc/shade.cuh and csrc/disney.cuh that the shade kernels call is run through a thin wrapper kernel
(tests/device_kat.cu, the product's own header code on the product's compiled tables) with the inputs the oracle is given, and
the outputs are compared number by number: Disney evaluate / generate, textures, the environment lookup, hit records with their
Transform chains and the OBJ loader's remap, the light mixture's pdf and sampling (generic and the lean kernels' staged list) and
the emission of DiffuseLight / Mix nests.  The images of test_gpu_parity.py tolerate a few wrong pixels; these tests do not.

Tolerances.  The device is built with -fmad=false and the oracle with -ffp-contract=off, so the two differ only where libm does:
- bit equality where no transcendental function is involved (solid, checker, gradient and image textures, hit points, normals and
  front faces, planar u, v, the remap, quad and triangle lights of a flat list, the cdf pick);
- REL = 1e-13 relative elsewhere (sin, pow, acos, atan2, exp, log in Disney, sphere lights and sphere u, v, Perlin noise, sums
  over a nested light list, which the oracle evaluates level by level and the device as one weighted sum); the components of a
  generated unit direction are measured against its length;
- None / error decisions identical everywhere.
"""
import ctypes as C
import math

import numpy as np
import pytest

import device_kat as dk
from scenes_util import obj_mesh_scene, random_graph_scene, random_rays
from test_disney_restatement import CASES, lobe_pdfs
from test_restatements import flat_material

REL = 1e-13
TINY = 5e-324
material_dtype = np.dtype([("kind", "<u4"), ("tex", "<u4"), ("inner", "<u4"), ("inner2", "<u4"), ("color", "<f8", (3,)), ("param", "<f8"),
                           ("v", "<f8", (16,))])
remap_dtype = np.dtype([("tex_ori", "<f8", (3,)), ("tex_u", "<f8", (3,)), ("tex_v", "<f8", (3,)), ("u_vec", "<f8", (3,)), ("v_vec", "<f8", (3,)),
                        ("normal", "<f8", (3, 3)), ("has_uv_vecs", "<u4"), ("normal_tex", "<u4")])
assert material_dtype.itemsize == 176 and remap_dtype.itemsize == 200
RT_OBJ_SPHERE, RT_MAT_DIFFUSE_LIGHT, RT_MAT_MIX, RT_MAT_REMAPPED = 1, 4, 7, 10
PRIM_SPHERE = 0

# per function: [values compared, bit-equal values, largest relative difference]
STATS = {}


@pytest.fixture(scope="module", autouse=True)
def report():
    yield
    if STATS:
        print("\n%-28s %10s %10s %12s" % ("function", "values", "bit-equal", "max rel"))
        for k, (n, eq, mx) in sorted(STATS.items()):
            print("%-28s %10d %10d %12.3e" % (k, n, eq, mx))


def compare(name, got, want, rel=0.0, floor=0.0):
    """got == want bit for bit where rel == 0; else within rel * max(|want|, floor).  floor = 1 measures the components of a unit
    vector against its length.  NaN and infinity patterns must agree exactly."""
    got, want = np.asarray(got, dtype=np.float64).ravel(), np.asarray(want, dtype=np.float64).ravel()
    assert got.shape == want.shape
    gn, wn = np.isnan(got), np.isnan(want)
    assert np.array_equal(gn, wn), f"{name}: NaN pattern differs at {np.flatnonzero(gn != wn)[:8]}"
    bits = (got.view(np.int64) == want.view(np.int64)) | (gn & wn)
    fin = np.isfinite(want) & ~bits
    assert np.array_equal(np.isinf(got), np.isinf(want)) and np.all(got[np.isinf(want)] == want[np.isinf(want)]), f"{name}: infinities differ"
    diff = np.abs(got[fin] - want[fin])
    scale = np.maximum(np.maximum(np.abs(want[fin]), floor), np.finfo(np.float64).tiny)
    relerr = diff / scale
    allowed = rel * scale
    bad = diff > allowed
    st = STATS.setdefault(name, [0, 0, 0.0])
    st[0] += got.size
    st[1] += int(bits.sum())
    st[2] = max(st[2], float(relerr.max()) if relerr.size else 0.0)
    if bad.any():
        k = np.flatnonzero(fin)[np.flatnonzero(bad)[0]]
        pytest.fail(f"{name}: {int(bad.sum())} of {got.size} values differ beyond the bound; first at flat index {k}: {got[k]!r} vs {want[k]!r}")


def flat_table(hs, field, dtype, n):
    d = hs.desc.contents
    buf = (C.c_char * (n * dtype.itemsize)).from_address(getattr(d, field))
    return np.frombuffer(buf, dtype=dtype).copy()


def unit(v):
    """UnitVec3::from_vec3's arithmetic, (1 / |v|) v; not finite for a zero vector."""
    v = np.asarray(v, dtype=np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        return (np.float64(1.0) / np.sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2])) * v


# ---------------------------------------------------------------- Disney BSDF
def with_y(rng, y, n):
    """n unit-ish vectors whose y is exactly `y` (x, z random, scaled so the length is about 1)."""
    xz = rng.normal(size=(n, 2))
    xz *= np.sqrt(max(1.0 - y * y, 0.0)) / np.linalg.norm(xz, axis=1)[:, None]
    return np.column_stack([xz[:, 0], np.full(n, y), xz[:, 1]])


def random_units(rng, n):
    v = rng.normal(size=(n, 3))
    return v / np.linalg.norm(v, axis=1)[:, None]


EDGE_Y = [0.0, -0.0, TINY, -TINY, 1e-300, -1e-300, 1e-17, -1e-17, 1.0, -1.0]


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_disney_evaluate(gpu, orc, name):
    p = CASES[name]
    rng = np.random.default_rng(7 + sum(map(ord, name)))
    v_out, v_in = [random_units(rng, 600)], [random_units(rng, 600)]
    for yo in EDGE_Y:  # grazing and exactly tangent directions on either side, against random and edge partners
        for yi in EDGE_Y:
            v_out.append(with_y(rng, yo, 2))
            v_in.append(with_y(rng, yi, 2))
    vo = random_units(rng, 20)
    v_out += [vo, vo, with_y(rng, 0.0, 4)]
    v_in += [vo, -vo, None]  # the same direction; the opposite one (a transmission pair through h = unit(2 v_in))
    v_in[-1] = -v_out[-1]    # opposite tangent directions: h = unit(0), the reference panics
    v_out, v_in = np.concatenate(v_out), np.concatenate(v_in)
    n_inf = 0
    for front in (True, False):
        refl, pdf, err = dk.disney_evaluate(p.flat(), p.thin, v_out, v_in, front)
        want_refl, want_pdf, want_err = np.zeros_like(refl), np.zeros_like(pdf), np.zeros(len(pdf), bool)
        for i in range(len(v_out)):
            got = orc.disney_evaluate(p.flat(), p.thin, v_out[i], v_in[i], front)
            if got is None:
                want_err[i] = True
            else:
                want_refl[i], want_pdf[i] = got
        assert np.array_equal(err, want_err), f"error decisions differ at {np.flatnonzero(err != want_err)[:8]}"
        ok = ~want_err
        compare("disney::evaluate_disney", refl[ok], want_refl[ok], rel=REL)
        compare("disney::evaluate_disney", pdf[ok], want_pdf[ok], rel=REL)
        n_inf += int(np.isinf(want_pdf[ok]).sum())
    assert len(v_out) >= 600
    if name in ("metal_aniso", "mirror"):
        assert n_inf > 0  # the zero-pdf -> +inf quirk is reached


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_disney_generate(gpu, orc, name):
    p = CASES[name]
    rng = np.random.default_rng(11 + sum(map(ord, name)))
    p_spec, p_diff, p_clear, p_trans = lobe_pdfs(p)
    # the lobe choice: picks exactly on each cumulative lobe probability and one ulp either side
    bounds = [p_spec, p_spec + p_clear, p_spec + p_diff + p_clear]
    picks_a = sorted({x for b in bounds for x in (np.nextafter(b, -1.0), b, np.nextafter(b, 2.0)) if 0.0 <= x < 1.0} | {0.0, np.nextafter(1.0, 0.0)})
    # the second coin (diffuse transmission / Fresnel reflection)
    picks_b = [0.0, p.diff_trans, np.nextafter(p.diff_trans, -1.0), np.nextafter(p.diff_trans, 2.0)]
    v_out = np.concatenate([random_units(rng, 260), with_y(rng, 0.0, 4), with_y(rng, TINY, 2), with_y(rng, -TINY, 2), with_y(rng, 1e-17, 2)])
    rows_vo, rows_pick, rows_u = [], [], []
    for vo in v_out:
        for a in picks_a + list(rng.uniform(size=4)):
            b = picks_b[rng.integers(0, len(picks_b))] if rng.uniform() < 0.5 else rng.uniform()
            u = rng.uniform(size=2) if rng.uniform() < 0.9 else np.array([0.0, np.nextafter(1.0, 0.0)])
            rows_vo.append(vo), rows_pick.append((a, b)), rows_u.append(u)
    vo, pick, u = np.array(rows_vo), np.array(rows_pick), np.array(rows_u)
    n = 0
    for front in (True, False):
        d, rc = dk.disney_generate(p.flat(), p.thin, vo, front, pick, u)
        want_rc, want_d = np.zeros(len(vo), np.int64), np.zeros_like(d)
        for i in range(len(vo)):
            got = orc.disney_generate(p.flat(), p.thin, vo[i], front, pick[i], u[i])
            if isinstance(got, str):
                want_rc[i] = -1
            elif got is not None:
                want_rc[i], want_d[i] = 1, got
        assert np.array_equal(rc, want_rc), f"Some / None / panic decisions differ at {np.flatnonzero(rc != want_rc)[:8]}"
        some = rc == 1
        compare("disney::generate_local", d[some], want_d[some], rel=REL, floor=1.0)  # unit directions
        n += len(vo)
    assert n >= 16000 // len(CASES)  # at least 16000 forced draws over all the parameter sets


# ---------------------------------------------------------------- textures and the environment
def texture_scene(rt):
    rng = np.random.default_rng(31)
    b = rt.Builder(31)
    img = rng.uniform(0.0, 1.0, (5, 7, 4)).astype(np.float32)
    row, col = rng.uniform(0.0, 1.0, (1, 6, 4)).astype(np.float32), rng.uniform(0.0, 1.0, (6, 1, 4)).astype(np.float32)
    texs = {
        "solid": b.solid(0.3, 0.6, 0.9),
        "checker": b.checker(0.5, b.solid(0.9, 0.1, 0.2), b.solid(0.05, 0.6, 0.3)),  # inv_scale 2: boundaries at multiples of 0.5
        "image_srgb": b.image(img),
        "image_linear": b.image(img, linear_format=True),
        "image_bilinear": b.image(img, raw=True),
        "row_nearest": b.image(row), "col_nearest": b.image(col),
        "row_bilinear": b.image(row, raw=True), "col_bilinear": b.image(col, raw=True),
        "missing": b.image_missing(),
        "noise": b.noise(1.7),
        "gradient": b.gradient([0.1, 0.2, 0.3], [0.9, 0.7, 0.5]),
    }
    objs = [b.sphere([3.0 * k, 0, 0], 1.0, b.lambertian(t)) for k, t in enumerate(texs.values())]
    hs = b.finish(b.list(objs), width=8, spp=1)
    return hs, {name: flat_material(hs, k)[1] for k, name in enumerate(texs)}


def edge_coords(w, h):
    """u or v values where lookups go wrong: 0, 1, just below 1, negative, > 1, exact texel edges and centres with their neighbours."""
    xs = {0.0, -0.0, 1.0, np.nextafter(1.0, 0.0), np.nextafter(0.0, 1.0), -1e-17, -0.25, -1.0, -1.5, 1.5, 2.0, 3.75, 1e-300}
    for n in (w, h, 1):
        for k in range(n + 1):
            for c in (k / n, (k + 0.5) / n):
                xs |= {c, np.nextafter(c, -1.0), np.nextafter(c, 2.0), c - 1.0, c + 2.0}
    return sorted(xs)


@pytest.mark.gpu
def test_texture_value(gpu, rt, orc):
    hs, tex = texture_scene(rt)
    ds, osc = dk.DeviceScene(hs), orc.OracleScene(hs)
    rng = np.random.default_rng(5)
    coords = edge_coords(7, 6)
    uv = np.array([(u, v) for u in coords for v in coords[:: 3]] + list(rng.uniform(-3.0, 3.0, (300, 2))))
    # p for checker, noise and gradient: integer and half-integer lattice points (negative ones included), one ulp off them,
    # and random points
    lat = np.array([-3.0, -1.0, -0.5, -0.0, 0.0, 0.5, 1.0, 2.5, -255.0, 256.0, -1e6])
    pts = [np.array([a, b, c]) for a in lat for b in lat[::2] for c in lat[::3]]
    pts += [np.nextafter(q, q + 1.0) for q in pts[::5]] + [np.nextafter(q, q - 1.0) for q in pts[::7]]
    pts = np.array(pts + list(rng.uniform(-40.0, 40.0, (400, 3))))
    for name, t in tex.items():
        if name in ("checker", "noise", "gradient"):
            u, v, p = rng.uniform(-2.0, 2.0, len(pts)), rng.uniform(-2.0, 2.0, len(pts)), pts
        else:
            u, v, p = uv[:, 0], uv[:, 1], rng.uniform(-5.0, 5.0, (len(uv), 3))
        got = ds.texture_value(t, u, v, p)
        want = np.array([osc.texture_value(t, u[i], v[i], p[i]) for i in range(len(p))])
        compare("texture_value:" + name, got, want, rel=REL if name == "noise" else 0.0)
    assert np.all(ds.texture_value(tex["missing"], uv[:, 0], uv[:, 1], np.zeros((len(uv), 3))) == [0.0, 1.0, 1.0])


@pytest.mark.gpu
def test_background_value(gpu, rt, orc):
    """shapes/environment.rs:14-24: the equirect (u, v) of the unit direction, computed here with the oracle's libm."""
    hs, tex = texture_scene(rt)
    ds, osc = dk.DeviceScene(hs), orc.OracleScene(hs)
    rng = np.random.default_rng(6)
    axes = [[1, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0], [0, 0, 1], [0, 0, -1], [1, 1, 0], [0, -1, 1], [3, 4, 0], [0, 0, 0], [1e-300, 0, 0]]
    dirs = np.concatenate([np.array(axes, dtype=np.float64), rng.normal(size=(1500, 3)) * rng.uniform(0.01, 100.0, (1500, 1))])
    for name in ("image_srgb", "image_bilinear", "checker", "gradient", "solid", "missing"):
        t = tex[name]
        got, ok = ds.background_value(t, dirs)
        want, want_ok = np.zeros_like(got), np.zeros(len(dirs), bool)
        for i, d in enumerate(dirs):
            pv = unit(d)
            if not np.all(np.isfinite(pv)):
                continue  # UnitVec3::from_vec3 panics
            want_ok[i] = True
            u = v = 0.0
            if name in ("image_srgb", "image_bilinear", "checker"):
                u = (math.pi - math.atan2(-pv[2], pv[0])) / (2.0 * math.pi)
                v = math.acos(-pv[1]) / math.pi
            want[i] = osc.texture_value(t, u, v, pv)
        assert np.array_equal(ok, want_ok)
        compare("background_value:" + name, got[ok], want[ok], rel=REL)


# ---------------------------------------------------------------- hit records
def ellipsoid_scene(rt):
    """test_gpu_parity.test_ellipsoids_and_nested_transforms' scene: non-uniform and mirroring scales, Transform chains, a moving sphere."""
    b = rt.Builder(9)
    m = b.empty()
    e1 = b.transform(b.sphere([0, 0, 0], 1.0, m), offset=[-2, 0, 0], quat=b.quat_axis_angle([0, 0, 1], 30.0), scale=[2.0, 0.5, 1.0])
    inner = b.transform(b.bvh([b.sphere([0, 0, 0], 0.7, m), b.quad([-1, -1, 1], [2, 0, 0], [0, 2, 0], m),
                               b.triangle([0, 1, -1], [1, 0, 0], [0, 1, 1], m)]), offset=[0.5, 0, 0], scale=[1, 2, 1])
    e2 = b.transform(b.list([inner, b.sphere_moving([0, -2, 0], [1, -2, 0], 0.5, m)]), offset=[2.5, 0.5, 0],
                     quat=b.quat_axis_angle([1, 1, 0], 50.0), scale=[0.8, 0.8, 1.6])
    e3 = b.transform(b.sphere([0, 0, 0], 1.0, m), offset=[0, 3, 0], scale=[-1.0, 1.0, 1.5])  # a mirroring scale
    return b.finish(b.list([e1, e2, e3]))


def oracle_hits(rt, osc, rays):
    keep, recs = [], []
    for i, r in enumerate(rays):
        h = osc.world_hit(r["origin"], r["direction"], float(r["time"]))
        if h is not None:
            keep.append(i), recs.append(h)
    return np.array(keep, dtype=np.int64), recs


def check_hit_records(rt, orc, hs, rays, min_hits):
    ds, osc = dk.DeviceScene(hs), orc.OracleScene(hs)
    keep, recs = oracle_hits(rt, osc, rays)
    assert len(keep) >= min_hits
    obj = np.array([h["prim_id"] for h in recs], dtype=np.uint32)
    prim = ds.prim_of_object[obj]
    assert np.all(prim != dk.RT_NONE)
    got = ds.surface_hit_info(prim, np.array([h["t"] for h in recs]), rays[keep])
    assert np.all(got["ok"])
    compare("surface_hit_info:p", got["p"], [h["p"] for h in recs])
    compare("surface_hit_info:normal", got["normal"], [h["normal"] for h in recs])
    assert np.array_equal(got["front_face"], [h["front_face"] for h in recs])
    sphere = hs.objects()["kind"][obj] == RT_OBJ_SPHERE
    for key in ("u", "v"):
        want = np.array([h[key] for h in recs])
        compare("surface_hit_info:planar_uv", got[key][~sphere], want[~sphere])
        compare("surface_hit_info:sphere_uv", got[key][sphere], want[sphere], rel=REL)  # acos / atan2
    return ds, osc, obj, got, recs


@pytest.mark.gpu
def test_surface_hit_info_ellipsoids_and_nested_transforms(gpu, rt, orc):
    hs = ellipsoid_scene(rt)
    rng = np.random.default_rng(4)
    o, d, t = random_rays(rng, 4000, extent=5.0)
    t[:300], t[300:600], t[600:900] = 0.0, 0.5, 1.0  # the moving sphere at both ends and the middle of the shutter
    _, _, obj, _, _ = check_hit_records(rt, orc, hs, rt.make_rays(o, d, t), 250)
    assert len(set(obj.tolist())) >= 5


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [5, 12])
def test_surface_hit_info_random_graphs(gpu, rt, orc, seed):
    hs = random_graph_scene(rt, seed, n_prims=90)
    rng = np.random.default_rng(seed)
    o, d, t = random_rays(rng, 3000, extent=6.0)
    check_hit_records(rt, orc, hs, rt.make_rays(o, d, t), 300)


@pytest.mark.gpu
def test_remap_record_on_obj_faces(gpu, rt, orc):
    """RemappedMaterial::remap_record (shapes/obj.rs:32-62) on the faces of obj_mesh_scene, with and without a normal map; the
    texel of the normal map is the oracle's, the rest is the reference's arithmetic restated."""
    hs = obj_mesh_scene(rt)
    rng = np.random.default_rng(8)
    n = 3000
    o = np.column_stack([rng.uniform(-3.2, 3.2, n), np.full(n, 4.0), rng.uniform(-3.2, 3.2, n)])
    d = np.column_stack([rng.normal(0, 0.2, n), -np.ones(n), rng.normal(0, 0.2, n)])
    ds, osc, obj, got, recs = check_hit_records(rt, orc, hs, rt.make_rays(o, d), 500)
    d_ = hs.desc.contents
    mats = flat_table(hs, "materials", material_dtype, d_.n_materials)
    remaps = flat_table(hs, "remaps", remap_dtype, d_.n_remaps)
    mat = hs.objects()["material"][obj]
    face = mats["kind"][mat] == RT_MAT_REMAPPED
    assert face.sum() >= 400
    idx = mats["inner2"][mat[face]]
    sel = {k: v[face] for k, v in got.items()}
    out = ds.remap_record(idx, sel)
    want_n, want_u, want_v, want_ok = [], [], [], []
    for k, r in enumerate(idx):
        R = remaps[r]
        h = sel
        u, v = h["u"][k], h["v"][k]
        tc = R["tex_ori"] + u * R["tex_u"] + v * R["tex_v"]
        ok = True
        raw = (1.0 - u - v) * R["normal"][0] + u * R["normal"][1] + v * R["normal"][2]
        nn = unit(raw)
        ok = ok and bool(np.all(np.isfinite(nn)))
        if R["normal_tex"] != dk.RT_NONE:
            c = osc.texture_value(int(R["normal_tex"]), tc[0], tc[1], h["p"][k]) * 2.0 - 1.0
            ok = ok and bool(R["has_uv_vecs"])
            nn = unit(R["u_vec"] * c[0] + R["v_vec"] * c[1] + nn * c[2])
            ok = ok and bool(np.all(np.isfinite(nn)))
        want_n.append(nn), want_u.append(tc[0]), want_v.append(tc[1]), want_ok.append(ok)
    assert np.array_equal(out["ok"], want_ok)
    compare("remap_record:normal", out["normal"], want_n)
    compare("remap_record:uv", np.column_stack([out["u"], out["v"]]), np.column_stack([want_u, want_v]))
    assert np.array_equal(out["front_face"], sel["front_face"]) and np.array_equal(out["p"], sel["p"])
    mapped = remaps["normal_tex"][idx] != dk.RT_NONE
    assert 100 <= mapped.sum() <= len(idx) - 100  # both branches


# ---------------------------------------------------------------- lights
# A light list is described as nested Python lists of leaves; ("T", child, kw) is a Transform.  expected_weights restates
# light_weights of the oracle: a list divides its weight among its children, a Transform passes it on.
def build_lights(b, spec):
    if isinstance(spec, list):
        return b.list([build_lights(b, s) for s in spec])
    if spec[0] == "T":
        return b.transform(build_lights(b, spec[1]), **spec[2])
    kind, args = spec
    m = b.empty()
    return b.sphere(*args, m) if kind == "sphere" else b.quad(*args, m) if kind == "quad" else b.triangle(*args, m)


def expected_weights(spec, w=1.0):
    if isinstance(spec, list):
        return [x for s in spec for x in expected_weights(s, w / float(len(spec)))]
    if spec[0] == "T":
        return expected_weights(spec[1], w)
    return [w]


QUAD = ("quad", ([-1.5, 5.5, -1.5], [3, 0, 0], [0, 0, 3]))
SPHERE = ("sphere", ([2.5, 2.0, 0.0], 0.6))
TRI = ("triangle", ([-4.0, 1.0, -2.0], [1.5, 0.5, 0.0], [0.0, 1.5, 1.0]))
FLAT = [QUAD, SPHERE, TRI]
NESTED = [QUAD, [SPHERE, TRI], ("T", [("quad", ([0, 0, 0], [1, 0, 0], [0, 0, 1])), ("sphere", ([0, 0, 0], 0.5)),
                                      ("triangle", ([0, 0, 0], [1, 0, 0], [0, 1, 0]))],
                                 dict(offset=[-3.0, 3.5, 1.0], quat=[0.9238795325112867, 0.0, 0.3826834323650898, 0.0], scale=[1.5, 0.7, 1.2])),
          [[("T", ("quad", ([-0.5, 0.0, -0.5], [1, 0, 0], [0, 0, 1])), dict(offset=[3.0, 4.0, -2.0], scale=[2.0, 1.0, -1.0]))]]]
QUAD_ONLY = [QUAD, ("quad", ([3.0, -1.0, -3.0], [0, 2, 0], [0, 0, 2])), ("triangle", ([-4.0, 1.0, -2.0], [1.5, 0.5, 0.0], [0.0, 1.5, 1.0]))]


def light_scene(rt, spec):
    b = rt.Builder(17)
    world = b.list([b.sphere([0, -100.5, 0], 100.0, b.lambertian(b.solid(0.5, 0.5, 0.5))), build_lights(b, spec)])
    return b.finish(world, build_lights(b, spec), width=8, spp=1)


@pytest.mark.parametrize("spec", ["FLAT", "NESTED", "QUAD_ONLY"])
def test_light_table_weights_and_cdf(rt, spec):
    """Runs without a device: the compiled light leaves weigh prod 1/len and their cdf is the running sum in the oracle's order."""
    s = globals()[spec]
    tab = dk.light_table(light_scene(rt, s))
    w = expected_weights(s)
    assert np.array_equal(tab["weight"], w)
    assert np.array_equal(tab["cdf"], np.cumsum(w))  # sequential binary64 sums, as light_weights' caller adds them
    kinds = {"quad": 1, "triangle": 2, "sphere": 0}
    flat_kinds = []

    def walk(x, xf):
        if isinstance(x, list):
            for c in x:
                walk(c, xf)
        elif x[0] == "T":
            walk(x[1], True)
        else:
            flat_kinds.append((kinds[x[0]], xf))
    walk(s, False)
    assert tab["kind"].tolist() == [k for k, _ in flat_kinds]
    assert ((tab["xform"] != dk.RT_NONE).tolist()) == [x for _, x in flat_kinds]


def light_origins(rng):
    c, r = np.array(SPHERE[1][0]), SPHERE[1][1]
    dirs = random_units(rng, 40)
    return np.concatenate([rng.uniform(-5.0, 5.0, (150, 3)),
                           c + 3.0 * r * dirs[:10],            # outside the sphere light
                           c + r * dirs[10:25],                # on it (to rounding)
                           c + 0.5 * r * dirs[25:35], c[None]])  # inside it and at its centre


def light_dirs(rng, origins, tab_pts):
    """Per origin: a random direction, directions towards points of the lights (hits), and directions parallel to the quad light."""
    o, d = [], []
    for x in origins:
        for q in tab_pts:
            o.append(x), d.append(q - x + rng.normal(0, 0.05, 3))
        o.append(x), d.append(rng.normal(size=3))
        o.append(x), d.append([rng.normal(), 0.0, rng.normal()])  # parallel to the quad light's plane y = 5.5
    return np.array(o), np.array(d)


LIGHT_POINTS = [np.array([0.0, 5.5, 0.0]), np.array([2.5, 2.0, 0.0]), np.array([-3.4, 2.2, -1.4]), np.array([-3.0, 3.5, 1.0]),
                np.array([3.0, 4.0, -2.0]), np.array([4.0, 0.0, -2.0])]


@pytest.mark.gpu
@pytest.mark.parametrize("spec", ["FLAT", "NESTED", "QUAD_ONLY"])
def test_lights_pdf_value(gpu, rt, orc, spec):
    s = globals()[spec]
    hs = light_scene(rt, s)
    ds, osc = dk.DeviceScene(hs), orc.OracleScene(hs)
    # the flat lists qualify for the lean kernels' staged list (at most four untransformed leaves of weight 1/n), the nested one does not
    assert ds.lights_flat == ds.has_lean == (spec != "NESTED")
    rng = np.random.default_rng(21)
    o, d = light_dirs(rng, light_origins(rng), LIGHT_POINTS)
    got = ds.lights_pdf(o, d)
    want = np.array([osc.lights_pdf_value(o[i], d[i]) for i in range(len(o))])
    assert (want > 0).sum() > len(o) // 6 and (want == 0).sum() > 100
    # a flat list of quads and triangles is pure binary64 arithmetic in the oracle's order; a sphere light's pdf has a sqrt, and a
    # nested list is summed level by level in the oracle, as one weighted sum on the device
    compare("lights_pdf_value:" + spec, got, want, rel=0.0 if spec == "QUAD_ONLY" else REL)
    if ds.has_lean:
        compare("lean_lights_pdf=generic", ds.lights_pdf(o, d, lean=True), got)


@pytest.mark.gpu
@pytest.mark.parametrize("spec", ["FLAT", "NESTED", "QUAD_ONLY"])
def test_lights_random(gpu, rt, orc, spec):
    s = globals()[spec]
    hs = light_scene(rt, s)
    ds, osc = dk.DeviceScene(hs), orc.OracleScene(hs)
    tab = dk.light_table(hs)
    cdf = tab["cdf"]
    rng = np.random.default_rng(22)
    # picks exactly at every cdf value and one ulp either side, where the leaf must be the oracle's; 0; random picks
    picks = sorted({x for c in cdf for x in (np.nextafter(c, -1.0), c, np.nextafter(c, 2.0)) if x < 1.0} | {0.0, np.nextafter(1.0, 0.0)})
    picks += list(rng.uniform(size=20))
    origins = light_origins(rng)
    rows = [(x, pk, *(rng.uniform(size=2) if rng.uniform() < 0.85 else (0.0, np.nextafter(1.0, 0.0)))) for x in origins for pk in picks]
    o = np.array([r[0] for r in rows])
    pick, r1, r2 = (np.array([r[k] for r in rows]) for k in (1, 2, 3))
    leaf = np.array([int(np.searchsorted(cdf, pk, side="right")) for pk in pick])  # first leaf with pick < cdf
    leaf = np.minimum(leaf, len(cdf) - 1)
    got, ok = ds.lights_random(o, pick, r1, r2)
    want, want_ok = np.zeros_like(got), np.zeros(len(o), bool)
    for i in range(len(o)):
        w = osc.lights_random(o[i], int(leaf[i]), r1[i], r2[i])
        if w is not None:
            want[i], want_ok[i] = w, True
    assert np.array_equal(ok, want_ok), f"ok decisions differ at {np.flatnonzero(ok != want_ok)[:8]}"
    plain = (tab["kind"][leaf] != PRIM_SPHERE) & (tab["xform"][leaf] == dk.RT_NONE) & ok
    other = ~plain & ok
    compare("lights_random:planar", got[plain], want[plain])  # quad and triangle leaves: no transcendental
    compare("lights_random:sphere_or_transformed", got[other], want[other], rel=REL)
    assert plain.any() and (spec == "QUAD_ONLY" or other.any())
    if ds.has_lean:
        lg, lok = ds.lights_random(o, pick, r1, r2, lean=True)
        assert np.array_equal(lok, ok)
        compare("lean_lights_random=generic", lg[ok], got[ok])


# ---------------------------------------------------------------- emission
def emission_scene(rt):
    rng = np.random.default_rng(41)
    b = rt.Builder(41)
    img = rng.uniform(0.0, 1.0, (5, 7, 4)).astype(np.float32)
    alpha = rng.uniform(0.0, 1.0, (4, 6, 4)).astype(np.float32)
    t_img, t_alpha, t_missing = b.image(img), b.image(alpha), b.image_missing()
    dl = lambda r, g, bb, inner=dk.RT_NONE: b.diffuse_light(b.solid(r, g, bb), inner)  # noqa: E731
    lam = b.lambertian(b.solid(0.5, 0.5, 0.5))
    mats = [
        dl(4, 3, 2),
        dl(4, 3, 2, inner=dl(0.5, 0.25, 0.125)),
        dl(1, 1, 1, inner=b.disney((0.7, 0.7, 0.9), roughness=0.5)),
        b.mix(dl(4, 3, 2), b.diffuse_light(t_img), 0.3),
        b.mix_image(dl(2, 5, 1), b.mix(dl(0.5, 0.25, 7), lam, 0.6), t_alpha),
        dl(3, 0.5, 0.25, inner=b.mix_image(dl(1, 2, 3), dl(9, 8, 7), t_missing)),
        b.mix(b.mix_image(lam, dl(1, 3, 5), t_alpha), b.mix(dl(6, 6, 6, inner=dl(0.1, 0.2, 0.3)), b.transparent(), 0.25), 0.7),
        lam,
    ]
    hs = b.finish(b.list([b.sphere([3.0 * k, 0, 0], 1.0, m) for k, m in enumerate(mats)]), width=8, spp=1)
    return hs, [flat_material(hs, k)[0] for k in range(len(mats))], alpha


def emitted_reference(osc, mats, m, u, v, p):
    """Material::emitted of the reference: DiffuseLight = its texture + its inner material's emission, Mix = m1 (1 - r) + m2 r."""
    M = mats[m]
    if M["kind"] == RT_MAT_DIFFUSE_LIGHT:
        e = osc.texture_value(int(M["tex"]), u, v, p)
        return e + (emitted_reference(osc, mats, int(M["inner"]), u, v, p) if M["inner"] != dk.RT_NONE else 0.0)
    if M["kind"] == RT_MAT_MIX:
        r = M["param"]
        if M["tex"] != dk.RT_NONE:
            r = osc.alpha(int(M["tex"]), u, v)
        return emitted_reference(osc, mats, int(M["inner"]), u, v, p) * (1.0 - r) + emitted_reference(osc, mats, int(M["inner2"]), u, v, p) * r
    return np.zeros(3)


@pytest.mark.gpu
def test_material_emitted(gpu, rt, orc):
    hs, flat, alpha = emission_scene(rt)
    ds, osc = dk.DeviceScene(hs), orc.OracleScene(hs)
    d_ = hs.desc.contents
    mats = flat_table(hs, "materials", material_dtype, d_.n_materials)
    texs = flat_table(hs, "textures", np.dtype([("kind", "<u4"), ("a", "<u4"), ("b", "<u4"), ("r", "<u4"), ("rest", "<f8", (8,))]), d_.n_textures)
    images = flat_table(hs, "images", np.dtype([("width", "<u4"), ("height", "<u4"), ("flags", "<u4"), ("r", "<u4"), ("off", "<u8")]), d_.n_images)
    texels = np.frombuffer((C.c_float * d_.n_texels).from_address(d_.texels), dtype=np.float32)

    def alpha_of(t, u, v):  # ImageTexture::alpha, texture.rs:102-109: the nearest texel's alpha (never decoded), 1 without an image
        if texs["a"][t] == dk.RT_NONE:
            return 1.0
        im = images[texs["a"][t]]
        w, h = int(im["width"]), int(im["height"])
        uu, vv = u - math.floor(u), 1.0 - (v - math.floor(v))
        i, j = min(int(uu * w), w - 1), min(int(vv * h), h - 1)
        return float(texels[int(im["off"]) + 4 * (j * w + i) + 3])
    osc.alpha = alpha_of
    rng = np.random.default_rng(3)
    coords = edge_coords(6, 4)
    uv = np.array([(u, v) for u in coords[::2] for v in coords[::4]] + list(rng.uniform(-2.0, 3.0, (200, 2))))
    p = rng.uniform(-3.0, 3.0, (len(uv), 3))
    for k, m in enumerate(flat):
        got = ds.material_emitted(m, uv[:, 0], uv[:, 1], p)
        want = np.array([emitted_reference(osc, mats, m, uv[i, 0], uv[i, 1], p[i]) for i in range(len(uv))])
        compare("material_emitted", got, want, rel=REL)
        if k == len(flat) - 1:
            assert np.all(got == 0.0)
