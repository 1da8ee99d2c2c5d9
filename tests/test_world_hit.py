"""The world-hit query, rt_world_hit / rt_world_hit_device.

For ray i, with t_max_i the per-ray bound or the scalar one, out[i] is the HitRecord the reference's world.hit(ray,
Interval(t_min, t_max_i)) returns, media included: every ConstantMedium m draws philox(seed; pixel = i, sample = 0, segment,
RT_MEDIUM_SLOT(m)).  An empty interval gives a miss record.

The reference is the oracle's own world.hit with that path context (tests/world_hit_oracle.cpp); the CPU tests below tie it to
closed forms and to the oracle's known-answer hook.  Tolerances follow test_device_kat.py: the device is built with -fmad=false and
the oracle with -ffp-contract=off, so they differ only where libm does - ids, kinds, front faces, normals, surface t and p and planar
u, v are bit-equal; sphere u, v (acos, atan2) and a medium's t and p (log) agree to REL."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

from scenes_util import final_reduced_scene, random_graph_scene, random_rays
from test_device_kat import ellipsoid_scene
from transmittance_oracle import TransmittanceOracle
from world_hit_oracle import WorldHitOracle, hit_record_dtype

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
REL = 1e-13
RT_OBJ_SPHERE, RT_OBJ_MEDIUM = 1, 7
NAMED = {
    "book2_final": ("book2_final", 7, [32, 4, 12]),
    "cornell_glass": ("cornell_glass", 7, [32, 4, 12]),
    "book1_final": ("book1_final", 7, [48, 4, 12]),
}


@pytest.fixture(autouse=True, params=["by_size", "four_wide", "binary"])
def tree_variant(request, monkeypatch):
    """Every test runs on the tree rt_scene_create picks by size, on the four-wide collapse forced and on the binary tree
    forced, so that each surface-pass variant is exercised."""
    if request.param == "four_wide":
        monkeypatch.setenv("RT2025_WIDE_BVH", "1")
    elif request.param == "binary":
        monkeypatch.setenv("RT2025_WIDE_BVH", "0")
    return request.param


def make_scene(rt, name):
    if name == "random_graph":
        return random_graph_scene(rt, 11, n_prims=72, with_media=True, width=32, spp=4, depth=8)
    if name == "final_reduced":
        return final_reduced_scene(rt, width=96, spp=4, depth=12)
    if name == "ellipsoids":
        return ellipsoid_scene(rt)
    n, seed, params = NAMED[name]
    return rt.named_scene(n, seed=seed, params=params)


def scene_box(hs):
    bb = hs.objects()["bbox"]
    lo, hi = bb[:, 0::2], bb[:, 1::2]
    ok = np.isfinite(lo).all(axis=1) & np.isfinite(hi).all(axis=1)
    return lo[ok].min(axis=0), hi[ok].max(axis=0)


def query_rays(rt, hs, rng, n):
    """Half rays from the scene's box in random directions, half segments between two points of it (direction b - a, so that
    t = 1 is the far end and |d| is not 1); the per-ray bounds end the segments, or fall short of or beyond them."""
    lo, hi = scene_box(hs)
    c, h = (lo + hi) / 2, (hi - lo) / 2
    m = n // 2
    o1 = c + rng.uniform(-1, 1, (m, 3)) * h
    d1 = rng.normal(size=(m, 3))
    a = c + rng.uniform(-1, 1, (n - m, 3)) * h
    b = c + rng.uniform(-1, 1, (n - m, 3)) * h
    rays = rt.make_rays(np.vstack([o1, a]), np.vstack([d1, b - a]), rng.uniform(0, 1, n))
    scale = float(np.linalg.norm(h))
    per_ray = np.concatenate([rng.uniform(0.0, 2.0, m) * scale, np.where(rng.uniform(0, 1, n - m) < 0.5, 1.0, rng.uniform(0.2, 1.5, n - m))])
    return rays, per_ray


def assert_same_records(rt, hs, got, want):
    assert got.dtype == want.dtype and got.shape == want.shape
    for f in ("kind", "prim_id", "inst_id", "material", "front_face"):
        bad = got[f] != want[f]
        assert not bad.any(), f"{f}: {int(bad.sum())} of {len(got)} rays differ, first at {np.flatnonzero(bad)[0]}: {got[bad][0]} vs {want[bad][0]}"
    bits = lambda a: np.ascontiguousarray(a, dtype=np.float64).view(np.int64)  # noqa: E731
    surf, med, miss = (want["kind"] == k for k in (rt.RT_HIT_SURFACE, rt.RT_HIT_MEDIUM, rt.RT_HIT_MISS))
    # misses and surfaces: bit for bit, except the u, v of spheres
    for f in ("t", "p", "normal"):
        assert np.array_equal(bits(got[f][surf | miss]), bits(want[f][surf | miss])), f"{f} of surface hits / misses differ"
    sphere = surf & (hs.objects()["kind"][np.where(surf, want["prim_id"], 0)] == RT_OBJ_SPHERE)
    for f in ("u", "v"):
        assert np.array_equal(bits(got[f][~sphere]), bits(want[f][~sphere])), f"{f} of planar hits / media / misses differ"
        g, w = got[f][sphere], want[f][sphere]
        assert np.all(np.abs(g - w) <= REL * np.abs(w)), f"sphere {f} beyond REL"
    # media: the normal bit for bit (no transcendental function), t and p to REL (libm log); p against its length
    assert np.array_equal(bits(got["normal"][med]), bits(want["normal"][med]))
    assert np.all(np.abs(got["t"][med] - want["t"][med]) <= REL * np.abs(want["t"][med])), "medium t beyond REL"
    pn = np.linalg.norm(want["p"][med], axis=1)[:, None]
    assert np.all(np.abs(got["p"][med] - want["p"][med]) <= REL * pn), "medium p beyond REL"
    assert (got["reserved"] == 0).all()


def assert_all_misses(rt, rec):
    assert (rec["kind"] == rt.RT_HIT_MISS).all() and np.isinf(rec["t"]).all() and (rec["t"] > 0).all()
    assert (rec["p"] == 0).all() and (rec["normal"] == 0).all() and (rec["u"] == 0).all() and (rec["v"] == 0).all()
    for f in ("prim_id", "inst_id", "material"):
        assert (rec[f] == rt.RT_NONE).all()
    assert (rec["front_face"] == 0).all()


# ---------------------------------------------------------------- CPU: the layout and the reference

def test_hit_record_layout_matches_the_header(rt, tmp_path):
    fields = [f for f in rt.rt_hit_record_dtype.names]
    src = tmp_path / "rec.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "rt2025.h"\nint main(void) {\n'
                   '  printf("%zu", sizeof(rt_hit_record));\n'
                   + "".join(f'  printf(" %zu", offsetof(rt_hit_record, {f}));\n' for f in fields)
                   + '  printf(" %u %u %u\\n", RT_HIT_MISS, RT_HIT_SURFACE, RT_HIT_MEDIUM);\n  return 0;\n}\n')
    exe = tmp_path / "rec"
    subprocess.check_call(["/usr/bin/gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    dt = rt.rt_hit_record_dtype
    assert got == [dt.itemsize] + [dt.fields[f][1] for f in fields] + [rt.RT_HIT_MISS, rt.RT_HIT_SURFACE, rt.RT_HIT_MEDIUM]
    assert dt == hit_record_dtype and dt.itemsize == 96


@pytest.mark.parametrize("name", ["random_graph", "ellipsoids"])
def test_reference_equals_the_known_answer_hook_without_media(rt, orc, name):
    hs = random_graph_scene(rt, 3, n_prims=60) if name == "random_graph" else ellipsoid_scene(rt)
    rng = np.random.default_rng(2)
    o, d, t = random_rays(rng, 1000, extent=4.0)
    rays = rt.make_rays(o, d, t)
    got = WorldHitOracle(hs).world_hit(rays, t_min=1e-3, seed=9, segment=3)
    osc = orc.OracleScene(hs)
    hits = 0
    for i in range(len(rays)):
        want = osc.world_hit(o[i], d[i], time=t[i], t_min=1e-3)
        g = got[i]
        if want is None:
            assert g["kind"] == rt.RT_HIT_MISS and g["prim_id"] == rt.RT_NONE and math.isinf(g["t"])
            continue
        hits += 1
        assert g["kind"] == rt.RT_HIT_SURFACE
        assert g["t"] == want["t"] and list(g["p"]) == want["p"] and list(g["normal"]) == want["normal"]
        assert g["u"] == want["u"] and g["v"] == want["v"] and bool(g["front_face"]) == want["front_face"]
        assert g["prim_id"] == want["prim_id"] and g["inst_id"] == want["inst_id"]
        assert g["material"] == hs.objects()["material"][want["prim_id"]]
    assert hits > 80


R, RHO = 2.0, 0.3


def medium_scene(rt, density=RHO, odd=False, scale=None):
    """A sphere medium of radius R at the origin; `odd`: a medium far away takes media[0], so this one is media[1] and draws
    component b.  Returns (host scene, medium object, Transform object or None)."""
    b = rt.Builder(1)
    objs = []
    if odd:
        objs.append(b.medium(b.sphere([100, 100, 100], 1.0, b.empty()), 1.0, b.solid(1, 1, 1)))
    med = b.medium(b.sphere([0, 0, 0], R, b.empty()), density, b.solid(0.5, 0.6, 0.7))
    top = xf = None
    if scale is not None:
        top = xf = b.transform(med, scale=[scale] * 3)
    objs.append(top if top is not None else med)
    return b.finish(b.list(objs)), med, xf


def draws(orc, seed, n, segment, medium_index):
    ab = (C.c_double * 2)()
    slot = 16 + (medium_index >> 1)  # RT_MEDIUM_SLOT
    out = np.empty(n)
    for i in range(n):
        orc.lib().orc_kat_draw(seed, i, 0, segment, slot, ab)
        out[i] = ab[1] if medium_index & 1 else ab[0]
    return out


@pytest.mark.parametrize("odd", [False, True])
def test_reference_matches_closed_forms(rt, orc, odd):
    n, seed, segment = 600, 77, 5
    xi = draws(orc, seed, n, segment, 1 if odd else 0)
    hd = (-1.0 / RHO) * np.log(xi)  # hit_distance
    close = lambda got, want: np.allclose(got, want, rtol=1e-14, atol=0.0)  # noqa: E731

    def check(rec, t1, t2, dlen, med, inst=None):
        scat = hd <= (t2 - t1) * dlen
        assert 0.2 < scat.mean() < 0.95
        assert np.array_equal(rec["kind"], np.where(scat, rt.RT_HIT_MEDIUM, rt.RT_HIT_MISS))
        assert close(rec["t"][scat], t1 + hd[scat] / dlen) and np.isinf(rec["t"][~scat]).all()
        assert (rec["prim_id"][scat] == med).all() and (rec["inst_id"][scat] == (rt.RT_NONE if inst is None else inst)).all()
        assert (rec["material"][scat] == hs.objects()["material"][med]).all()
        assert (rec["u"] == 0).all() and (rec["v"] == 0).all()
        return scat

    # from outside, through the centre: t1 = 8, t2 = 12; d has a negative x, so the normal (1, 0, 0) faces the ray
    hs, med, _ = medium_scene(rt, odd=odd)
    osc = WorldHitOracle(hs)
    o, d = np.array([6.0, 0.0, -8.0]), np.array([-0.6, 0.0, 0.8])
    rays = rt.make_rays([o] * n, [d] * n)
    rec = osc.world_hit(rays, seed=seed, segment=segment)
    scat = check(rec, 8.0, 12.0, 1.0, med)
    assert close(rec["p"][scat], o + rec["t"][scat][:, None] * d)
    assert (rec["front_face"][scat] == 1).all() and (rec["normal"][scat] == [1.0, 0.0, 0.0]).all()
    # a direction of length 2: the same chord at half the t
    rec = osc.world_hit(rt.make_rays([o] * n, [2 * d] * n), seed=seed, segment=segment)
    check(rec, 4.0, 6.0, 2.0, med)
    # from inside: t1 = -2 is clamped up to t_min, then to 0
    for t_min in (0.0, 1e-8):
        rec = osc.world_hit(rt.make_rays([[0, 0, 0]] * n, [[0, 0, 1]] * n), t_min=t_min, seed=seed, segment=segment)
        scat = check(rec, t_min, 2.0, 1.0, med)
        assert (rec["front_face"][scat] == 0).all() and (rec["normal"][scat] == [-1.0, 0.0, 0.0]).all()
    # t_max_i cuts the chord: t2 = 10
    rec = osc.world_hit(rays, t_max=np.full(n, 10.0), seed=seed, segment=segment)
    check(rec, 8.0, 10.0, 1.0, med)
    # a scaled Transform over the medium: the local direction has length 1/2, the chord [6, 14] of the world ray counts 2R
    hs, med, xf = medium_scene(rt, odd=odd, scale=2.0)
    osc = WorldHitOracle(hs)
    o, d = np.array([0.0, 0.0, -10.0]), np.array([0.0, 0.0, 1.0])
    rec = osc.world_hit(rt.make_rays([o] * n, [d] * n), seed=seed, segment=segment)
    scat = check(rec, 6.0, 14.0, 0.5, med, inst=xf)
    assert close(rec["p"][scat], o + rec["t"][scat][:, None] * d)
    assert (rec["normal"][scat] == [-1.0, 0.0, 0.0]).all()  # local d.x = 0: not a front face



def test_reference_density_zero_and_infinite(rt):
    n = 300
    rays = rt.make_rays([[6.0, 0.0, -8.0]] * n, [[-0.6, 0.0, 0.8]] * n)
    rec = WorldHitOracle(medium_scene(rt, density=0.0)[0]).world_hit(rays, seed=3)
    assert (rec["kind"] == rt.RT_HIT_MISS).all()
    rec = WorldHitOracle(medium_scene(rt, density=float("inf"))[0]).world_hit(rays, seed=3)
    assert (rec["kind"] == rt.RT_HIT_MEDIUM).all() and (rec["t"] == 8.0).all()  # the entry point


def test_without_a_device_there_is_no_world_hit(rt):
    """Without a device no scene can be created (RT_ERR_NO_DEVICE), so there is nothing to query; with one the query runs.
    Null arguments are refused before anything is dereferenced."""
    L = rt.product_lib()
    hs = medium_scene(rt)[0]
    opts = rt.rt_build_opts(C.sizeof(rt.rt_build_opts), 0, -1, 0)
    h = C.c_void_p()
    rc = L.rt_scene_create(hs.desc, C.byref(opts), C.byref(h))
    ray = rt.make_rays([[6.0, 0.0, -8.0]], [[-0.6, 0.0, 0.8]])
    out = np.zeros(1, dtype=rt.rt_hit_record_dtype)
    st = rt.rt_stats()
    if L.rt_device_count() < 1:
        assert rc == -3 and not h.value  # RT_ERR_NO_DEVICE
    else:
        assert rc == 0
        assert L.rt_world_hit(h, ray.ctypes.data, None, 1, 1e-8, float("inf"), 1, 0, 0, out.ctypes.data, C.byref(st)) == 0
        L.rt_scene_destroy(h)
    fake_scene = C.c_void_p(ray.ctypes.data)  # never dereferenced: the arguments are checked first
    for scene, rays, o in ((None, ray.ctypes.data, out.ctypes.data), (fake_scene, None, out.ctypes.data), (fake_scene, ray.ctypes.data, None)):
        assert L.rt_world_hit(scene, rays, None, 1, 1e-8, float("inf"), 1, 0, 0, o, C.byref(st)) == -1
        assert "null" in L.rt_last_error().decode()
        assert L.rt_world_hit_device(scene, rays, None, 1, 1e-8, float("inf"), 1, 0, 0, o, None, C.byref(st)) == -1
        assert "null" in L.rt_last_error().decode()


# ---------------------------------------------------------------- GPU

@pytest.mark.gpu
@pytest.mark.parametrize("name", ["book2_final", "cornell_glass", "book1_final", "random_graph", "final_reduced", "ellipsoids"])
def test_world_hit_matches_oracle(gpu, rt, orc, name):
    hs = make_scene(rt, name)
    sc, osc = rt.Scene(hs), WorldHitOracle(hs)
    rng = np.random.default_rng(len(name))
    rays, per_ray = query_rays(rt, hs, rng, 6000)
    if name in NAMED or name in ("random_graph", "final_reduced"):
        rays = np.concatenate([np.load(os.path.join(GOLDEN, name + ".npz"))["rays"][:2000], rays])
        per_ray = np.concatenate([np.full(len(rays) - len(per_ray), np.inf), per_ray])
    lo, hi = scene_box(hs)
    finite = float(np.linalg.norm(hi - lo)) * 0.3
    kinds = 0
    for seed, segment, t_min, t_max in ((1, 0, 0.0, per_ray), (2, 3, 1e-8, float("inf")), (3, 7, 1e-3, per_ray), (4, 1, 1e-8, finite)):
        got, st = sc.world_hit(rays, t_min=t_min, t_max=t_max, seed=seed, segment=segment)
        want = osc.world_hit(rays, t_min=t_min, t_max=t_max, seed=seed, segment=segment)
        assert_same_records(rt, hs, got, want)
        assert st.segments == len(rays) and st.kernel_launches == 2
        kinds |= np.bitwise_or.reduce(1 << want["kind"].astype(np.int64))
    assert kinds & 0b011 == 0b011  # misses and surface hits
    if sc.info().n_media:
        assert kinds & 0b100, "no medium hit"


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cornell_glass", "book1_final", "ellipsoids", "random_graph_no_media", "book2_final", "random_graph"])
def test_world_hit_agrees_with_the_other_queries(gpu, rt, name):
    hs = random_graph_scene(rt, 8, n_prims=90) if name == "random_graph_no_media" else make_scene(rt, name)
    sc = rt.Scene(hs)
    rays, per_ray = query_rays(rt, hs, np.random.default_rng(3), 40000)
    for t_min, t_max in ((1e-8, float("inf")), (0.0, 3.0), (1e-3, per_ray)):
        rec, _ = sc.world_hit(rays, t_min=t_min, t_max=t_max, seed=11)
        occ, _ = sc.occluded(rays, t_min=t_min, t_max=t_max)
        hit = rec["kind"] != rt.RT_HIT_MISS
        assert hit[occ == 1].all()  # a surface hit inside the interval: never a miss
        if sc.info().n_media:
            continue
        assert np.array_equal(hit, occ == 1) and (rec["kind"] != rt.RT_HIT_MEDIUM).all()
        if np.ndim(t_max) == 0:
            ch, _ = sc.closest_hit(rays, t_min=t_min, t_max=t_max)
            assert np.array_equal(rec["t"].view(np.int64), ch["t"].view(np.int64))
            assert np.array_equal(rec["prim_id"], ch["prim_id"]) and np.array_equal(rec["inst_id"], ch["inst_id"])
            assert np.array_equal(rec["u"].astype(np.float32), ch["u"]) and np.array_equal(rec["v"].astype(np.float32), ch["v"])


def segment_rays(rt, rng, n, lo, hi):
    lo, hi = np.asarray(lo, dtype=np.float64), np.asarray(hi, dtype=np.float64)
    a = lo + rng.uniform(0, 1, (n, 3)) * (hi - lo)
    b = lo + rng.uniform(0, 1, (n, 3)) * (hi - lo)
    length = np.linalg.norm(b - a, axis=1)
    return rt.make_rays(a, (b - a) / length[:, None], rng.uniform(0, 1, n)), length


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["random_graph", "final_reduced"])
def test_miss_frequency_is_the_transmittance(gpu, rt, name):
    """Replicated 2^16 times (the draws differ by ray index), a ray misses with the probability rt_transmittance gives."""
    hs = make_scene(rt, name)
    sc = rt.Scene(hs)
    rng = np.random.default_rng(21)
    if name == "final_reduced":
        bb = hs.objects()["bbox"][hs.objects()["kind"] == RT_OBJ_MEDIUM][0]
        lo, hi = bb[0::2], bb[1::2]
        c, h = (lo + hi) / 2, (hi - lo) * 0.75
        rays, length = segment_rays(rt, rng, 20000, c - h, c + h)
    else:
        rays, length = segment_rays(rt, rng, 20000, [-5, -5, -5], [5, 5, 5])
    T, _ = sc.transmittance(rays, t_max=length)
    pick = np.flatnonzero((T > 0.15) & (T < 0.85))[:4]
    assert len(pick) == 4
    N = 1 << 16
    rep = np.repeat(rays[pick], N)
    rec, _ = sc.world_hit(rep, t_max=np.repeat(length[pick], N), seed=2024, segment=2)
    for k, i in enumerate(pick):
        f = (rec["kind"][k * N:(k + 1) * N] == rt.RT_HIT_MISS).mean()
        assert abs(f - T[i]) <= 5 * math.sqrt(T[i] * (1 - T[i]) / N), (i, f, T[i])
        assert (rec["kind"][k * N:(k + 1) * N] != rt.RT_HIT_SURFACE).all()


@pytest.mark.gpu
def test_determinism_and_draw_addresses(gpu, rt, monkeypatch):
    hs = random_graph_scene(rt, 5, n_prims=100, with_media=True)
    rays, per_ray = query_rays(rt, hs, np.random.default_rng(4), 30000)
    outs = []
    for wide in (None, "1", "0"):
        if wide is None:
            monkeypatch.delenv("RT2025_WIDE_BVH", raising=False)
        else:
            monkeypatch.setenv("RT2025_WIDE_BVH", wide)
        sc = rt.Scene(hs)
        outs.append(sc.world_hit(rays, t_max=per_ray, seed=7, segment=4)[0])
        outs.append(sc.world_hit(rays, t_max=per_ray, seed=7, segment=4)[0])
        sc.close()
    for o in outs[1:]:
        assert o.tobytes() == outs[0].tobytes()
    sc = rt.Scene(hs)
    base = outs[0]
    med = base["kind"] == rt.RT_HIT_MEDIUM
    assert med.sum() > 500
    for kw in (dict(seed=7, segment=5), dict(seed=8, segment=4)):
        other = sc.world_hit(rays, t_max=per_ray, **kw)[0]
        changed = (other["kind"] != base["kind"]) | (other["t"] != base["t"])
        assert changed[med].mean() > 0.5
        surf = (base["kind"] == rt.RT_HIT_SURFACE) & (other["kind"] == rt.RT_HIT_SURFACE)
        assert np.array_equal(other["t"][surf], base["t"][surf])


@pytest.mark.gpu
def test_device_entry_equals_host_entry(gpu, rt):
    import torch
    hs = random_graph_scene(rt, 4, n_prims=150, with_media=True)
    sc = rt.Scene(hs)
    rays, per_ray = query_rays(rt, hs, np.random.default_rng(6), 50001)
    want, _ = sc.world_hit(rays, t_min=0.1, t_max=per_ray, seed=3, segment=9)
    want_scalar, _ = sc.world_hit(rays, t_min=0.1, t_max=5.0, seed=3, segment=9)
    d_rays = torch.from_numpy(rays.view(np.float64).reshape(-1, 7).copy()).cuda()
    d_tmax = torch.from_numpy(per_ray).cuda()
    nbytes = len(rays) * rt.rt_hit_record_dtype.itemsize
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        d_out = torch.full((nbytes,), 7, dtype=torch.uint8, device="cuda")
        st = sc.world_hit_device(d_rays.data_ptr(), len(rays), d_out.data_ptr(), d_tmax.data_ptr(), t_min=0.1, seed=3, segment=9,
                                 flags=rt.RT_OPT_COUNT, stream=s.cuda_stream)
        d_out2 = torch.full((nbytes,), 7, dtype=torch.uint8, device="cuda")
        sc.world_hit_device(d_rays.data_ptr(), len(rays), d_out2.data_ptr(), t_min=0.1, t_max=5.0, seed=3, segment=9, stream=s.cuda_stream)
    s.synchronize()
    assert d_out.cpu().numpy().tobytes() == want.tobytes()
    assert d_out2.cpu().numpy().tobytes() == want_scalar.tobytes()
    assert st.segments == len(rays) and st.kernel_launches == 2 and st.ms_total > 0
    assert st.node_visits > 0 and st.prim_tests > 0
    _, occ = sc.occluded(rays, t_min=0.1, t_max=per_ray, flags=rt.RT_OPT_COUNT)
    assert st.prim_tests > occ.prim_tests


@pytest.mark.gpu
def test_edge_cases(gpu, rt, orc):
    # zero rays
    b = rt.Builder(1)
    sc = rt.Scene(b.finish(b.list([b.sphere([0, 0, 0], 1.0, b.empty())])))
    got, st = sc.world_hit(np.zeros(0, dtype=rt.rt_ray_dtype))
    assert len(got) == 0 and st.segments == 0 and st.kernel_launches == 0
    o, d, t = random_rays(np.random.default_rng(1), 5000)
    rays = rt.make_rays(o, d, t)
    # an empty world misses everything
    b = rt.Builder(1)
    assert_all_misses(rt, rt.Scene(b.finish(b.list([]))).world_hit(rays)[0])
    # media under a Transform, under a BVH and under a Transform of a BVH, next to surfaces; then zero and infinite densities
    for densities in ((0.3, 0.5, 0.2), (0.0, 0.5, 0.2), (float("inf"), 0.5, 0.0)):
        b = rt.Builder(2)
        m, iso = b.lambertian(b.solid(0.5, 0.5, 0.5)), b.solid(0.9, 0.9, 0.9)
        fog = b.transform(b.medium(b.sphere([0.3, 0, 0], 1.5, b.empty()), densities[0], iso), offset=[0.2, -0.4, 0.3],
                          quat=b.quat_axis_angle([1, 2, 0.5], 40.0), scale=[1.6, 0.8, 1.2])
        boxed = b.bvh([b.medium(b.box([-2, 2, -2], [2, 3, 2], b.empty()), densities[1], iso), b.sphere([3, 0, 0], 0.7, m),
                       b.quad([-1, -1, -3], [2, 0, 0], [0, 2, 0], m)])
        nested = b.transform(b.bvh([b.medium(b.sphere([0, 0, 0], 1.0, b.empty()), densities[2], iso), b.triangle([-1, -1, 3], [2, 0, 0], [0, 2, 0], m)]),
                             offset=[-3, 0, 1], scale=[1.5, 1.5, 1.5])
        hs = b.finish(b.list([fog, boxed, nested]))
        sc, osc = rt.Scene(hs), WorldHitOracle(hs)
        for t_min, t_max in ((1e-8, float("inf")), (0.5, 6.0)):
            got = sc.world_hit(rays, t_min=t_min, t_max=t_max, seed=5, segment=1)[0]
            want = osc.world_hit(rays, t_min=t_min, t_max=t_max, seed=5, segment=1)
            assert_same_records(rt, hs, got, want)
        meds = hs.objects()["kind"] == RT_OBJ_MEDIUM
        hit_media = set(want["prim_id"][want["kind"] == rt.RT_HIT_MEDIUM].tolist())
        for k, obj in enumerate(np.flatnonzero(meds)):  # media in creation order: fog, box, nested
            assert (obj in hit_media) == (densities[k] > 0.0), (densities, k)
        if math.isinf(densities[0]):  # scatters where the ray enters the boundary
            T = TransmittanceOracle(hs).transmittance(rays, t_min=t_min, t_max=t_max)
            assert ((want["kind"] == rt.RT_HIT_MEDIUM) & (want["prim_id"] == np.flatnonzero(meds)[0])).sum() > 100
            assert (want["kind"][T == 0.0] != rt.RT_HIT_MISS).all()
    # empty intervals and NaN bounds: miss records, whatever the scene holds
    tm = np.where(np.arange(len(rays)) % 2 == 0, np.nan, 0.25)
    assert_all_misses(rt, sc.world_hit(rays, t_min=0.5, t_max=tm, seed=5)[0])
    assert_all_misses(rt, sc.world_hit(rays, t_min=float("nan"), seed=5)[0])
    assert_all_misses(rt, sc.world_hit(rays, t_min=3.0, t_max=2.0, seed=5)[0])


@pytest.mark.gpu
def test_stats_and_counters(gpu, rt):
    hs = make_scene(rt, "book2_final")
    sc = rt.Scene(hs)
    rays, per_ray = query_rays(rt, hs, np.random.default_rng(8), 20000)
    rec, st = sc.world_hit(rays, t_max=per_ray, flags=rt.RT_OPT_COUNT)
    assert st.segments == len(rays) and st.kernel_launches == 2 and st.ms_total > 0
    assert st.node_visits > 0 and st.prim_tests > 0
    rec2, st2 = sc.world_hit(rays, t_max=per_ray)
    assert rec2.tobytes() == rec.tobytes() and st2.node_visits == 0
