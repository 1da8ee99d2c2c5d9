"""The transmittance query, rt_transmittance / rt_transmittance_device.

For ray i, with t_max_i the per-ray bound or the scalar one, out[i] is the probability that world.hit(ray, [t_min, t_max_i])
returns None when every ConstantMedium draws its own uniform number: 0 where a surface is hit in the interval (exactly where
rt_occluded answers 1), else the product over the media of exp(L / neg_inv_density), L being the distance_inside_boundary of
ConstantMedium::hit (volume.rs:42-58) on the caller's interval.  An empty interval gives 1.

The reference is the oracle's own world.hit traversal with the free-flight comparison of ConstantMedium::hit replaced by its
probability (tests/transmittance_oracle.cpp); the CPU tests below tie it to closed forms and to the oracle's ConstantMedium::hit
itself with forced draws.  The arithmetic before exp is the
same binary64 on both sides, so the device matches the oracle to the last ulps of exp, with the zero pattern exact."""
import ctypes as C
import math
import os

import numpy as np
import pytest

from scenes_util import final_reduced_scene, random_graph_scene, random_rays
from transmittance_oracle import TransmittanceOracle

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
NAMED = {
    "book2_final": ("book2_final", 7, [32, 4, 12]),
    "cornell_glass": ("cornell_glass", 7, [32, 4, 12]),
    "book1_final": ("book1_final", 7, [48, 4, 12]),
}


@pytest.fixture(autouse=True, params=["by_size", "four_wide", "binary"])
def tree_variant(request, monkeypatch):
    """Every test runs on the tree rt_scene_create picks by size, on the four-wide collapse forced and on the binary tree
    forced, so that each occlusion-pass variant the query runs first is exercised."""
    if request.param == "four_wide":
        monkeypatch.setenv("RT2025_WIDE_BVH", "1")
    elif request.param == "binary":
        monkeypatch.setenv("RT2025_WIDE_BVH", "0")
    return request.param


def golden_scene(rt, name):
    if name == "random_graph":
        return random_graph_scene(rt, 11, n_prims=72, with_media=True, width=32, spp=4, depth=8)
    if name == "final_reduced":
        return final_reduced_scene(rt, width=96, spp=4, depth=12)
    n, seed, params = NAMED[name]
    return rt.named_scene(n, seed=seed, params=params)


def assert_same_transmittance(got, want):
    """Zero pattern and NaN pattern exact; elsewhere the last ulps of exp (CUDA's against libm's) may differ."""
    assert got.dtype == np.float64 and got.shape == want.shape
    assert np.array_equal(got == 0.0, want == 0.0), f"{int(((got == 0.0) != (want == 0.0)).sum())} zero-pattern mismatches"
    np.testing.assert_allclose(got, want, rtol=1e-14, atol=0.0, equal_nan=True)


def segment_rays(rt, rng, n, lo, hi):
    """Segments between two uniform points of the box [lo, hi]: unit directions, t_max_i = |b - a|."""
    lo, hi = np.asarray(lo, dtype=np.float64), np.asarray(hi, dtype=np.float64)
    a = lo + rng.uniform(0, 1, (n, 3)) * (hi - lo)
    b = lo + rng.uniform(0, 1, (n, 3)) * (hi - lo)
    length = np.linalg.norm(b - a, axis=1)
    return rt.make_rays(a, (b - a) / length[:, None], rng.uniform(0, 1, n)), length


def medium_bbox(hs):
    """The bounding box (lo, hi) of the scene's first ConstantMedium, as the reference computed it."""
    objs = hs.objects()
    bb = objs["bbox"][objs["kind"] == 7][0]  # RT_OBJ_MEDIUM
    return bb[0::2], bb[1::2]


# ---------------------------------------------------------------- CPU: the reference

R, RHO = 2.0, 0.3


def one_medium(rt, density=RHO, surface=False, scale=None):
    b = rt.Builder(1)
    med = b.medium(b.sphere([0, 0, 0], R, b.empty()), density, b.solid(1, 1, 1))
    if scale is not None:
        med = b.transform(med, scale=[scale] * 3)
    objs = [med]
    if surface:
        objs.append(b.sphere([0, 0, 5], 1.0, b.lambertian(b.solid(0.5, 0.5, 0.5))))
    return b.finish(b.list(objs))


def test_reference_matches_closed_forms(rt):
    osc = TransmittanceOracle(one_medium(rt))
    o, z = [0, 0, -10], [0, 0, 1]
    rays = rt.make_rays([o], [z])
    close = lambda got, want: math.isclose(got, want, rel_tol=1e-12)  # noqa: E731
    assert close(osc.transmittance(rays)[0], math.exp(-2 * R * RHO))              # through the centre
    assert close(osc.transmittance(rays, t_max=10.0)[0], math.exp(-R * RHO))      # up to the centre
    inside = rt.make_rays([[0, 0, 0]], [z])
    assert close(osc.transmittance(inside, t_min=0.0)[0], math.exp(-R * RHO))     # from inside: t1 < 0 becomes 0
    # a longer direction: the same segment, with the t bounds scaled to match
    d3 = rt.make_rays([o], [[0, 0, 3]])
    assert close(osc.transmittance(d3)[0], math.exp(-2 * R * RHO))
    assert close(osc.transmittance(d3, t_max=10.0 / 3.0)[0], math.exp(-R * RHO))
    # per-ray bounds, an empty interval and a NaN bound
    got = osc.transmittance(rt.make_rays([o] * 4, [z] * 4), t_max=np.array([np.inf, 10.0, 5.0, np.nan]))
    assert close(got[0], math.exp(-2 * R * RHO)) and close(got[1], math.exp(-R * RHO)) and got[2] == 1.0 and got[3] == 1.0
    # a scaled Transform over the medium: ray_length is measured in the medium's space (volume.rs:55), so the world
    # chord of 4R counts as 2R
    assert close(TransmittanceOracle(one_medium(rt, scale=2.0)).transmittance(rays)[0], math.exp(-2 * R * RHO))
    # density 0 lets everything through; a surface in the interval stops everything
    assert TransmittanceOracle(one_medium(rt, density=0.0)).transmittance(rays)[0] == 1.0
    blocked = TransmittanceOracle(one_medium(rt, surface=True))
    assert blocked.transmittance(rays)[0] == 0.0
    assert close(blocked.transmittance(rays, t_max=13.0)[0], math.exp(-2 * R * RHO))


def single_medium_scene(rt, kind):
    b = rt.Builder(3)
    iso = b.solid(0.8, 0.8, 0.8)
    if kind == "sphere":
        med = b.medium(b.sphere([0.5, -0.3, 0.2], 2.5, b.empty()), 0.35, iso)
    elif kind == "box":
        med = b.medium(b.box([-2, -1.5, -2.5], [2.5, 2, 1.5], b.empty()), 0.2, iso)
    elif kind == "transformed_sphere":
        med = b.transform(b.medium(b.sphere([0.3, 0, 0], 1.5, b.empty()), 0.5, iso), offset=[0.2, -0.4, 0.3],
                          quat=b.quat_axis_angle([1, 2, 0.5], 40.0), scale=[1.6, 0.8, 1.2])
    else:  # the boundary sphere alone under a Transform
        med = b.medium(b.transform(b.sphere([0, 0, 0], 1.5, b.empty()), offset=[0.3, 0.2, -0.1], scale=[1.5, 1.5, 1.5]), 0.5, iso)
    return b.finish(b.list([med]))


@pytest.mark.parametrize("kind", ["sphere", "box", "transformed_sphere", "sphere_under_transform"])
def test_forced_draws_tie_transmittance_to_constant_medium_hit(rt, orc, kind):
    """T is the threshold of the reference's own comparison: ConstantMedium::hit scatters iff the draw is at least T."""
    hs = single_medium_scene(rt, kind)
    osc = orc.OracleScene(hs)
    rng = np.random.default_rng(7)
    o, _, t = random_rays(rng, 1000, extent=4.0)
    d = rng.uniform(-1.0, 1.0, (len(o), 3)) - o  # aimed near the medium
    t_max = rng.uniform(0.2, 1.5, len(o))
    T = TransmittanceOracle(hs).transmittance(rt.make_rays(o, d, t), t_max=t_max)
    inside = np.flatnonzero((T > 0) & (T < 1))
    assert len(inside) > 100
    for i in inside[:120]:
        kw = dict(time=t[i], t_max=t_max[i])
        assert osc.world_hit(o[i], d[i], xi=(T[i] * (1 + 1e-9),) * 2, **kw) is not None  # the medium: the world holds nothing else
        assert osc.world_hit(o[i], d[i], xi=(T[i] * (1 - 1e-9),) * 2, **kw) is None


def test_null_arguments_are_refused_without_a_device(rt):
    L = rt.product_lib()
    ray = np.zeros(1, dtype=rt.rt_ray_dtype)
    out = np.zeros(1, dtype=np.float64)
    fake_scene = C.c_void_p(ray.ctypes.data)  # never dereferenced: the arguments are checked first
    st = rt.rt_stats()
    for scene, rays, o in ((None, ray.ctypes.data, out.ctypes.data), (fake_scene, None, out.ctypes.data), (fake_scene, ray.ctypes.data, None)):
        assert L.rt_transmittance(scene, rays, None, 1, 1e-8, float("inf"), 0, o, C.byref(st)) == -1
        assert "null" in L.rt_last_error().decode()
        assert L.rt_transmittance_device(scene, rays, None, 1, 1e-8, float("inf"), 0, o, None, C.byref(st)) == -1
        assert "null" in L.rt_last_error().decode()


# ---------------------------------------------------------------- GPU

@pytest.mark.gpu
@pytest.mark.parametrize("name", ["book2_final", "cornell_glass", "book1_final", "random_graph", "final_reduced"])
def test_transmittance_on_golden_scenes(gpu, rt, orc, name):
    fx = np.load(os.path.join(GOLDEN, name + ".npz"))
    hs = golden_scene(rt, name)
    sc = rt.Scene(hs)
    rays = fx["rays"]
    T, st = sc.transmittance(rays)
    occ = sc.occluded(rays)[0]
    assert np.array_equal(occ, fx["hits"]["prim_id"] != rt.RT_NONE)
    assert (T[occ] == 0.0).all()
    assert st.kernel_launches == 2 and st.segments == len(rays)
    if sc.info().n_media == 0:
        assert np.array_equal(T, 1.0 - occ)
    if name == "book2_final":  # every unoccluded ray leaves through the global mist
        assert (~occ).sum() > 100 and ((T[~occ] > 0) & (T[~occ] < 1)).all()
    assert_same_transmittance(T, TransmittanceOracle(hs).transmittance(rays))


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_transmittance_matches_oracle_on_random_graphs(gpu, rt, orc, seed):
    """Transforms, lists, BVHs, a sphere medium and a box medium (the general-boundary variant)."""
    hs = random_graph_scene(rt, seed, n_prims=120, with_media=True)
    sc, osc = rt.Scene(hs), TransmittanceOracle(hs)
    rng = np.random.default_rng(seed)
    o, d, t = random_rays(rng, 30000)
    rays = rt.make_rays(o, d, t)
    per_ray = np.where(np.arange(len(rays)) % 5 == 0, np.inf, rng.uniform(-0.5, 9.0, len(rays)))
    for t_min in (1e-8, 0.5, -1.0):
        for t_max in (float("inf"), 4.0, per_ray):
            want = osc.transmittance(rays, t_min=t_min, t_max=t_max)
            got, _ = sc.transmittance(rays, t_min=t_min, t_max=t_max)
            assert_same_transmittance(got, want)
            assert np.array_equal(got == 0.0, sc.occluded(rays, t_min=t_min, t_max=t_max)[0])
    part = (want > 0) & (want < 1)
    assert part.mean() > 0.2 and (want == 0).mean() > 0.1


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["final_reduced", "sphere_under_transform", "transformed_sphere"])
def test_each_media_variant_matches_oracle(gpu, rt, orc, kind):
    """The general-boundary variant on the fog mesh of config 4, and the Transform variant where the medium and its sphere
    have different Transforms (the sphere's own local ray) or share one."""
    rng = np.random.default_rng(12)
    if kind == "final_reduced":
        hs = final_reduced_scene(rt, width=96, spp=4, depth=12)
        lo, hi = medium_bbox(hs)
        c, h = (lo + hi) / 2, (hi - lo) * 0.75
        rays, length = segment_rays(rt, rng, 40000, c - h, c + h)
    else:
        hs = single_medium_scene(rt, kind)
        rays, length = segment_rays(rt, rng, 40000, [-4, -4, -4], [4, 4, 4])
    sc, osc = rt.Scene(hs), TransmittanceOracle(hs)
    got, _ = sc.transmittance(rays, t_max=length)
    want = osc.transmittance(rays, t_max=length)
    assert_same_transmittance(got, want)
    assert ((want > 0) & (want < 1)).mean() > 0.1
    assert_same_transmittance(sc.transmittance(rays)[0], osc.transmittance(rays))


@pytest.mark.gpu
def test_edge_cases(gpu, rt, orc):
    # zero rays
    b = rt.Builder(1)
    sc = rt.Scene(b.finish(b.list([b.sphere([0, 0, 0], 1.0, b.empty())])))
    got, st = sc.transmittance(np.zeros(0, dtype=rt.rt_ray_dtype))
    assert len(got) == 0 and st.segments == 0 and st.kernel_launches == 0
    assert len(sc.transmittance(np.zeros(0, dtype=rt.rt_ray_dtype), t_max=np.zeros(0))[0]) == 0
    o, d, t = random_rays(np.random.default_rng(1), 5000)
    rays = rt.make_rays(o, d, t)
    # an empty world lets everything through
    b = rt.Builder(1)
    assert (rt.Scene(b.finish(b.list([]))).transmittance(rays)[0] == 1.0).all()
    # a world of media only, then density 0 and an infinite density
    for densities in ((5.0, 0.5), (0.0, 0.5), (float("inf"), 0.5), (0.0, 0.0)):
        b = rt.Builder(1)
        fog = b.medium(b.sphere([0, 0, 0], 3.0, b.empty()), densities[0], b.solid(1, 1, 1))
        box = b.medium(b.box([-6, -6, -6], [6, 6, 6], b.empty()), densities[1], b.solid(1, 1, 1))
        hs = b.finish(b.list([fog, box]))
        got = rt.Scene(hs).transmittance(rays)[0]
        assert_same_transmittance(got, TransmittanceOracle(hs).transmittance(rays))
        if densities == (0.0, 0.0):
            assert (got == 1.0).all()
        if math.isinf(densities[0]):
            assert (got == 0.0).sum() > 300
    # empty intervals and NaN bounds
    tm = np.where(np.arange(len(rays)) % 2 == 0, np.nan, 0.25)
    assert (rt.Scene(hs).transmittance(rays, t_min=0.5, t_max=tm)[0] == 1.0).all()
    assert (rt.Scene(hs).transmittance(rays, t_min=float("nan"))[0] == 1.0).all()
    assert (rt.Scene(hs).transmittance(rays, t_min=3.0, t_max=2.0)[0] == 1.0).all()
    # axis-parallel, zero and degenerate directions, a NaN origin, in a scene with surfaces and media
    b = rt.Builder(1)
    m = b.empty()
    hs = b.finish(b.list([b.bvh([b.sphere([0, 0, 0], 1.0, m), b.quad([-1, -1, -3], [2, 0, 0], [0, 2, 0], m),
                                 b.triangle([-1, -1, 3], [2, 0, 0], [0, 2, 0], m), b.sphere([4, 0, 0], 0.5, m)]),
                          b.medium(b.sphere([0, 0, 0], 8.0, b.empty()), 0.1, b.solid(1, 1, 1)),
                          b.medium(b.box([-2, 2, -2], [2, 3, 2], b.empty()), 0.7, b.solid(1, 1, 1))]))
    sc, osc = rt.Scene(hs), TransmittanceOracle(hs)
    o = [[0, 0, 5], [0, 0, 5], [-5, 0, 0], [0, 0, 0], [0, 0, 5], [float("nan"), 0, 5], [0.25, 0.25, -10], [0, 0, 5], [0, 2.5, 5]]
    d = [[0, 0, -1], [0, 0, 1], [1, 0, 0], [0, 1, 0], [0, 0, 0], [0, 0, -1], [0, 0, 1e-30], [0, 0, -1e300], [0, 0, -1]]
    rays = rt.make_rays(o, d)
    got = sc.transmittance(rays)[0]
    assert_same_transmittance(got, osc.transmittance(rays))
    assert np.array_equal(got == 0.0, sc.occluded(rays)[0])


@pytest.mark.gpu
def test_device_entry_equals_host_entry(gpu, rt):
    import torch
    hs = random_graph_scene(rt, 4, n_prims=150, with_media=True)
    sc = rt.Scene(hs)
    rng = np.random.default_rng(6)
    o, d, t = random_rays(rng, 50001)
    rays = rt.make_rays(o, d, t)
    t_max = rng.uniform(0.0, 12.0, len(rays))
    want, _ = sc.transmittance(rays, t_min=0.1, t_max=t_max)
    want_scalar, _ = sc.transmittance(rays, t_min=0.1, t_max=5.0)
    d_rays = torch.from_numpy(rays.view(np.float64).reshape(-1, 7).copy()).cuda()
    d_tmax = torch.from_numpy(t_max).cuda()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        d_out = torch.full((len(rays),), 7.0, dtype=torch.float64, device="cuda")
        st = sc.transmittance_device(d_rays.data_ptr(), len(rays), d_out.data_ptr(), d_tmax.data_ptr(), t_min=0.1, flags=rt.RT_OPT_COUNT,
                                     stream=s.cuda_stream)
        d_out2 = torch.full((len(rays),), 7.0, dtype=torch.float64, device="cuda")
        sc.transmittance_device(d_rays.data_ptr(), len(rays), d_out2.data_ptr(), t_min=0.1, t_max=5.0, stream=s.cuda_stream)
    s.synchronize()
    assert np.array_equal(d_out.cpu().numpy(), want)
    assert np.array_equal(d_out2.cpu().numpy(), want_scalar)
    assert st.segments == len(rays) and st.kernel_launches == 2 and st.ms_total > 0
    _, occ = sc.occluded(rays, t_min=0.1, t_max=t_max, flags=rt.RT_OPT_COUNT)
    assert st.node_visits >= occ.node_visits and st.prim_tests >= occ.prim_tests and st.prim_tests > occ.prim_tests


@pytest.mark.gpu
@pytest.mark.parametrize("knobs", [
    {"RT2025_FIFO_SLOTS": "0"}, {"RT2025_FIFO_SLOTS": "64", "RT2025_REFILL_MIN": "1"},
    {"RT2025_PARK_LEAVES": "0"}, {"RT2025_PARK_LEAVES": "1"},
])
def test_every_traversal_mode_gives_the_same_answer(gpu, rt, orc, monkeypatch, knobs):
    """The traversal knobs of the occlusion pass change when a lane stops, never what it finds."""
    for k, v in knobs.items():
        monkeypatch.setenv(k, v)
    rng = np.random.default_rng(5)
    o, d, t = random_rays(rng, 20000)
    for hs, rays in ((rt.named_scene("book2_final", seed=7, params=[48, 9, 20]), rt.make_rays(o * 40 + 250, d, t)),
                     (random_graph_scene(rt, 13, n_prims=90, with_media=True), rt.make_rays(o, d, t))):
        sc, osc = rt.Scene(hs), TransmittanceOracle(hs)
        t_max = rng.uniform(0.0, 30.0, len(rays))
        assert_same_transmittance(sc.transmittance(rays)[0], osc.transmittance(rays))
        assert_same_transmittance(sc.transmittance(rays, t_max=t_max)[0], osc.transmittance(rays, t_max=t_max))
        sc.close()
