"""The occlusion (any-hit) query, rt_occluded / rt_occluded_device.

For ray i, with t_max_i the per-ray bound or the scalar one, out[i] = 1 iff some surface primitive has a hit t with
Interval::contains(t_min, t_max_i, t).  The primitive tests are the reference's binary64 arithmetic and box culling is
conservative, so the answer is exactly

    closest_hit(ray, t_min, inf).prim_id != RT_NONE and closest_hit(...).t <= t_max_i

and every check below is bit-exact: against the oracle, the committed golden hits and the product's own closest hit."""
import ctypes as C
import os

import numpy as np
import pytest

from scenes_util import final_reduced_scene, random_graph_scene, random_rays

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
NAMED = {
    "book2_final": ("book2_final", 7, [32, 4, 12]),
    "cornell_glass": ("cornell_glass", 7, [32, 4, 12]),
    "book1_final": ("book1_final", 7, [48, 4, 12]),
}


@pytest.fixture(autouse=True, params=["by_size", "four_wide", "binary"])
def tree_variant(request, monkeypatch):
    """Every test runs on the tree rt_scene_create picks by size, on the four-wide collapse forced and on the binary tree
    forced, so that each kernel variant the occlusion query shares with closest hit is exercised."""
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


def expected(rt, hits, t_max):
    """The occlusion answer implied by closest hits on [t_min, inf)."""
    return (hits["prim_id"] != rt.RT_NONE) & (hits["t"] <= t_max)


def soup_rays(rt, rng, n):
    """Half primary rays from a pinhole in front of the unit cube, half incoherent rays from inside it."""
    o = np.concatenate([np.tile([0.5, 0.5, -2.0], (n // 2, 1)), rng.uniform(0, 1, (n // 2, 3))])
    tgt = rng.uniform(-0.2, 1.2, (n // 2, 3))
    tgt[:, 2] = 0.0
    d = np.concatenate([tgt - o[: n // 2], rng.normal(size=(n // 2, 3))])
    return rt.make_rays(o, d, rng.uniform(0, 1, n))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["book2_final", "cornell_glass", "book1_final", "random_graph", "final_reduced"])
def test_occlusion_matches_golden(gpu, rt, name):
    fx = np.load(os.path.join(GOLDEN, name + ".npz"))
    sc = rt.Scene(golden_scene(rt, name))
    got, st = sc.occluded(fx["rays"])
    assert got.dtype == np.bool_
    assert np.array_equal(got, fx["hits"]["prim_id"] != rt.RT_NONE)
    assert st.kernel_launches == 1 and st.segments == len(got)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_occlusion_matches_oracle_on_random_graphs(gpu, rt, orc, seed):
    """Transforms, lists, BVHs and media (which never occlude)."""
    hs = random_graph_scene(rt, seed, n_prims=120, with_media=True)
    sc, osc = rt.Scene(hs), orc.OracleScene(hs)
    rng = np.random.default_rng(seed)
    o, d, t = random_rays(rng, 30000)
    rays = rt.make_rays(o, d, t)
    want = osc.closest_hit(rays, mode=0)
    hit = want["prim_id"] != rt.RT_NONE
    assert 0.2 < hit.mean() < 0.95
    assert np.array_equal(sc.occluded(rays)[0], hit)
    assert np.array_equal(sc.occluded(rays, t_min=0.5, t_max=7.0)[0], osc.closest_hit(rays, t_min=0.5, t_max=7.0, mode=0)["prim_id"] != rt.RT_NONE)

    # per-ray t_max around the closest hit t*: t* itself is inside, the next double below is not
    t_star = np.where(hit, want["t"], 1.0)
    miss_tmax = rng.uniform(0.0, 20.0, len(rays))
    for tm, ans in ((t_star, hit), (np.nextafter(t_star, -np.inf), np.zeros_like(hit))):
        got, _ = sc.occluded(rays, t_max=np.where(hit, tm, miss_tmax))
        assert np.array_equal(got, ans)
    for scale in (0.5, 2.0):
        tm = np.where(hit, scale * t_star, miss_tmax)
        got, _ = sc.occluded(rays, t_max=tm)
        assert np.array_equal(got, expected(rt, want, tm))

    # empty intervals: a NaN bound or t_max_i < t_min
    tm = np.where(np.arange(len(rays)) % 2 == 0, np.nan, 0.25)
    assert not sc.occluded(rays, t_min=0.5, t_max=tm)[0].any()
    assert not sc.occluded(rays, t_min=float("nan"))[0].any()
    assert not sc.occluded(rays, t_min=3.0, t_max=2.0)[0].any()


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["tri_soup", "sphere_soup"])
def test_soup_occlusion_matches_oracle(gpu, rt, orc, shape):
    """Config 5 at 200k primitives: the four-wide global tree and the Transform-free single-kind variants."""
    hs = rt.named_scene(shape, seed=5, params=[200_000])
    sc, osc = rt.Scene(hs), orc.OracleScene(hs)
    n = 60_000
    rays = soup_rays(rt, np.random.default_rng(3), n)
    want = osc.closest_hit(rays, mode=0)
    hit = want["prim_id"] != rt.RT_NONE
    assert hit.mean() > 0.3
    got, _ = sc.occluded(rays)
    assert np.array_equal(got, hit)
    counted, st = sc.occluded(rays, flags=rt.RT_OPT_COUNT)
    assert np.array_equal(counted, got)
    _, ch = sc.closest_hit(rays, flags=rt.RT_OPT_COUNT)
    assert 0 < st.node_visits <= ch.node_visits and 0 < st.prim_tests <= ch.prim_tests


@pytest.mark.gpu
@pytest.mark.parametrize("knobs", [
    {"RT2025_FIFO_SLOTS": "0"}, {"RT2025_FIFO_SLOTS": "32", "RT2025_REFILL_MIN": "16"}, {"RT2025_FIFO_SLOTS": "64", "RT2025_REFILL_MIN": "1"},
    {"RT2025_PARK_LEAVES": "0"}, {"RT2025_PARK_LEAVES": "1"},
])
def test_every_traversal_mode_gives_the_same_answer(gpu, rt, orc, monkeypatch, knobs):
    """Direct refill vs prepared-ray FIFOs, the refill threshold and postponed leaves change when a lane stops, never what it finds."""
    for k, v in knobs.items():
        monkeypatch.setenv(k, v)
    rng = np.random.default_rng(5)
    o, d, t = random_rays(rng, 20000)
    for hs, rays in ((rt.named_scene("book2_final", seed=7, params=[48, 9, 20]), rt.make_rays(o * 40 + 250, d, t)),
                     (random_graph_scene(rt, 13, n_prims=90, with_media=True), rt.make_rays(o, d, t)),
                     (rt.named_scene("tri_soup", seed=9, params=[60_000]), soup_rays(rt, rng, 20000))):
        sc, osc = rt.Scene(hs), orc.OracleScene(hs)
        want = osc.closest_hit(rays, mode=0)
        t_max = np.where(np.arange(len(rays)) % 3 == 0, np.inf, rng.uniform(0.0, 2.0, len(rays)) * np.where(np.isinf(want["t"]), 1.0, want["t"]))
        assert np.array_equal(sc.occluded(rays)[0], want["prim_id"] != rt.RT_NONE)
        assert np.array_equal(sc.occluded(rays, t_max=t_max)[0], expected(rt, want, t_max))
        sc.close()


@pytest.mark.gpu
def test_device_lbvh_build_gives_the_same_answer(gpu, rt, orc):
    for shape in ("tri_soup", "sphere_soup"):
        hs = rt.named_scene(shape, seed=9, params=[60_000])
        sc, osc = rt.Scene(hs, flags=rt.RT_BUILD_DEVICE_LBVH), orc.OracleScene(hs)
        assert sc.info().n_nodes == 60_000 - 1
        rays = soup_rays(rt, np.random.default_rng(4), 40_000)
        want = osc.closest_hit(rays, mode=0)
        t_max = np.where(np.isinf(want["t"]), 1.0, want["t"])
        assert np.array_equal(sc.occluded(rays)[0], want["prim_id"] != rt.RT_NONE)
        assert np.array_equal(sc.occluded(rays, t_max=t_max)[0], want["prim_id"] != rt.RT_NONE)
        assert not sc.occluded(rays, t_max=np.nextafter(t_max, -np.inf))[0].any()


@pytest.mark.gpu
def test_moving_sphere_and_time(gpu, rt, orc):
    b = rt.Builder(1)
    hs = b.finish(b.list([b.sphere_moving([0, 0, 0], [4, 0, 0], 1.0, b.empty())]))
    sc, osc = rt.Scene(hs), orc.OracleScene(hs)
    # straight down the z axis: the sphere is there at time 0 and 4 units away at time 1
    rays = rt.make_rays([[0, 0, 6], [0, 0, 6]], [[0, 0, -1], [0, 0, -1]], [0.0, 1.0])
    assert sc.occluded(rays)[0].tolist() == [True, False]
    rng = np.random.default_rng(2)
    o = np.column_stack([rng.uniform(-2, 6, 4000), rng.uniform(-1.5, 1.5, 4000), np.full(4000, 6.0)])
    rays = rt.make_rays(o, np.tile([0, 0, -1.0], (4000, 1)), rng.uniform(0, 1, 4000))
    want = osc.closest_hit(rays, mode=0)
    assert np.array_equal(sc.occluded(rays)[0], want["prim_id"] != rt.RT_NONE)
    assert (want["prim_id"] == 0).sum() > 300


@pytest.mark.gpu
def test_ellipsoids_and_nested_transforms(gpu, rt, orc):
    b = rt.Builder(9)
    m = b.empty()
    e1 = b.transform(b.sphere([0, 0, 0], 1.0, m), offset=[-2, 0, 0], quat=b.quat_axis_angle([0, 0, 1], 30.0), scale=[2.0, 0.5, 1.0])
    inner = b.transform(b.bvh([b.sphere([0, 0, 0], 0.7, m), b.quad([-1, -1, 1], [2, 0, 0], [0, 2, 0], m),
                               b.triangle([0, 1, -1], [1, 0, 0], [0, 1, 1], m)]), offset=[0.5, 0, 0], scale=[1, 2, 1])
    e2 = b.transform(b.list([inner, b.sphere_moving([0, -2, 0], [1, -2, 0], 0.5, m)]), offset=[2.5, 0.5, 0],
                     quat=b.quat_axis_angle([1, 1, 0], 50.0), scale=[0.8, 0.8, 1.6])
    hs = b.finish(b.list([e1, e2]))
    sc, osc = rt.Scene(hs), orc.OracleScene(hs)
    o, d, t = random_rays(np.random.default_rng(4), 40000, extent=5.0)
    rays = rt.make_rays(o, d, t)
    want = osc.closest_hit(rays, mode=0)
    hit = want["prim_id"] != rt.RT_NONE
    assert hit.sum() > 2000 and len(set(want["inst_id"][hit].tolist())) >= 2
    t_star = np.where(hit, want["t"], np.inf)
    assert np.array_equal(sc.occluded(rays)[0], hit)
    assert np.array_equal(sc.occluded(rays, t_max=t_star)[0], hit)
    assert not sc.occluded(rays, t_max=np.nextafter(t_star, -np.inf))[0][hit].any()


@pytest.mark.gpu
def test_edge_cases(gpu, rt, orc):
    # zero rays
    b = rt.Builder(1)
    sc = rt.Scene(b.finish(b.list([b.sphere([0, 0, 0], 1.0, b.empty())])))
    got, st = sc.occluded(np.zeros(0, dtype=rt.rt_ray_dtype))
    assert len(got) == 0 and st.segments == 0
    got, st = sc.occluded(np.zeros(0, dtype=rt.rt_ray_dtype), t_max=np.zeros(0))
    assert len(got) == 0
    o, d, t = random_rays(np.random.default_rng(1), 5000)
    rays = rt.make_rays(o, d, t)
    # an empty world, and a world of media only: nothing occludes
    b = rt.Builder(1)
    sc = rt.Scene(b.finish(b.list([])))
    assert not sc.occluded(rays)[0].any()
    b = rt.Builder(1)
    fog = b.medium(b.sphere([0, 0, 0], 3.0, b.empty()), 5.0, b.solid(1, 1, 1))
    box = b.medium(b.box([-6, -6, -6], [6, 6, 6], b.empty()), 0.5, b.solid(1, 1, 1))
    sc = rt.Scene(b.finish(b.list([fog, box])))
    assert not sc.occluded(rays)[0].any()
    # axis-parallel, zero and degenerate directions, a NaN origin: the same answer as closest hit
    b = rt.Builder(1)
    m = b.empty()
    hs = b.finish(b.list([b.bvh([b.sphere([0, 0, 0], 1.0, m), b.quad([-1, -1, -3], [2, 0, 0], [0, 2, 0], m),
                                 b.triangle([-1, -1, 3], [2, 0, 0], [0, 2, 0], m), b.sphere([4, 0, 0], 0.5, m)])]))
    sc, osc = rt.Scene(hs), orc.OracleScene(hs)
    o = [[0, 0, 5], [0, 0, 5], [-5, 0, 0], [0, 0, 0], [0, 0, 5], [float("nan"), 0, 5], [0.25, 0.25, -10], [0, 0, 5]]
    d = [[0, 0, -1], [0, 0, 1], [1, 0, 0], [0, 1, 0], [0, 0, 0], [0, 0, -1], [0, 0, 1e-30], [0, 0, -1e300]]
    rays = rt.make_rays(o, d)
    ch, _ = sc.closest_hit(rays)
    assert np.array_equal(sc.occluded(rays)[0], ch["prim_id"] != rt.RT_NONE)
    assert np.array_equal(sc.occluded(rays)[0], osc.closest_hit(rays, mode=0)["prim_id"] != rt.RT_NONE)


@pytest.mark.gpu
def test_device_entry_equals_host_entry(gpu, rt):
    import torch
    hs = random_graph_scene(rt, 4, n_prims=150, with_media=True)
    sc = rt.Scene(hs)
    rng = np.random.default_rng(6)
    o, d, t = random_rays(rng, 50001)
    rays = rt.make_rays(o, d, t)
    t_max = rng.uniform(0.0, 12.0, len(rays))
    want, _ = sc.occluded(rays, t_min=0.1, t_max=t_max)
    want_scalar, _ = sc.occluded(rays, t_min=0.1, t_max=5.0)
    d_rays = torch.from_numpy(rays.view(np.float64).reshape(-1, 7).copy()).cuda()
    d_tmax = torch.from_numpy(t_max).cuda()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        d_out = torch.full((len(rays),), 7, dtype=torch.uint8, device="cuda")
        st = sc.occluded_device(d_rays.data_ptr(), len(rays), d_out.data_ptr(), d_tmax.data_ptr(), t_min=0.1, flags=rt.RT_OPT_COUNT,
                                stream=s.cuda_stream)
        d_out2 = torch.full((len(rays),), 7, dtype=torch.uint8, device="cuda")
        sc.occluded_device(d_rays.data_ptr(), len(rays), d_out2.data_ptr(), t_min=0.1, t_max=5.0, stream=s.cuda_stream)
    s.synchronize()
    assert np.array_equal(d_out.cpu().numpy(), want.view(np.uint8))
    assert np.array_equal(d_out2.cpu().numpy(), want_scalar.view(np.uint8))
    assert st.segments == len(rays) and st.kernel_launches == 1 and st.node_visits > 0 and st.prim_tests > 0 and st.ms_total > 0


def test_null_arguments_are_refused_without_a_device(rt):
    L = rt.product_lib()
    ray = np.zeros(1, dtype=rt.rt_ray_dtype)
    out = np.zeros(1, dtype=np.uint8)
    fake_scene = C.c_void_p(ray.ctypes.data)  # never dereferenced: the arguments are checked first
    st = rt.rt_stats()
    for scene, rays, o in ((None, ray.ctypes.data, out.ctypes.data), (fake_scene, None, out.ctypes.data), (fake_scene, ray.ctypes.data, None)):
        assert L.rt_occluded(scene, rays, None, 1, 1e-8, float("inf"), 0, o, C.byref(st)) == -1
        assert "null" in L.rt_last_error().decode()
        assert L.rt_occluded_device(scene, rays, None, 1, 1e-8, float("inf"), 0, o, None, C.byref(st)) == -1
