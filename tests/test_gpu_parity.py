"""GPU parity tests: the CUDA core (through the C ABI) against the oracle and the committed
golden fixtures.  Integer outputs (primitive / instance ids) must be bit-exact; hit distances
bit-exact (the north star allows 1e-5 relative); same-seed images within 1e-6 relative for all
but a vanishing fraction of pixels (a path whose branch flips on a last-bit libm difference)."""
import os

import numpy as np
import pytest

from scenes_util import compare_hits, final_reduced_scene, materials_scene, random_graph_scene, random_rays

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True, params=["by_size", "four_wide", "binary"])
def tree_variant(request, monkeypatch):
    """Every test of this module runs three times: with the tree rt_scene_create picks by scene size (the four-wide collapse
    in shared memory for the smallest scenes, the binary tree in shared memory for book-sized ones, the four-wide tree in
    global memory for the soups), with the four-wide collapse forced and with the binary tree forced, so that empty worlds,
    single primitives, ties, Transforms, media and degenerate rays are all checked on every traversal variant."""
    if request.param == "four_wide":
        monkeypatch.setenv("RT2025_WIDE_BVH", "1")
    elif request.param == "binary":
        monkeypatch.setenv("RT2025_WIDE_BVH", "0")
    return request.param
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

NAMED = {
    "book2_final": ("book2_final", 7, [32, 4, 12]),
    "cornell_glass": ("cornell_glass", 7, [32, 4, 12]),
    "book1_final": ("book1_final", 7, [48, 4, 12]),
}


def golden_scene(rt, name):
    if name == "random_graph":
        return random_graph_scene(rt, 11, n_prims=72, with_media=True, width=32, spp=4, depth=8)
    if name == "final_reduced":
        return final_reduced_scene(rt, width=96, spp=4, depth=12)
    n, seed, params = NAMED[name]
    return rt.named_scene(n, seed=seed, params=params)


def image_close(img, ref, frac_bad=2e-3, rel=1e-6):
    diff = np.abs(img - ref)
    bad = (diff > rel * (1 + np.abs(ref))).any(axis=2)
    assert bad.mean() <= frac_bad, f"{int(bad.sum())}/{bad.size} pixels differ (max {diff.max():.3e})"
    assert abs(img.mean() - ref.mean()) <= 1e-3 * ref.mean() + 1e-9


@pytest.mark.parametrize("name", ["book2_final", "cornell_glass", "book1_final", "random_graph", "final_reduced"])
def test_closest_hit_matches_golden(gpu, rt, name):
    fx = np.load(os.path.join(GOLDEN, name + ".npz"))
    sc = rt.Scene(golden_scene(rt, name))
    got, st = sc.closest_hit(fx["rays"])
    compare_hits(rt, got, fx["hits"])
    assert st.kernel_launches == 1


@pytest.mark.parametrize("name", ["book2_final", "cornell_glass", "book1_final", "random_graph", "final_reduced"])
def test_render_matches_golden_image(gpu, rt, name):
    fx = np.load(os.path.join(GOLDEN, name + ".npz"))
    sc = rt.Scene(golden_scene(rt, name))
    img, st = sc.render(seed=int(fx["render_seed"]))
    assert st.paths == int(fx["paths"])
    # an error marks a sample on which the reference would panic; the device stops a path whose
    # throughput is exactly zero, so it can only meet fewer of them than the full recursion
    assert int(st.errors) <= int(fx["errors"])
    image_close(img, fx["image"], frac_bad=5e-3)


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_closest_hit_matches_oracle_on_random_graphs(gpu, rt, orc, seed):
    hs = random_graph_scene(rt, seed, n_prims=120)
    sc, osc = rt.Scene(hs), orc.OracleScene(hs)
    assert np.array_equal(sc.ranks(), osc.ranks())
    rng = np.random.default_rng(seed)
    o, d, t = random_rays(rng, 30000)
    rays = rt.make_rays(o, d, t)
    got, _ = sc.closest_hit(rays)
    compare_hits(rt, got, osc.closest_hit(rays, mode=0))
    # a finite interval and a shifted t_min
    got, _ = sc.closest_hit(rays, t_min=0.5, t_max=7.0)
    compare_hits(rt, got, osc.closest_hit(rays, t_min=0.5, t_max=7.0, mode=0))


def test_closest_hit_on_a_tree_larger_than_shared_memory(gpu, rt, orc):
    """6000 primitives: the binary tree (about 5000 nodes) only partly fits in a traversal CTA's shared memory, so the forced-binary
    variant of this module walks the mixed shared / global-memory node loop in direct mode (book-sized trees are entirely in
    shared memory, the soups entirely in global memory), and the by-size variant the four-wide tree fed from the FIFOs."""
    hs = random_graph_scene(rt, 21, n_prims=6000, with_lights=False)
    sc, osc = rt.Scene(hs), orc.OracleScene(hs)
    assert np.array_equal(sc.ranks(), osc.ranks())
    o, d, t = random_rays(np.random.default_rng(21), 40000)
    rays = rt.make_rays(o, d, t)
    got, st = sc.closest_hit(rays, flags=rt.RT_OPT_COUNT)
    compare_hits(rt, got, osc.closest_hit(rays, mode=0))
    assert st.node_visits > 0 and st.prim_tests > 0
    img, _ = sc.render(seed=4)
    image_close(img, osc.render(seed=4)[0])


def test_ellipsoids_and_nested_transforms(gpu, rt, orc):
    # a Sphere under a non-uniform scale is an ellipsoid (shapes.rs:74-84); Transforms nest
    b = rt.Builder(9)
    m = b.empty()
    e1 = b.transform(b.sphere([0, 0, 0], 1.0, m), offset=[-2, 0, 0], quat=b.quat_axis_angle([0, 0, 1], 30.0), scale=[2.0, 0.5, 1.0])
    inner = b.transform(b.bvh([b.sphere([0, 0, 0], 0.7, m), b.quad([-1, -1, 1], [2, 0, 0], [0, 2, 0], m),
                               b.triangle([0, 1, -1], [1, 0, 0], [0, 1, 1], m)]), offset=[0.5, 0, 0], scale=[1, 2, 1])
    e2 = b.transform(b.list([inner, b.sphere_moving([0, -2, 0], [1, -2, 0], 0.5, m)]), offset=[2.5, 0.5, 0],
                     quat=b.quat_axis_angle([1, 1, 0], 50.0), scale=[0.8, 0.8, 1.6])
    e3 = b.transform(b.sphere([0, 0, 0], 1.0, m), offset=[0, 3, 0], scale=[-1.0, 1.0, 1.5])  # a mirroring scale
    hs = b.finish(b.list([e1, e2, e3]))
    sc, osc = rt.Scene(hs), orc.OracleScene(hs)
    rng = np.random.default_rng(4)
    o, d, t = random_rays(rng, 40000, extent=5.0)
    rays = rt.make_rays(o, d, t)
    got, _ = sc.closest_hit(rays)
    want = osc.closest_hit(rays, mode=0)
    compare_hits(rt, got, want)
    assert (want["prim_id"] != rt.RT_NONE).sum() > 2000
    assert len(set(want["inst_id"].tolist())) >= 4


def test_hits_are_bit_exact(gpu, rt, orc):
    # every primitive is intersected with the reference's own arithmetic: t is bit-identical
    hs = random_graph_scene(rt, 5, n_prims=150)
    sc, osc = rt.Scene(hs), orc.OracleScene(hs)
    rng = np.random.default_rng(5)
    o, d, t = random_rays(rng, 30000)
    rays = rt.make_rays(o, d, t)
    got, _ = sc.closest_hit(rays)
    want = osc.closest_hit(rays, mode=0)
    assert np.array_equal(got["prim_id"], want["prim_id"])
    assert np.array_equal(got["t"], want["t"])


def test_tie_rules(gpu, rt, orc):
    # hits.rs:42 first child wins; bvh.rs:78-84 right child wins; both through the rank order
    for container, winner in (("list", 0), ("bvh", 1)):
        b = rt.Builder(1)
        m = b.empty()
        q = [b.quad([-1, -1, 0], [2, 0, 0], [0, 2, 0], m) for _ in range(2)]
        inner = b.list(q) if container == "list" else b.list([b.bvh(q)])
        hs = b.finish(inner)
        rays = rt.make_rays([[0.2, 0.3, 5], [0.9, -0.9, 2]], [[0, 0, -1], [0, 0, -1]])
        got, _ = rt.Scene(hs).closest_hit(rays)
        assert got["prim_id"].tolist() == [winner, winner]
        assert got["t"].tolist() == [5.0, 2.0]
    # five overlapping coplanar quads in a BVH: the median split decides (see the oracle test)
    b = rt.Builder(1)
    m = b.empty()
    xs = [3.0, 0.0, 4.0, 1.0, 2.0]
    hs = b.finish(b.list([b.bvh([b.quad([x, -1, 0], [10, 0, 0], [0, 2, 0], m) for x in xs])]))
    sc, osc = rt.Scene(hs), orc.OracleScene(hs)
    rng = np.random.default_rng(0)
    o = np.column_stack([rng.uniform(-1, 15, 2000), rng.uniform(-1.5, 1.5, 2000), np.full(2000, 5.0)])
    rays = rt.make_rays(o, np.tile([0, 0, -1.0], (2000, 1)))
    got, _ = sc.closest_hit(rays)
    compare_hits(rt, got, osc.closest_hit(rays, mode=0))
    assert len(set(got["prim_id"].tolist())) >= 5


def test_edge_cases(gpu, rt, orc):
    # empty world
    b = rt.Builder(1)
    hs = b.finish(b.list([]), width=8, spp=1, background=b.solid(0.25, 0.5, 1.0))
    sc = rt.Scene(hs)
    got, _ = sc.closest_hit(rt.make_rays([[0, 0, 0]], [[0, 0, 1]]))
    assert got["prim_id"][0] == rt.RT_NONE and np.isinf(got["t"][0])
    img, st = sc.render(seed=1)
    assert np.array_equal(img, np.broadcast_to([0.25, 0.5, 1.0], img.shape)) and st.segments == st.paths
    # zero rays
    got, _ = sc.closest_hit(np.zeros(0, dtype=rt.rt_ray_dtype))
    assert len(got) == 0
    # axis-parallel, zero-component and degenerate directions; NaN origin never hits
    b = rt.Builder(1)
    m = b.empty()
    hs = b.finish(b.list([b.bvh([b.sphere([0, 0, 0], 1.0, m), b.quad([-1, -1, -3], [2, 0, 0], [0, 2, 0], m),
                                 b.triangle([-1, -1, 3], [2, 0, 0], [0, 2, 0], m), b.sphere([4, 0, 0], 0.5, m)])]))
    sc, osc = rt.Scene(hs), orc.OracleScene(hs)
    o = [[0, 0, 5], [0, 0, 5], [-5, 0, 0], [0, 0, 0], [0, 0, 5], [float("nan"), 0, 5], [0.25, 0.25, -10], [0, 0, 5]]
    d = [[0, 0, -1], [0, 0, 1], [1, 0, 0], [0, 1, 0], [0, 0, 0], [0, 0, -1], [0, 0, 1e-30], [0, 0, -1e300]]
    rays = rt.make_rays(o, d)
    got, _ = sc.closest_hit(rays)
    want = osc.closest_hit(rays, mode=0)
    assert np.array_equal(got["prim_id"], want["prim_id"])
    hit = want["prim_id"] != rt.RT_NONE
    assert np.array_equal(got["t"][hit], want["t"][hit])


def test_moving_sphere_and_time(gpu, rt, orc):
    b = rt.Builder(1)
    hs = b.finish(b.list([b.sphere_moving([0, 0, 0], [4, 0, 0], 1.0, b.empty())]))
    sc, osc = rt.Scene(hs), orc.OracleScene(hs)
    rng = np.random.default_rng(2)
    o = np.column_stack([rng.uniform(-2, 6, 4000), rng.uniform(-1.5, 1.5, 4000), np.full(4000, 6.0)])
    rays = rt.make_rays(o, np.tile([0, 0, -1.0], (4000, 1)), rng.uniform(0, 1, 4000))
    got, _ = sc.closest_hit(rays)
    want = osc.closest_hit(rays, mode=0)
    assert np.array_equal(got["prim_id"], want["prim_id"]) and np.array_equal(got["t"], want["t"])
    assert (want["prim_id"] == 0).sum() > 300


@pytest.mark.parametrize("name,seed,params", [("book2_final", 3, [64, 9, 40]), ("cornell_glass", 3, [64, 9, 50]),
                                              ("book1_final", 3, [96, 9, 50])])
def test_same_seed_image_matches_oracle(gpu, rt, orc, name, seed, params):
    hs = rt.named_scene(name, seed=seed, params=params)
    sc, osc = rt.Scene(hs), orc.OracleScene(hs)
    img, st = sc.render(seed=17)
    ref, ost = osc.render(seed=17)
    assert st.paths == ost.paths and st.errors == ost.errors
    image_close(img, ref)


def test_materials_textures_and_lights_vs_oracle(gpu, rt, orc):
    hs = materials_scene(rt)
    sc, osc = rt.Scene(hs), orc.OracleScene(hs)
    img, st = sc.render(seed=23)
    ref, ost = osc.render(seed=23)
    assert st.paths == ost.paths
    assert int(st.errors) <= int(ost.errors)
    image_close(img, ref, frac_bad=5e-3)


def test_media_including_transformed_boundaries(gpu, rt, orc):
    b = rt.Builder(4)
    white = b.lambertian(b.solid(0.7, 0.7, 0.7))
    floor = b.quad([-8, -2, -8], [16, 0, 0], [0, 0, 16], white)
    light = b.quad([-2, 6, -2], [4, 0, 0], [0, 0, 4], b.diffuse_light(b.solid(9, 9, 9)))
    fog_box = b.transform(b.box([-1, -1, -1], [1, 1, 1], b.empty()), offset=[-2, 0, 0], quat=b.quat_axis_angle([0, 1, 0], 30.0))
    m1 = b.medium(fog_box, 0.9, b.solid(0.9, 0.9, 0.9))
    m2 = b.transform(b.medium(b.sphere([0, 0, 0], 1.0, b.empty()), 1.5, b.solid(0.2, 0.3, 0.9)), offset=[2, 0, 0], scale=[1.5, 1.5, 1.5])
    m3 = b.medium(b.sphere([0, 0, 0], 30.0, b.empty()), 0.01, b.solid(1, 1, 1))
    world = b.list([floor, light, m1, m2, m3, b.sphere([0, 0, -3], 1.0, b.dielectric(b.solid(1, 1, 1), 1.5))])
    lights = b.list([b.quad([-2, 6, -2], [4, 0, 0], [0, 0, 4], b.empty())])
    hs = b.finish(world, lights, width=48, spp=16, max_depth=12, vfov=45, look_from=(0, 2, 10), look_at=(0, 0, 0))
    sc, osc = rt.Scene(hs), orc.OracleScene(hs)
    assert sc.info().n_media == 3
    img, st = sc.render(seed=5)
    ref, ost = osc.render(seed=5)
    assert st.paths == ost.paths and st.errors == ost.errors
    image_close(img, ref, frac_bad=5e-3)


def test_partitions_sample_ranges_and_capacity(gpu, rt):
    # multi-GPU decomposition (rt_render_opts.part_*) and stratum ranges must add up to the whole,
    # and the answer must not depend on how many paths are in flight
    hs = rt.named_scene("book2_final", seed=5, params=[72, 9, 20])
    sc = rt.Scene(hs)
    whole, st = sc.render(seed=3)
    parts = [sc.render(seed=3, part_index=k, part_count=3)[0] for k in range(3)]
    nz = [(p != 0).any(axis=2) for p in parts]
    assert not (nz[0] & nz[1]).any() and not (nz[1] & nz[2]).any()
    assert np.allclose(sum(parts), whole, rtol=1e-12, atol=1e-14)
    halves = sc.render(seed=3, sample_begin=0, sample_end=5)[0] + sc.render(seed=3, sample_begin=5, sample_end=9)[0]
    assert np.allclose(halves, whole, rtol=1e-12, atol=1e-14)
    small, st2 = sc.render(seed=3, max_paths_in_flight=4096)
    assert np.allclose(small, whole, rtol=1e-12, atol=1e-14)
    assert st2.paths == st.paths and st2.segments == st.segments and st2.iterations > st.iterations
    f32, _ = sc.render(seed=3, accum_type=rt.RT_ACCUM_F32)
    assert f32.dtype == np.float32 and np.allclose(f32, whole, rtol=1e-6, atol=1e-7)
    other, _ = sc.render(seed=4)
    assert not np.allclose(other, whole)


def test_media_order_does_not_change_the_image(gpu, rt, orc):
    """Scenes whose media all have sphere boundaries sample them BEFORE extend (which then only looks for surfaces up to
    the scatter point, with the medium's t and tie rank as the incumbent); the classic order samples them after.  Same
    candidates, same winner: images and segment counts must agree, also where a medium shares a boundary with a surface."""
    for hs in (rt.named_scene("book2_final", seed=7, params=[40, 9, 12]),
               random_graph_scene(rt, 8, n_prims=60, with_media=True, width=24, spp=9, depth=6)):
        sc = rt.Scene(hs)
        a, sa = sc.render(seed=5)
        b, sb = sc.render(seed=5, classic_media_order=True)
        image_close(a, b, frac_bad=0.0, rel=1e-9)
        assert sa.segments == sb.segments and sa.errors == sb.errors
        ref, _ = orc.OracleScene(hs).render(seed=5)
        image_close(a, ref)
    # a surface exactly at the scatter distance cannot be constructed on purpose, but a medium inside a glass shell
    # exercises "surface nearer than the scatter point" and "scatter point nearer" on every path
    b = rt.Builder(3)
    shell = b.sphere([0, 0, 0], 1.0, b.dielectric(b.solid(1, 1, 1), 1.5))
    fog = b.medium(b.sphere([0, 0, 0], 0.999, b.empty()), 1.5, b.solid(0.8, 0.3, 0.2))
    floor = b.quad([-4, -1.2, -4], [8, 0, 0], [0, 0, 8], b.lambertian(b.solid(0.6, 0.6, 0.6)))
    hs = b.finish(b.list([shell, fog, floor]), width=32, spp=16, max_depth=12, vfov=35, look_from=(0, 1, 5), background=b.solid(0.7, 0.8, 1.0))
    sc = rt.Scene(hs)
    a, sa = sc.render(seed=2)
    c, sc_ = sc.render(seed=2, classic_media_order=True)
    image_close(a, c, frac_bad=0.0, rel=1e-9)
    image_close(a, orc.OracleScene(hs).render(seed=2)[0])
    assert sa.segments == sc_.segments


def _walk_scene(rt, variant):
    """An optically thick medium (radius x density >= 1) whose scatter points go to the random-walk kernel."""
    b = rt.Builder(11)
    floor = b.quad([-6, -1.5, -6], [12, 0, 0], [0, 0, 12], b.lambertian(b.solid(0.6, 0.6, 0.6)))
    lamp = b.quad([-1.5, 4, -1.5], [3, 0, 0], [0, 0, 3], b.diffuse_light(b.solid(12, 12, 12)))
    lights = b.list([b.quad([-1.5, 4, -1.5], [3, 0, 0], [0, 0, 3], b.empty())])
    things = [floor, lamp]
    if variant == "surfaces_inside":  # a metal ball and a quad INSIDE the boundary: the walk must see them (entry leaves)
        things += [b.medium(b.sphere([0, 0, 0], 1.2, b.empty()), 4.0, b.solid(0.3, 0.5, 0.9)),
                   b.sphere([0.3, 0.1, 0.0], 0.35, b.metal([0.9, 0.8, 0.7], 0.05)),
                   b.quad([-0.9, -0.4, -0.5], [0.6, 0, 0], [0, 0.5, 0.3], b.lambertian(b.solid(0.8, 0.2, 0.2))),
                   b.sphere([0, 0, 0], 1.2, b.dielectric(b.solid(1, 1, 1), 1.5))]
    elif variant == "overlapping":  # two thick media that overlap, and a thin fog around everything
        things += [b.medium(b.sphere([-0.5, 0, 0], 1.0, b.empty()), 3.0, b.solid(0.9, 0.4, 0.3)),
                   b.medium(b.sphere([0.5, 0, 0], 1.0, b.empty()), 5.0, b.solid(0.3, 0.9, 0.4)),
                   b.medium(b.sphere([0, 0, 0], 40.0, b.empty()), 0.01, b.solid(1, 1, 1))]
    elif variant == "many_neighbours":  # more overlapping leaves than entry slots: traversal from the world root
        things += [b.medium(b.sphere([0, 0, 0], 1.2, b.empty()), 4.0, b.solid(0.3, 0.5, 0.9))]
        for k in range(24):
            things.append(b.sphere([0.8 * np.cos(k), 0.5 * np.sin(2.0 * k), 0.8 * np.sin(k)], 0.12, b.lambertian(b.solid(0.2 + 0.03 * k, 0.5, 0.5))))
    else:  # "moving_transformed": a moving boundary below a rotated, scaled Transform
        things += [b.transform(b.medium(b.sphere_moving([0, 0, 0], [0.3, 0.1, 0], 1.0, b.empty()), 3.0, b.solid(0.7, 0.7, 0.2)),
                               offset=[0.2, 0, 0], quat=b.quat_axis_angle([0, 1, 1], 25.0), scale=[1.2, 1.2, 1.2]),
                   b.sphere([0.2, 0, 0], 0.3, b.lambertian(b.solid(0.2, 0.8, 0.8)))]
    return b.finish(b.list(things), lights, width=40, spp=16, max_depth=24, vfov=35, look_from=(0, 1.5, 6), background=b.solid(0.5, 0.6, 0.8))


@pytest.mark.parametrize("variant", ["surfaces_inside", "overlapping", "many_neighbours", "moving_transformed"])
def test_random_walk_kernel_vs_wavefront_and_oracle(gpu, rt, orc, variant, monkeypatch):
    """k_walk keeps a path inside an optically thick medium in registers from scatter point to scatter point.  The draws are
    addressed, so the image, the segment count and the error count must be those of the plain wavefront (walk switched
    off), with and without the entry-leaf shortcut, and the image must match the oracle."""
    hs = _walk_scene(rt, variant)
    monkeypatch.setenv("RT2025_TAIL_PATHS", "0")  # these frames are small enough for k_tail to finish them after one iteration
    sc = rt.Scene(hs)
    a, sa = sc.render(seed=9)  # (a queue this short cuts every walk after four segments: the drain rule of k_walk)
    assert sa.walk_segments > 0
    monkeypatch.setenv("RT2025_WALK_DRAIN_QUEUE", "0")  # walks of any length
    a2, sa2 = sc.render(seed=9)
    assert sa2.walk_segments > sa.walk_segments and sa2.segments == sa.segments and sa2.errors == sa.errors
    image_close(a2, a, frac_bad=0.0, rel=1e-9)
    monkeypatch.setenv("RT2025_WALK_NO_ENTRIES", "1")
    b_, sb = rt.Scene(hs).render(seed=9)
    monkeypatch.delenv("RT2025_WALK_NO_ENTRIES")
    monkeypatch.setenv("RT2025_WALK_MIN_DEPTH", "0")
    c, sc_ = rt.Scene(hs).render(seed=9)
    monkeypatch.delenv("RT2025_WALK_MIN_DEPTH")
    assert sc_.walk_segments == 0 and sb.walk_segments == sa2.walk_segments
    assert sa.segments == sb.segments == sc_.segments and sa.errors == sb.errors == sc_.errors
    assert sc_.iterations >= sa.iterations
    image_close(a, c, frac_bad=0.0, rel=1e-9)
    image_close(b_, c, frac_bad=0.0, rel=1e-9)
    ref, ost = orc.OracleScene(hs).render(seed=9)
    image_close(a, ref)


def test_binning_does_not_change_the_image(gpu, rt):
    import ctypes as C
    hs = rt.named_scene("book2_final", seed=5, params=[64, 4, 20])
    sc = rt.Scene(hs)
    a, _ = sc.render(seed=3)
    o = sc.render_opts(seed=3)
    o.reserved[0] = 1  # material binning off
    img = np.zeros_like(a)
    st = rt.rt_stats()
    assert sc.L.rt_render(sc.h, C.byref(hs.camera), C.byref(o), img.ctypes.data, C.byref(st)) == 0
    assert np.allclose(img, a, rtol=1e-12, atol=1e-14)


def test_tonemap_matches_oracle(gpu, rt, orc):
    rng = np.random.default_rng(1)
    img = rng.gamma(0.7, 0.8, (40, 50, 3))
    img[0, 0] = [0, 1, 0.0031308]
    for toon in (0, 1):
        got = rt.tonemap(img, toon)
        want = orc.tonemap(img, toon)
        assert np.abs(got.astype(int) - want.astype(int)).max() <= 1  # pow() last-bit differences only
        assert (got != want).mean() < 1e-3
    with pytest.raises(rt.RtError):
        bad = img.copy()
        bad[3, 3, 1] = np.nan
        rt.tonemap(bad)


def test_full_size_properties_book2(gpu, rt):
    """Config 2 at BASELINE.json's full resolution (one stratum per pixel-sample block): properties
    that do not need the oracle — energy is finite and non-negative, the light is seen, stats add up."""
    hs = rt.named_scene("book2_final", seed=7, params=[800, 1000, 40])
    sc = rt.Scene(hs)
    img, st = sc.render(seed=1, sample_begin=0, sample_end=16, accum_type=rt.RT_ACCUM_F32)
    assert st.paths == 800 * 800 * 16 and st.errors == 0
    assert np.isfinite(img).all() and (img >= 0).all()
    full_scale = 961 / 16  # accum holds sum * pixel_sample_scale
    mean = img.mean() * full_scale
    assert 0.2 < mean < 1.0
    assert img.max() * full_scale > 5.0  # the 7,7,7 light quad is visible
    assert 3.0 < st.segments / st.paths < 6.0


@pytest.mark.parametrize("shape", ["tri_soup", "sphere_soup"])
def test_soup_closest_hit_matches_oracle(gpu, rt, orc, shape):
    """Config 5 at a size the oracle finishes in seconds: 200k primitives, primary + incoherent rays."""
    hs = rt.named_scene(shape, seed=5, params=[200_000])
    sc, osc = rt.Scene(hs), orc.OracleScene(hs)
    assert np.array_equal(sc.ranks(), osc.ranks())
    rng = np.random.default_rng(3)
    n = 60_000
    o = np.concatenate([np.tile([0.5, 0.5, -2.0], (n // 2, 1)), rng.uniform(0, 1, (n // 2, 3))])
    tgt = rng.uniform(-0.2, 1.2, (n // 2, 3))
    tgt[:, 2] = 0.0
    d = np.concatenate([tgt - o[: n // 2], rng.normal(size=(n // 2, 3))])
    rays = rt.make_rays(o, d, rng.uniform(0, 1, n))
    got, st = sc.closest_hit(rays, flags=rt.RT_OPT_COUNT)
    want = osc.closest_hit(rays, mode=0)
    compare_hits(rt, got, want)
    assert (want["prim_id"] != rt.RT_NONE).mean() > 0.3
    assert st.node_visits / n < 200 and st.prim_tests / n < 40


def test_four_wide_tree_gives_the_same_hits_and_images(gpu, rt, orc, monkeypatch):
    """Scenes beyond the caches are traversed through a four-wide collapse of the SAH tree (the 200k soups above take
    that path by size).  Forced here on small scenes with Transforms, media and every tie rule: ids, t and same-seed
    images must not depend on which tree was walked."""
    monkeypatch.setenv("RT2025_WIDE_BVH", "1")
    for seed in (2, 5):
        hs = random_graph_scene(rt, seed, n_prims=120, with_media=True, width=24, spp=4, depth=6)
        sc, osc = rt.Scene(hs), orc.OracleScene(hs)
        assert sc.info().node_bytes == 128
        rng = np.random.default_rng(seed)
        o, d, t = random_rays(rng, 20000)
        rays = rt.make_rays(o, d, t)
        compare_hits(rt, sc.closest_hit(rays)[0], osc.closest_hit(rays, mode=0))
        img, st = sc.render(seed=3)
        ref, _ = osc.render(seed=3)
        image_close(img, ref)
    hs = rt.named_scene("book2_final", seed=7, params=[32, 4, 12])
    wide = rt.Scene(hs)
    monkeypatch.setenv("RT2025_WIDE_BVH", "0")
    binary = rt.Scene(hs)
    assert wide.info().node_bytes == 128 and binary.info().node_bytes == 64
    fx = np.load(os.path.join(GOLDEN, "book2_final.npz"))
    a, b = wide.closest_hit(fx["rays"])[0], binary.closest_hit(fx["rays"])[0]
    assert np.array_equal(a["prim_id"], b["prim_id"]) and np.array_equal(a["t"], b["t"])
    image_close(wide.render(seed=2025)[0], binary.render(seed=2025)[0])


def test_device_lbvh_build_gives_the_same_hits(gpu, rt, orc):
    """RT_BUILD_DEVICE_LBVH: the world tree comes from the Morton-code builder on the GPU (csrc/lbvh.cu).  Ids, t and
    tie ranks must not depend on the builder."""
    for shape in ("tri_soup", "sphere_soup"):
        hs = rt.named_scene(shape, seed=9, params=[60_000])
        sc, osc = rt.Scene(hs, flags=rt.RT_BUILD_DEVICE_LBVH), orc.OracleScene(hs)
        info = sc.info()
        assert info.n_nodes == 60_000 - 1  # one primitive per leaf: the radix tree, not the SAH tree
        assert np.array_equal(sc.ranks(), osc.ranks())
        rng = np.random.default_rng(4)
        n = 40_000
        o = np.concatenate([np.tile([0.5, 0.5, -2.0], (n // 2, 1)), rng.uniform(0, 1, (n // 2, 3))])
        tgt = rng.uniform(-0.2, 1.2, (n // 2, 3))
        tgt[:, 2] = 0.0
        d = np.concatenate([tgt - o[: n // 2], rng.normal(size=(n // 2, 3))])
        rays = rt.make_rays(o, d, rng.uniform(0, 1, n))
        compare_hits(rt, sc.closest_hit(rays)[0], osc.closest_hit(rays, mode=0))
    # a rendered frame through the device-built tree: 6000 primitives of every kind under lists, BVHs and Transforms
    hs = random_graph_scene(rt, 21, n_prims=6000, with_media=True, width=24, spp=4, depth=5)
    sc, osc = rt.Scene(hs, flags=rt.RT_BUILD_DEVICE_LBVH), orc.OracleScene(hs)
    assert np.array_equal(sc.ranks(), osc.ranks())
    o, d, t = random_rays(np.random.default_rng(2), 20000)
    rays = rt.make_rays(o, d, t)
    compare_hits(rt, sc.closest_hit(rays)[0], osc.closest_hit(rays, mode=0))
    image_close(sc.render(seed=6)[0], osc.render(seed=6)[0])
    # a small world (below the builder's minimum) silently takes the host builder
    hs = rt.named_scene("cornell_glass", seed=7, params=[32, 4, 12])
    a, b = rt.Scene(hs, flags=rt.RT_BUILD_DEVICE_LBVH), rt.Scene(hs)
    assert a.info().n_nodes == b.info().n_nodes


def test_soup_at_full_batch_size_properties(gpu, rt):
    """1M triangles, 2^22 rays: properties that need no oracle — every reported hit re-verifies against
    its own primitive record through a second, single-ray query window [t, t]."""
    hs = rt.named_scene("tri_soup", seed=5, params=[1_000_000])
    sc = rt.Scene(hs)
    rng = np.random.default_rng(8)
    n = 1 << 22
    rays = rt.make_rays(rng.uniform(0, 1, (n, 3)), rng.normal(size=(n, 3)))
    got, _ = sc.closest_hit(rays)
    hit = got["prim_id"] != rt.RT_NONE
    assert 0.5 < hit.mean() <= 1.0
    assert np.all(got["t"][hit] >= 1e-8) and np.all(np.isinf(got["t"][~hit]))
    # idempotence: asking again inside the degenerate interval [t, t] returns the same primitive
    sub = np.nonzero(hit)[0][:20000]
    for i in sub[:50]:
        again, _ = sc.closest_hit(rays[i:i + 1], t_min=got["t"][i], t_max=got["t"][i])
        assert again["prim_id"][0] == got["prim_id"][i] and again["t"][0] == got["t"][i]
    # shrinking t_max below the hit must never report that primitive at that distance again
    far, _ = sc.closest_hit(rays[sub], t_max=1e-3)
    assert np.all((far["prim_id"] == rt.RT_NONE) | (far["t"] <= 1e-3))


def test_corrupted_descriptions_do_not_fault_the_device(gpu, rt):
    """scripts/fuzz_gpu.py: single-word corruptions (indices and numbers) of every table, then create + closest hit +
    render.  In a process of its own: a CUDA fault would poison the context of the remaining tests."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "scripts", "fuzz_gpu.py"), "11", "800"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-1500:]
    assert "create=0 hit=0 render=0" in r.stdout and "create=-1" in r.stdout


def test_cpp_dropin_camera_render(gpu, rt, tmp_path):
    """examples/final_scene.cpp builds the Cornell box with the reference's constructors and calls
    Camera::render(world, lights) -> RgbImage: the 8-bit result must equal rendering the same flattened
    scene through the Python binding (same seed) and tone-mapping it."""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.check_call(["make", "-s", "-C", root, "examples"])
    out = tmp_path / "c.ppm"
    msg = subprocess.check_output([os.path.join(root, "examples", "final_scene"), "mini_cornell", "64", "16", "10", str(out)]).decode()
    assert "0 errors" in msg
    data = out.read_bytes()
    header, pixels = data.split(b"\n255\n", 1)
    assert header == b"P6\n64 64"
    got = np.frombuffer(pixels, dtype=np.uint8).reshape(64, 64, 3)
    hs = rt.named_scene("cornell_shipped", seed=7, params=[64, 16, 10])
    img, st = rt.Scene(hs).render(seed=0x2025)
    want = rt.tonemap(img, 0)
    assert np.array_equal(got, want)
    assert got.mean() > 20


def test_disney_vs_oracle(gpu, rt, orc):
    from scenes_util import disney_scene
    for lights in (True, False):
        hs = disney_scene(rt, lights, width=64, spp=16)
        sc, osc = rt.Scene(hs), orc.OracleScene(hs)
        img, st = sc.render(seed=9)
        ref, ost = osc.render(seed=9)
        assert st.paths == ost.paths and int(st.errors) <= int(ost.errors)
        image_close(img, ref, frac_bad=5e-3)


def test_obj_faces_with_remapped_materials_vs_oracle(gpu, rt, orc):
    from scenes_util import obj_mesh_scene
    hs = obj_mesh_scene(rt)
    sc, osc = rt.Scene(hs), orc.OracleScene(hs)
    rng = np.random.default_rng(1)
    o, d, t = random_rays(rng, 20000, extent=4.0)
    rays = rt.make_rays(o, d, t)
    got, _ = sc.closest_hit(rays)
    compare_hits(rt, got, osc.closest_hit(rays, mode=0))
    img, st = sc.render(seed=4)
    ref, ost = osc.render(seed=4)
    assert st.paths == ost.paths and int(st.errors) <= int(ost.errors)
    image_close(img, ref, frac_bad=5e-3)


def test_tonemap_device_equals_host_entry(gpu, rt):
    import torch
    rng = np.random.default_rng(3)
    img = (rng.random((37, 53, 3)) * 1.6).astype(np.float32)
    for toon in (0, 1):
        want = rt.tonemap(img, toon)
        d_in = torch.from_numpy(img).cuda()
        d_out = torch.empty((37, 53, 3), dtype=torch.uint8, device="cuda")
        rt.tonemap_device(d_in.data_ptr(), 37 * 53, d_out.data_ptr(), toon, rt.RT_ACCUM_F32, torch.cuda.current_stream().cuda_stream)
        assert np.array_equal(d_out.cpu().numpy(), want)
    bad = torch.full((4, 4, 3), float("nan"), dtype=torch.float32, device="cuda")
    out = torch.empty((4, 4, 3), dtype=torch.uint8, device="cuda")
    with pytest.raises(RuntimeError):
        rt.tonemap_device(bad.data_ptr(), 16, out.data_ptr())


def test_render_rgb8_equals_render_then_tonemap(gpu, rt):
    hs = rt.named_scene("cornell_glass", seed=3, params=[48, 9, 12])
    sc = rt.Scene(hs)
    rgb, st = sc.render_rgb8(seed=6)
    img, _ = sc.render(seed=6)
    assert np.array_equal(rgb, rt.tonemap(img, 0)) and rgb.dtype == np.uint8 and st.paths == 48 * 48 * 9


def test_render_multi_in_one_process(gpu, rt):
    """rt_render_multi with as many GPUs as the box has (1 on the default test box): equals rt_render."""
    n = gpu.rt_device_count()
    hs = rt.named_scene("book2_final", seed=5, params=[64, 9, 20])
    scenes = [rt.Scene(hs, device=k) for k in range(min(n, 4))]
    img, st = rt.render_multi(scenes, seed=3)
    ref, rst = scenes[0].render(seed=3)
    assert st.paths == rst.paths and st.segments == rst.segments
    assert np.allclose(img, ref, rtol=1e-12, atol=1e-14)
    # ... ending like Camera::render: the reduced frame is encoded on GPU 0 and only the bytes come back
    rgb, st8 = rt.render_multi_rgb8(scenes, seed=3)
    assert np.array_equal(rgb, rt.tonemap(ref, 0)) and st8.paths == rst.paths
    f32, _ = rt.render_multi(scenes, seed=3, accum_type=rt.RT_ACCUM_F32)
    assert f32.dtype == np.float32 and np.allclose(f32, ref, rtol=1e-6, atol=1e-7)
    with pytest.raises(rt.RtError):
        rt.render_multi([scenes[0], scenes[0]], seed=3)  # two handles on one device


def test_two_renders_share_a_gpu(gpu, rt):
    """Two scenes rendered from two host threads on one GPU at the same time: each borrows a workspace of its own."""
    import threading
    a = rt.Scene(rt.named_scene("cornell_glass", seed=3, params=[48, 9, 12]))
    b = rt.Scene(rt.named_scene("book1_final", seed=3, params=[64, 4, 12]))
    want = [a.render(seed=5)[0], b.render(seed=6)[0]]
    got = [None, None]

    def work(k, sc, seed):
        for _ in range(3):
            got[k] = sc.render(seed=seed)[0]
    th = [threading.Thread(target=work, args=(0, a, 5)), threading.Thread(target=work, args=(1, b, 6))]
    [t.start() for t in th]
    [t.join() for t in th]
    assert np.allclose(got[0], want[0], rtol=1e-12, atol=1e-14) and np.allclose(got[1], want[1], rtol=1e-12, atol=1e-14)


def test_zero_depth_is_black(gpu, rt):
    # ray_color returns black at depth 0 before it looks at the world (camera.rs:282)
    hs = rt.named_scene("cornell_glass", seed=3, params=[16, 4, 0])
    img, st = rt.Scene(hs).render(seed=1)
    assert not img.any() and st.segments == 0 and st.paths == 16 * 16 * 4


def _psnr8(a, b):
    mse = np.mean((a.astype(np.float64) - b.astype(np.float64)) ** 2)
    return 10 * np.log10(255.0 ** 2 / max(mse, 1e-12))


def test_independent_seeds_are_statistically_consistent(gpu, rt, orc):
    """North-star checks (2) and (3): an oracle render with ANOTHER seed differs from the GPU render only
    by Monte Carlo noise, and both converge to the same image (PSNR >= 40 dB at high spp).  Config 3
    (Cornell + glass sphere, mixture-pdf light sampling) at reduced resolution, full 961 spp."""
    hs = rt.named_scene("cornell_glass", seed=7, params=[64, 1000, 50])
    sc, osc = rt.Scene(hs), orc.OracleScene(hs)
    assert hs.camera.sqrt_spp == 31
    ref_other_seed, ost = osc.render(seed=1001)         # the "reference" at the config's spp, its own seed
    gpu = [sc.render(seed=s)[0] for s in range(1, 41)]   # 40 independent GPU renders of 961 spp each
    assert ost.errors == 0
    # (3) same-spp check: E|a-b|^2 = var_a + var_b for independent estimates, whoever produced them
    clip = lambda x: np.minimum(x, 4.0)  # the light itself is 15: keep fireflies from dominating the statistic
    mse_gpu_pairs = np.mean([np.mean((clip(gpu[2 * k]) - clip(gpu[2 * k + 1])) ** 2) for k in range(8)])
    mse_vs_oracle = np.mean([np.mean((clip(ref_other_seed) - clip(g)) ** 2) for g in gpu[:8]])
    assert 0.8 < mse_vs_oracle / mse_gpu_pairs < 1.25
    # per-pixel: the oracle image lies within 6 sigma of the GPU sample mean (sigma from the 40 renders)
    stack = np.stack([clip(g) for g in gpu])
    mean, sd = stack.mean(axis=0), stack.std(axis=0, ddof=1)
    z = np.abs(clip(ref_other_seed) - mean) / (sd * np.sqrt(1 + 1 / 40) + 1e-3)
    assert (z > 6).mean() < 2e-3
    # (2) convergence: 8 x 961 spp against the disjoint 32 x 961 spp average, and the oracle's single render
    converged = rt.tonemap(np.mean(gpu[8:], axis=0))
    high = rt.tonemap(np.mean(gpu[:8], axis=0))
    assert _psnr8(high, converged) >= 40.0
    assert _psnr8(rt.tonemap(ref_other_seed), converged) >= 30.0
    # (2') against the ORACLE's converged render (tests/golden/make_converged.py: 32 x 961 spp, seeds of its own): the GPU's
    # 40 x 961 spp mean must agree to >= 40 dB after the 8-bit encode
    fx = np.load(os.path.join(GOLDEN, "cornell_glass_converged.npz"))
    assert int(fx["errors"]) == 0 and not set(fx["seeds"].tolist()) & set(range(1, 41))
    assert _psnr8(rt.tonemap(np.mean(gpu, axis=0)), rt.tonemap(fx["image"])) >= 40.0
    assert abs(np.mean(gpu) - fx["image"].mean()) < 0.01 * fx["image"].mean()


def test_hand_derived_hit_vectors(gpu, rt):
    """The paper-derived vectors of tests/test_oracle_kat_hand.py (Sphere / Quad / Triangle / Transform::hit) on the device:
    t, u, v exact, misses are misses - no oracle in the loop."""
    from test_oracle_kat_hand import HIT_VECTORS
    for name, (make, vectors) in sorted(HIT_VECTORS.items()):
        sc = rt.Scene(make(rt))
        for o, d, time, t_min, t_max, want in vectors:
            got, _ = sc.closest_hit(rt.make_rays([o], [d], [time]), t_min=t_min, t_max=t_max)
            if want is None:
                assert got["prim_id"][0] == rt.RT_NONE and np.isinf(got["t"][0]), (name, o, d)
            else:
                assert got["prim_id"][0] != rt.RT_NONE, (name, o, d)
                assert got["t"][0] == want["t"] and got["u"][0] == np.float32(want["u"]) and got["v"][0] == np.float32(want["v"]), (name, o, d)


@pytest.mark.parametrize("name,params,strata", [("book1_final", [1200, 10, 50], 2), ("book2_final", [800, 1000, 40], 2),
                                                ("cornell_glass", [600, 1000, 50], 2)])
def test_baseline_resolution_strata_match_oracle(gpu, rt, orc, name, params, strata):
    """Configs 1-3 at BASELINE.json's own resolution and sampling grid (1200x675 / 3x3, 800x800 / 31x31, 600x600 / 31x31):
    strata [0, 2) of the real frame, same seed, against the oracle (about a second of CPU each)."""
    hs = rt.named_scene(name, seed=7, params=params)
    cam = hs.camera
    assert (cam.image_width, cam.image_height, cam.sqrt_spp) == {"book1_final": (1200, 675, 3), "book2_final": (800, 800, 31),
                                                                 "cornell_glass": (600, 600, 31)}[name]
    sc, osc = rt.Scene(hs), orc.OracleScene(hs)
    img, st = sc.render(seed=33, sample_begin=0, sample_end=strata)
    ref, ost = osc.render(seed=33, sample_begin=0, sample_end=strata)
    assert st.paths == ost.paths == cam.image_width * cam.image_height * strata and int(st.errors) <= int(ost.errors)
    image_close(img, ref)


def test_medium_inside_bvh_and_transform(gpu, rt, orc):
    """ConstantMedium below a BVH (the reference clamps the exit to the interval the BVH has already shrunk, volume.rs:46-47 with
    bvh.rs:78-84) and below Transform(BVH): same winners as taking the minimum over all children on [1e-8, inf)."""
    b = rt.Builder(6)
    white = b.lambertian(b.solid(0.7, 0.7, 0.7))
    fog1 = b.medium(b.sphere([-1.5, 0, 0], 1.2, b.empty()), 1.1, b.solid(0.9, 0.5, 0.3))
    fog2 = b.medium(b.box([-0.8, -0.8, -0.8], [0.8, 0.8, 0.8], b.empty()), 0.7, b.solid(0.3, 0.6, 0.9))
    inner = b.bvh([b.sphere([-1.5, 0, 0], 0.5, white), fog1, b.quad([-3, -1.3, -2], [6, 0, 0], [0, 0, 4], white),
                   b.sphere([-1.5, 0.2, 1.6], 0.4, b.metal([0.9, 0.9, 0.9], 0.1))])
    moved = b.transform(b.bvh([fog2, b.sphere([0, 0, 0], 0.3, white), b.triangle([-1, -1, -1.2], [2, 0, 0], [0, 2, 0], white)]),
                        offset=[1.8, 0.2, 0.0], quat=b.quat_axis_angle([0, 1, 0], 25.0), scale=[1.2, 1.2, 1.2])
    light = b.quad([-1, 3.5, -1], [2, 0, 0], [0, 0, 2], b.diffuse_light(b.solid(12, 12, 12)))
    world = b.list([b.bvh([inner, moved, light])])
    lights = b.list([b.quad([-1, 3.5, -1], [2, 0, 0], [0, 0, 2], b.empty())])
    hs = b.finish(world, lights, width=56, spp=16, max_depth=12, vfov=40, look_from=(0, 1.5, 8), look_at=(0, 0, 0), background=b.solid(0.05, 0.06, 0.1))
    sc, osc = rt.Scene(hs), orc.OracleScene(hs)
    assert sc.info().n_media == 2 and np.array_equal(sc.ranks(), osc.ranks())
    for classic in (False, True):
        img, st = sc.render(seed=12, classic_media_order=classic)
        ref, ost = osc.render(seed=12)
        assert st.paths == ost.paths and int(st.errors) <= int(ost.errors)
        image_close(img, ref, frac_bad=5e-3)


@pytest.mark.parametrize("knobs", [
    {"RT2025_FIFO_SLOTS": "64", "RT2025_REFILL_MIN": "1"}, {"RT2025_FIFO_SLOTS": "32", "RT2025_REFILL_MIN": "16"}, {"RT2025_FIFO_SLOTS": "0"},
    {"RT2025_MEDIA_FIRST": "2"}, {"RT2025_MEDIA_FIRST": "0"}, {"RT2025_TAIL_PATHS": "0"}, {"RT2025_TAIL_PATHS": "1000000"},
    {"RT2025_PATHS_IN_FLIGHT": "8192", "RT2025_TAIL_PATHS": "100"}, {"RT2025_PARK_LEAVES": "1", "RT2025_FIFO_SLOTS": "64"},
])
def test_every_traversal_and_scheduling_mode_gives_the_same_answer(gpu, rt, orc, monkeypatch, knobs):
    """The tuning knobs pick between code paths that must not change results: prepared-ray FIFO vs direct refill, postponed leaves,
    media sampled after / ahead of / inside extend, the tail kernel, the wavefront capacity.  Ids and t bit-exact, images equal."""
    scenes = [rt.named_scene("book2_final", seed=7, params=[48, 9, 20]),
              random_graph_scene(rt, 13, n_prims=90, with_media=True, width=32, spp=9, depth=8)]
    base = []
    rng = np.random.default_rng(5)
    o, d, t = random_rays(rng, 20000)
    rays = rt.make_rays(o * 40 + 250, d, t)  # through the book-2 box and the random graph alike
    for hs in scenes:
        sc = rt.Scene(hs)
        base.append((sc.closest_hit(rays)[0], sc.render(seed=11)))
        sc.close()
    for k, v in knobs.items():
        monkeypatch.setenv(k, v)
    for hs, (hits0, (img0, st0)) in zip(scenes, base):
        sc = rt.Scene(hs)
        hits = sc.closest_hit(rays)[0]
        assert np.array_equal(hits["prim_id"], hits0["prim_id"]) and np.array_equal(hits["t"], hits0["t"])
        img, st = sc.render(seed=11)
        assert st.paths == st0.paths and st.segments == st0.segments and st.errors == st0.errors
        assert np.allclose(img, img0, rtol=1e-11, atol=1e-13)
        ref, _ = orc.OracleScene(hs).render(seed=11)
        image_close(img, ref, frac_bad=5e-3)
        sc.close()
