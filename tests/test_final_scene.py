"""BASELINE.json config 4: `obj_scene()` (reference src/main.rs:207-382) on the assets the reference ships, with an
image-backed equirect environment (shapes/environment.rs:14-24 over ImageTexture, texture.rs:102-174).

CPU tests cover the asset pack, the loader output and the oracle; `-m gpu` tests are the parity tests proper
(ids and t bit-exact, same-seed images, the environment lookup against an independent numpy restatement).
"""
import json
import os

import numpy as np
import pytest

from scenes_util import _pkg_module, compare_hits, final_reduced_scene, table_digests

KIND = dict(sphere=1, quad=2, tri=3, list=4, bvh=5, transform=6, medium=7)
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def image_close(img, ref, frac_bad=5e-3, rel=1e-6):
    diff = np.abs(img - ref)
    bad = (diff > rel * (1 + np.abs(ref))).any(axis=2)
    assert bad.mean() <= frac_bad, f"{int(bad.sum())}/{bad.size} pixels differ (max {diff.max():.3e})"
    assert abs(img.mean() - ref.mean()) <= 1e-3 * ref.mean() + 1e-9


def equirect_lookup(env, d):
    """Environment::value + ImageTexture nearest texel, restated in numpy: environment.rs:14-24, texture.rs:111-119."""
    p = d / np.linalg.norm(d, axis=1, keepdims=True)
    theta = np.arccos(-p[:, 1])
    phi = np.pi - np.arctan2(-p[:, 2], p[:, 0])
    u, v = phi / (2 * np.pi), theta / np.pi
    u, v = u - np.floor(u), 1.0 - (v - np.floor(v))
    h, w = env.shape[:2]
    i = np.minimum((u * w).astype(np.int64), w - 1)
    j = np.minimum((v * h).astype(np.int64), h - 1)
    return env[j, i, :3].astype(np.float64)


def sky_only_scene(rt, env, width=64, spp=1):
    b = rt.Builder(1)
    hs = b.finish(b.list([]), width=width, aspect=2.0, spp=spp, max_depth=4, vfov=100.0, look_from=(0, 0, 0), look_at=(0.3, 0.2, -1),
                  background=b.image(env, raw=False, linear_format=True))
    hs._builder = b
    return hs


def test_final_scene_structure(rt):
    hs = final_reduced_scene(rt)
    d = hs.desc.contents
    o = hs.objects()
    # 13 of the 15 OBJ files, 38 234 non-degenerate triangles (counted from the shipped files), 3 boards + portal quad
    # + the 6 quads of build_box in the world, 2 boards in the lights list
    assert (o["kind"] == KIND["tri"]).sum() == 38234 and d.n_remaps == 38234
    assert (o["kind"] == KIND["quad"]).sum() == 4 + 6 + 2
    assert (o["kind"] == KIND["medium"]).sum() == 1 and (o["kind"] == KIND["transform"]).sum() == 6
    assert d.n_images == 10  # 9 material images + the environment
    world = o[d.world_root]
    assert world["kind"] == KIND["list"] and world["child_count"] == 18  # 20 world.add() calls minus the two missing meshes
    cam = hs.camera
    assert (cam.image_width, cam.image_height) == (96, 54) and cam.background_tex != rt.RT_NONE


def test_pack_equals_reference_files(rt):
    """The committed pack is the parse of the reference's files: object graph, geometry, remap frames and material records
    of the scene built from the pack are byte-identical to those of obj_scene() on the reference's assets/ directory, stored
    as digests in final_assets_tables.json by make_final_pack.py (only the texel pools differ: reduced images)."""
    with open(os.path.join(GOLDEN, "final_assets_tables.json")) as f:
        want = json.load(f)
    assert table_digests(final_reduced_scene(rt)) == want


def test_environment_lookup_oracle(rt, orc):
    """Row a30 on the CPU: the oracle's Environment::value over an image texture against the numpy restatement."""
    env = _pkg_module(rt, "scenes").synthetic_hdr_environment(64, 32)
    assert env.max() > 4.0  # genuinely HDR: no 8-bit clamp anywhere
    hs = sky_only_scene(rt, env)
    img, st = orc.OracleScene(hs).render(seed=5)
    cam = hs.camera
    px = np.array([(i, j) for j in range(cam.image_height) for i in range(cam.image_width)])
    rays = orc.camera_rays(cam, 5, px, 0)
    want = equirect_lookup(env, rays["direction"]).reshape(cam.image_height, cam.image_width, 3)
    assert st.segments == st.paths and st.errors == 0
    assert np.array_equal(img, want)
    # hand-derived: +x looks at the image centre, +y at the top row... v' = 1 - v flips the rows (texture.rs:113)
    for d, (u, v) in (((1, 0, 0), (0.5, 0.5)), ((0, 0, 1), (0.25, 0.5)), ((0, 1, 0), (0.5, 1.0))):
        got = equirect_lookup(env, np.array([d], dtype=np.float64))[0]
        h, w = env.shape[:2]
        uu, vv = u - np.floor(u), 1.0 - (v - np.floor(v))
        assert np.array_equal(got, env[min(int(vv * h), h - 1), min(int(uu * w), w - 1), :3].astype(np.float64))


def test_final_scene_oracle_sees_every_feature(rt, orc):
    hs = final_reduced_scene(rt, width=96, spp=4, depth=12)
    osc = orc.OracleScene(hs)
    img, st = osc.render(seed=3)
    assert st.errors == 0 and np.isfinite(img).all() and 0.2 < img.mean() < 2.0
    assert 2.0 < st.segments / st.paths < 6.0
    assert img[:10].mean() > 0.05  # the top rows look past the meshes into the environment


@pytest.mark.gpu
def test_environment_lookup_gpu(gpu, rt, orc):
    """Row a30 on the device: acos/atan2 equirect lookup into an HDR-flagged image texture, bit for bit."""
    env = _pkg_module(rt, "scenes").synthetic_hdr_environment(128, 64)
    hs = sky_only_scene(rt, env, width=96, spp=4)
    sc = rt.Scene(hs)
    img, st = sc.render(seed=5)
    ref, _ = orc.OracleScene(hs).render(seed=5)
    assert st.segments == st.paths and st.errors == 0
    # device acos/atan2 may differ from libm in the last bit: a texel boundary flips for a vanishing share of samples
    bad = (np.abs(img - ref) > 1e-12 * (1 + np.abs(ref))).any(axis=2)
    assert bad.mean() < 5e-3
    one = sky_only_scene(rt, env, width=96, spp=1)
    img1, _ = rt.Scene(one).render(seed=5)
    cam = one.camera
    px = np.array([(i, j) for j in range(cam.image_height) for i in range(cam.image_width)])
    want = equirect_lookup(env, orc.camera_rays(cam, 5, px, 0)["direction"]).reshape(cam.image_height, cam.image_width, 3)
    assert ((img1 != want).any(axis=2)).mean() < 5e-3 and img1.max() > 4.0


@pytest.mark.gpu
def test_final_scene_hits_bit_exact(gpu, rt, orc):
    hs = final_reduced_scene(rt, width=192, spp=4, depth=12)
    sc, osc = rt.Scene(hs), orc.OracleScene(hs)
    assert np.array_equal(sc.ranks(), osc.ranks())
    info = sc.info()
    assert info.n_prims >= 38234 and info.n_media == 1 and info.n_lights == 2
    rng = np.random.default_rng(12)
    cam = hs.camera
    n = 16384
    px = np.stack([rng.integers(0, cam.image_width, n), rng.integers(0, cam.image_height, n)], axis=1)
    prim = orc.camera_rays(cam, 9, px, 0)
    h = osc.closest_hit(prim)
    hit = h["prim_id"] != rt.RT_NONE
    p = prim["origin"] + np.where(hit, h["t"], 0.0)[:, None] * prim["direction"]
    sec = rt.make_rays(p, rng.normal(size=(n, 3)), prim["time"])  # rays leaving first-hit points in random directions
    rays = np.concatenate([prim, sec])
    got, st = sc.closest_hit(rays, flags=rt.RT_OPT_COUNT)
    want = osc.closest_hit(rays, mode=0)
    compare_hits(rt, got, want)
    assert (want["prim_id"] != rt.RT_NONE).mean() > 0.5 and len(rays) >= 30000
    assert len(set(want["inst_id"].tolist())) >= 3  # boards / the black box sit under Transforms


@pytest.mark.gpu
def test_final_scene_image_parity(gpu, rt, orc):
    hs = final_reduced_scene(rt, width=128, spp=16, depth=30)
    sc, osc = rt.Scene(hs), orc.OracleScene(hs)
    img, st = sc.render(seed=21)
    ref, ost = osc.render(seed=21)
    assert st.paths == ost.paths and int(st.errors) <= int(ost.errors)
    image_close(img, ref)
    assert ref[:8].mean() > 0.05  # environment texels reach the frame


@pytest.mark.gpu
def test_final_scene_full_resolution_strata(gpu, rt, orc):
    """1920x1080 (assets/Final/camera.json), 3000 -> 54^2 spp, depth 30: two strata of the real frame against the oracle."""
    hs = final_reduced_scene(rt, width=1920, spp=3000, depth=30)
    assert (hs.camera.image_width, hs.camera.image_height, hs.camera.sqrt_spp) == (1920, 1080, 54)
    sc, osc = rt.Scene(hs), orc.OracleScene(hs)
    img, st = sc.render(seed=4, sample_begin=0, sample_end=2)
    ref, ost = osc.render(seed=4, sample_begin=0, sample_end=2)
    assert st.paths == ost.paths == 1920 * 1080 * 2 and int(st.errors) <= int(ost.errors)
    image_close(img, ref)
