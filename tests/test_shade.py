"""The shade query and camera rays: rt_shade / rt_shade_device and rt_camera_rays / rt_camera_rays_device.

rt_shade runs the step of ray_color after world.hit (camera.rs:288-321) on rt_hit_records, with the draws of (seed, pixel = row
index, sample 0, segment), and updates the path state in place.  With rt_camera_rays and rt_world_hit it makes a client path loop:

    rays = camera_rays(cam, seed, 0); beta = 1; radiance = 0; state = RT_PATH_ALIVE
    for seg in range(cam.max_depth):
        rec = sc.world_hit(rays, t_min=1e-8, t_max=where(state & 1, inf, nan), seed=seed, segment=seg)
        sc.shade(rec, rays, beta, radiance, state, seed=seed, segment=seg, camera=cam)
    image = radiance * cam.pixel_sample_scale

which is rt_render at one sample per pixel.  Checks: that loop against rt_render; each segment bit for bit against the render's own
step (shade_one<SC_OTHER> through tests/device_kat.cu) and against the oracle's ray_step with the rules of test_segment_kat.py; camera
rays against the oracle's Camera::get_ray; inactive rows, determinism, draw addresses, the device entries and malformed records."""
import ctypes as C

import numpy as np
import pytest

import device_kat as dk
from scenes_util import disney_scene, final_reduced_scene, materials_scene, obj_mesh_scene, random_graph_scene
from test_segment_kat import REL, SCATTER_RAY, compare, expected_beta

NAMED = {
    "cornell_glass": ("cornell_glass", 7, [32, 4, 12]),
    "book1_final": ("book1_final", 7, [48, 4, 12]),
    "book2_final": ("book2_final", 7, [32, 4, 12]),
}
SCENES = ["cornell_glass", "book1_final", "book2_final", "random_graph", "final_reduced", "materials", "disney", "obj_mesh"]
BIT_EQUAL = {}  # scene: [pixels, bit-equal pixels] of the client loop against rt_render


@pytest.fixture(scope="module", autouse=True)
def report():
    yield
    if BIT_EQUAL:
        print("\n%-16s %8s %10s %9s" % ("scene", "pixels", "bit-equal", "fraction"))
        for k, (n, eq) in sorted(BIT_EQUAL.items()):
            print("%-16s %8d %10d %9.6f" % (k, n, eq, eq / n))


def make_scene(rt, name):
    if name == "random_graph":
        return random_graph_scene(rt, 11, n_prims=72, with_media=True, width=32, spp=4, depth=8)
    if name == "final_reduced":
        return final_reduced_scene(rt, width=64, spp=4, depth=12)
    if name == "materials":
        return materials_scene(rt)
    if name == "disney":
        return disney_scene(rt, width=48)
    if name == "obj_mesh":
        return obj_mesh_scene(rt, width=48)
    n, seed, params = NAMED[name]
    return rt.named_scene(n, seed=seed, params=params)


def one_spp_camera(rt, hs):
    """The scene's camera at one sample per pixel: the client loop addresses its draws with sample 0."""
    cam = rt.rt_camera.from_buffer_copy(hs.camera)
    cam.sqrt_spp, cam.recip_sqrt_spp, cam.pixel_sample_scale = 1, 1.0, 1.0
    return cam


def client_loop(rt, sc, cam, seed, each_segment=None):
    """The loop of the module docstring on host arrays.  Returns (image, segments traced, errors).  each_segment(seg, rays, beta,
    records, live) sees every segment's inputs before rt_shade runs."""
    rays = rt.camera_rays(cam, seed, 0)
    n = len(rays)
    beta, radiance = np.ones((n, 3)), np.zeros((n, 3))
    state = np.full(n, rt.RT_PATH_ALIVE, np.uint8)
    segments = errors = 0
    for seg in range(cam.max_depth):
        live = (state & rt.RT_PATH_ALIVE) != 0
        segments += int(live.sum())
        rec, _ = sc.world_hit(rays, t_min=1e-8, t_max=np.where(live, np.inf, np.nan), seed=seed, segment=seg)
        if each_segment is not None:
            each_segment(seg, rays.copy(), beta.copy(), rec, live)
        st = sc.shade(rec, rays, beta, radiance, state, seed=seed, segment=seg, camera=cam)
        assert st.segments == n and st.kernel_launches == 1
        assert st.errors == int(((state & rt.RT_PATH_ERROR) != 0)[live].sum())
        errors += st.errors
        if not (state & rt.RT_PATH_ALIVE).any():
            break
    return (radiance * cam.pixel_sample_scale).reshape(cam.image_height, cam.image_width, 3), segments, errors


def shade_rows(rt, sc, cam, rec, rays, beta, seed, seg, rows):
    """rt_shade on the rows `rows` alone, radiance from zero: (next rays, next beta, contribution, alive, error) of those rows."""
    # the row index is the pixel of the draws: the whole batch goes in, the other rows switched off
    full_r, full_b, full_rad = rays.copy(), beta.copy(), np.zeros((len(rays), 3))
    full_s = np.zeros(len(rays), np.uint8)
    full_s[rows] = rt.RT_PATH_ALIVE
    sc.shade(rec, full_r, full_b, full_rad, full_s, seed=seed, segment=seg, camera=cam)
    r, b, rad, state = full_r[rows], full_b[rows], full_rad[rows], full_s[rows]
    return r, b, rad, (state & rt.RT_PATH_ALIVE) != 0, (state & rt.RT_PATH_ERROR) != 0


# ---------------------------------------------------------------- CPU: the ABI and argument checks

def test_symbols_are_exported(rt):
    L = rt.product_lib()
    for name in ("rt_shade", "rt_shade_device", "rt_camera_rays", "rt_camera_rays_device"):
        assert name in rt.ABI_SYMBOLS and hasattr(L, name)
    assert (rt.RT_PATH_ALIVE, rt.RT_PATH_ERROR) == (1, 2)


def test_null_and_invalid_arguments_are_refused(rt):
    """Null pointers are refused before anything is dereferenced; a bad stratum or too many pixels before the device is looked
    for.  Without a device camera rays return RT_ERR_NO_DEVICE (and no scene exists to shade)."""
    L = rt.product_lib()
    b = rt.Builder(1)
    hs = b.finish(b.list([b.sphere([0, 0, 0], 1.0, b.lambertian(b.solid(0.5, 0.5, 0.5)))]), width=8, spp=4)
    cam = rt.rt_camera.from_buffer_copy(hs.camera)
    rec = np.zeros(1, rt.rt_hit_record_dtype)
    ray = rt.make_rays([[0.0, 0.0, 5.0]], [[0.0, 0.0, -1.0]])
    beta, rad, state = np.ones((1, 3)), np.zeros((1, 3)), np.ones(1, np.uint8)
    st = rt.rt_stats()
    fake = C.c_void_p(ray.ctypes.data)  # never dereferenced: the pointers are checked first
    args = [fake, C.byref(cam), rec.ctypes.data, 1, 1, 0, 0, ray.ctypes.data, beta.ctypes.data, rad.ctypes.data, state.ctypes.data]
    for k in (0, 1, 2, 7, 8, 9, 10):
        a = list(args)
        a[k] = None
        assert L.rt_shade(*a, C.byref(st)) == -1 and "null" in L.rt_last_error().decode()
        assert L.rt_shade_device(*a, None, C.byref(st)) == -1 and "null" in L.rt_last_error().decode()
    a = list(args)
    a[6] = 1  # RT_OPT_COUNT: rt_shade takes no flags
    assert L.rt_shade(*a, C.byref(st)) == -1 and "flags" in L.rt_last_error().decode()
    assert L.rt_shade_device(*a, None, C.byref(st)) == -1 and "flags" in L.rt_last_error().decode()
    out = np.zeros(cam.image_width * cam.image_height, rt.rt_ray_dtype)
    for f, extra in ((L.rt_camera_rays, ()), (L.rt_camera_rays_device, (None,))):
        assert f(None, 1, 0, out.ctypes.data, *extra) == -1
        assert f(C.byref(cam), 1, 0, None, *extra) == -1
        assert f(C.byref(cam), 1, 4, out.ctypes.data, *extra) == -1 and "sample" in L.rt_last_error().decode()  # sqrt_spp^2 == 4
        big = rt.rt_camera.from_buffer_copy(cam)
        big.image_width, big.image_height = 65536, 65536
        assert f(C.byref(big), 1, 0, out.ctypes.data, *extra) == -1 and "pixels" in L.rt_last_error().decode()
        if L.rt_device_count() < 1:
            assert f(C.byref(cam), 1, 3, out.ctypes.data, *extra) == -3  # RT_ERR_NO_DEVICE
        elif not extra:  # (the device entry would write to a host buffer)
            assert f(C.byref(cam), 1, 3, out.ctypes.data) == 0


# ---------------------------------------------------------------- GPU

@pytest.mark.gpu
@pytest.mark.parametrize("seed", [3, 0x9E3779B97F4A7C15])
@pytest.mark.parametrize("name", SCENES)
def test_client_loop_equals_render(gpu, rt, name, seed):
    hs = make_scene(rt, name)
    sc = rt.Scene(hs)
    cam = one_spp_camera(rt, hs)
    img, segments, errors = client_loop(rt, sc, cam, seed)
    ref, st = sc.render(camera=cam, seed=seed)
    assert st.paths == cam.image_width * cam.image_height
    assert segments == st.segments and errors == st.errors, (segments, st.segments, errors, st.errors)
    assert np.allclose(img, ref, rtol=1e-11, atol=1e-13)
    eq = (img.view(np.int64) == ref.view(np.int64)).all(axis=2)
    n, k = BIT_EQUAL.get(name, [0, 0])
    BIT_EQUAL[name] = [n + eq.size, k + int(eq.sum())]
    assert eq.all(), f"{name}: {int((~eq).sum())} of {eq.size} pixels are not bit-equal to rt_render"


def record_inputs(ds, rec):
    """The internal (t, prim, kind) the render's step gets for a record: device primitive or medium index (no shared children)."""
    kind = rec["kind"].astype(np.uint32)
    prim = np.full(len(rec), 0xFFFFFFFF, np.uint32)
    surf, med = kind == 1, kind == 2
    prim[surf] = ds.prim_of_object[rec["prim_id"][surf]]
    medium_of_object = {int(o): m for m, o in enumerate(ds.medium_object)}
    prim[med] = [medium_of_object[int(o)] for o in rec["prim_id"][med]]
    return np.where(kind == 0, np.inf, rec["t"]), prim, kind


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cornell_glass", "book2_final", "materials", "disney"])
def test_same_bits_as_the_render_step(gpu, rt, name):
    """Every segment of the loop through rt_shade and through shade_one<SC_OTHER> given the record's internal (t, prim, kind)."""
    hs = make_scene(rt, name)
    sc, ds = rt.Scene(hs), dk.DeviceScene(hs)
    cam = one_spp_camera(rt, hs)
    seed = 17
    seen = [0, 0]

    def check(seg, rays, beta, rec, live):
        rows = np.flatnonzero(live)
        r, b, rad, alive, err = shade_rows(rt, sc, cam, rec, rays, beta, seed, seg, rows)
        t, prim, kind = record_inputs(ds, rec[rows])
        ids6 = np.column_stack([rows, np.zeros_like(rows), np.full(len(rows), seg), prim, kind, np.full(len(rows), cam.max_depth)])
        want = ds.shade_step(cam, 8, 0, rays[rows], beta[rows], t, ids6, np.full(len(rows), seed, np.uint64))
        assert np.array_equal(alive, want["alive"]) and np.array_equal(err, want["errors"] > 0)
        bits = lambda a: np.ascontiguousarray(a, dtype=np.float64).view(np.int64)  # noqa: E731
        assert np.array_equal(bits(rad), bits(want["contribution"]))
        for got_v, key in ((r["origin"], "o"), (r["direction"], "d"), (r["time"], "time"), (b, "nbeta")):
            assert np.array_equal(bits(got_v[alive]), bits(want[key][alive])), key
        seen[0] += len(rows)
        seen[1] += int(err.sum())

    client_loop(rt, sc, cam, seed, check)
    assert seen[0] > 1000


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cornell_glass", "book2_final", "random_graph", "materials", "disney", "obj_mesh"])
def test_against_the_oracle(gpu, rt, orc, name):
    """rt_world_hit + rt_shade against the oracle's ray_step with ids (i, 0, segment) on the same rays: hit kinds, alive, error and
    NaN patterns exact; contributions of surface hits, next origins of surface hits and times bit-equal; directions, throughputs,
    and whatever a medium's t (log) or a background lookup reaches within REL."""
    hs = make_scene(rt, name)
    sc, osc = rt.Scene(hs), orc.OracleScene(hs)
    cam = one_spp_camera(rt, hs)
    seed = 5
    seen = [0]

    def check(seg, rays, beta, rec, live):
        rows = np.flatnonzero(live)
        r, b, rad, alive, err = shade_rows(rt, sc, cam, rec, rays, beta, seed, seg, rows)
        ids3 = np.column_stack([rows, np.zeros_like(rows), np.full(len(rows), seg)]).astype(np.uint32)
        st = osc.shade_step(rays[rows], np.full(len(rows), seed, np.uint64), ids3, camera=cam)
        assert np.array_equal(st["hit"], rec["kind"][rows].astype(np.int64)), f"{name}: hit kinds differ in segment {seg}"
        bt = beta[rows]
        with np.errstate(all="ignore"):
            c = bt * np.where((st["hit"] == 0)[:, None], st["background"], st["emission"])
        nan_c = np.isnan(c).any(axis=1)
        miss_error = (st["hit"] == 0) & st["error"]
        want_acc = np.where((c != 0.0) & ~nan_c[:, None] & ~miss_error[:, None], c, 0.0)
        nb = expected_beta(st, bt)
        want_alive = st["goes_on"] & ~st["error"] & (seg + 1 < cam.max_depth) & (nb != 0.0).any(axis=1)
        assert np.array_equal(alive, want_alive), f"{name}: alive differs in segment {seg}"
        assert np.array_equal(err, st["error"] | (nan_c & ~miss_error)), f"{name}: error bit differs in segment {seg}"
        mag = lambda v: np.max(np.abs(v), axis=1, keepdims=True)  # noqa: E731
        surf = st["hit"] == 1
        compare("shade: contribution (surface)", rad[surf], want_acc[surf])
        compare("shade: contribution (miss, medium)", rad[~surf], want_acc[~surf], rel=REL, scale=mag(want_acc[~surf]))
        on = st["goes_on"] & ~st["error"] & alive
        compare("shade: next origin (surface)", r["origin"][on & surf], st["o"][on & surf])
        compare("shade: next origin (medium)", r["origin"][on & ~surf], st["o"][on & ~surf], rel=REL, scale=mag(st["o"][on & ~surf]))
        compare("shade: next time", r["time"][on], st["time"][on])
        exact_d = on & surf & (st["kind"] == SCATTER_RAY) & ~st["fuzzed"]
        compare("shade: next direction (ray, no fuzz)", r["direction"][exact_d], st["d"][exact_d])
        compare("shade: next direction", r["direction"][on & ~exact_d], st["d"][on & ~exact_d], rel=REL, scale=mag(st["d"][on & ~exact_d]))
        ray = on & surf & (st["kind"] == SCATTER_RAY)
        compare("shade: next throughput (ray)", b[ray], nb[ray])
        compare("shade: next throughput", b[on & ~ray], nb[on & ~ray], rel=REL, scale=mag(nb[on & ~ray]))
        seen[0] += len(rows)

    client_loop(rt, sc, cam, seed, check)
    assert seen[0] > 1000


@pytest.mark.gpu
@pytest.mark.parametrize("defocus", [0.0, 2.5])
def test_camera_rays_match_the_oracle(gpu, rt, orc, defocus):
    """Bit for bit the render's camera_ray (through tests/device_kat.cu) for every pixel; against the oracle's Camera::get_ray with
    the rule of test_segment_kat.py: bit for bit without defocus, origins and directions within REL with it (sincos, sqrt)."""
    b = rt.Builder(1)
    hs = b.finish(b.list([b.sphere([0, 0, 0], 1.0, b.lambertian(b.solid(0.5, 0.5, 0.5)))]), width=24, aspect=24 / 17, spp=9, vfov=40,
                  look_from=(0.3, 1.1, 7), look_at=(0, 0, 0), defocus_angle=defocus, focus_dist=6.5)
    cam = hs.camera
    W, H = cam.image_width, cam.image_height
    assert (W, H, cam.sqrt_spp) == (24, 17, 3)
    ij = [(p % W, p // W) for p in range(W * H)]
    for seed in (0, 2 ** 64 - 1):
        for sample in (0, 8):
            got = rt.camera_rays(cam, seed, sample)
            render = dk.camera_ray(cam, seed, [p[0] for p in ij], [p[1] for p in ij], sample)
            assert got.tobytes() == np.ascontiguousarray(render).astype(rt.rt_ray_dtype).tobytes(), (seed, sample)
            want = orc.camera_rays(cam, seed, ij, sample)
            rel = REL if defocus else 0.0
            for f in ("origin", "direction"):
                compare("camera ray " + f, got[f], want[f], rel=rel, scale=np.max(np.abs(want[f]), axis=1, keepdims=True))
            compare("camera ray time", got["time"], want["time"])


@pytest.mark.gpu
def test_state_handling(gpu, rt):
    """Inactive rows come back byte for byte; calls repeat bit for bit; another seed or segment changes the draws."""
    hs = make_scene(rt, "book2_final")
    sc = rt.Scene(hs)
    cam = one_spp_camera(rt, hs)
    rays = rt.camera_rays(cam, 9, 0)
    n = len(rays)
    rec, _ = sc.world_hit(rays, seed=9, segment=0)
    rng = np.random.default_rng(1)
    inactive = rng.uniform(size=n) < 0.3
    state0 = np.where(inactive, rng.choice([0, 2, 0xFC, 0xFE], n), rt.RT_PATH_ALIVE | rng.choice([0, 0xFC], n)).astype(np.uint8)

    def run(seed=9, segment=0):
        r, bt = rays.copy(), np.ones((n, 3))
        r.view(np.uint8).reshape(n, -1)[inactive] = 0xA5
        bt.view(np.uint8).reshape(n, -1)[inactive] = 0x5A
        rad = np.full((n, 3), 0.25)
        rad.view(np.uint8).reshape(n, -1)[inactive] = 0x3C
        s = state0.copy()
        st = sc.shade(rec, r, bt, rad, s, seed=seed, segment=segment, camera=cam)
        return r, bt, rad, s, st

    r, bt, rad, s, st = run()
    for a in (r, bt, rad):
        assert (a.view(np.uint8).reshape(n, -1)[inactive] == a.view(np.uint8).reshape(n, -1)[inactive][0, 0]).all()
    assert np.array_equal(s[inactive], state0[inactive])
    assert ((s[~inactive] & ~np.uint8(3)) == 0).all()  # active rows: only the two defined bits
    assert st.segments == n and st.errors == int((s[~inactive] & 2).astype(bool).sum())
    alive = (s & 1).astype(bool)
    assert alive.sum() > n // 4
    r2, bt2, rad2, s2, _ = run()
    assert r.tobytes() == r2.tobytes() and bt.tobytes() == bt2.tobytes() and rad.tobytes() == rad2.tobytes() and s.tobytes() == s2.tobytes()
    for kw in (dict(seed=10), dict(segment=1)):
        r3, _, _, s3, _ = run(**kw)
        both = alive & (s3 & 1).astype(bool)
        changed = (r3["direction"] != r["direction"]).any(axis=1)
        assert changed[both].mean() > 0.5, kw  # (a smooth Dielectric's or Metal's reflection takes no draw)
    # the depth cut, and segments the reference never runs
    cam1 = rt.rt_camera.from_buffer_copy(cam)
    cam1.max_depth = 1
    s1 = state0.copy()
    sc.shade(rec, rays.copy(), np.ones((n, 3)), np.zeros((n, 3)), s1, seed=9, segment=0, camera=cam1)
    assert not (s1[~inactive] & 1).any()
    L = rt.product_lib()
    for c, seg in ((cam1, 1), (cam, cam.max_depth)):
        assert L.rt_shade(sc.h, C.byref(c), rec.ctypes.data, n, 9, seg, 0, rays.copy().ctypes.data, np.ones((n, 3)).ctypes.data,
                          np.zeros((n, 3)).ctypes.data, state0.copy().ctypes.data, None) == -1
    bad = rt.rt_camera.from_buffer_copy(cam)
    bad.background_tex = sc.info().n_textures
    assert L.rt_shade(sc.h, C.byref(bad), rec.ctypes.data, n, 9, 0, 0, rays.copy().ctypes.data, np.ones((n, 3)).ctypes.data,
                      np.zeros((n, 3)).ctypes.data, state0.copy().ctypes.data, None) == -1
    assert "background_tex" in L.rt_last_error().decode()


@pytest.mark.gpu
def test_malformed_records_end_their_path(gpu, rt):
    """kind 7 or a material beyond the table: RT_PATH_ERROR and nothing else of the row changes; the other rows are as without them."""
    hs = make_scene(rt, "cornell_glass")
    sc = rt.Scene(hs)
    cam = one_spp_camera(rt, hs)
    rays = rt.camera_rays(cam, 4, 0)
    n = len(rays)
    rec, _ = sc.world_hit(rays, seed=4, segment=0)

    def run(records):
        r, bt, rad, s = rays.copy(), np.ones((n, 3)), np.zeros((n, 3)), np.full(n, rt.RT_PATH_ALIVE, np.uint8)
        st = sc.shade(records, r, bt, rad, s, seed=4, segment=0, camera=cam)
        return r, bt, rad, s, st

    base = run(rec)
    bad = rec.copy()
    k = np.arange(0, n, 7)
    bad["kind"][k[0::2]] = 7
    m = k[1::2][rec["kind"][k[1::2]] != rt.RT_HIT_MISS]
    bad["material"][m] = sc.info().n_materials + np.arange(len(m))
    bad["material"][m[::3]] = 0xFFFFFFFF
    got = run(bad)
    hit = np.zeros(n, bool)
    hit[k[0::2]] = True
    hit[m] = True
    assert (got[3][hit] == rt.RT_PATH_ERROR).all()
    assert got[0][hit].tobytes() == rays[hit].tobytes() and (got[1][hit] == 1.0).all() and (got[2][hit] == 0.0).all()
    for a, b in zip(got[:4], base[:4]):
        assert a[~hit].tobytes() == b[~hit].tobytes()
    assert got[4].errors == int(((got[3] & rt.RT_PATH_ERROR) != 0).sum())


@pytest.mark.gpu
def test_device_entries_on_a_torch_stream(gpu, rt):
    import torch
    hs = make_scene(rt, "random_graph")
    sc = rt.Scene(hs)
    cam = one_spp_camera(rt, hs)
    n = cam.image_width * cam.image_height
    want_img, _, _ = client_loop(rt, sc, cam, 6)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        d_rays = torch.empty(n * 7, dtype=torch.float64, device="cuda")
        d_rec = torch.empty(n * rt.rt_hit_record_dtype.itemsize, dtype=torch.uint8, device="cuda")
        d_beta = torch.ones(n * 3, dtype=torch.float64, device="cuda")
        d_rad = torch.zeros(n * 3, dtype=torch.float64, device="cuda")
        d_state = torch.full((n,), rt.RT_PATH_ALIVE, dtype=torch.uint8, device="cuda")
        d_tmax = torch.empty(n, dtype=torch.float64, device="cuda")
        inf = torch.tensor(float("inf"), dtype=torch.float64, device="cuda")
        nan = torch.tensor(float("nan"), dtype=torch.float64, device="cuda")
        rt.camera_rays_device(cam, 6, 0, d_rays.data_ptr(), stream=s.cuda_stream)
        for seg in range(cam.max_depth):
            torch.where((d_state & 1) != 0, inf, nan, out=d_tmax)
            sc.world_hit_device(d_rays.data_ptr(), n, d_rec.data_ptr(), d_tmax.data_ptr(), t_min=1e-8, seed=6, segment=seg, stream=s.cuda_stream)
            st = sc.shade_device(d_rec.data_ptr(), n, d_rays.data_ptr(), d_beta.data_ptr(), d_rad.data_ptr(), d_state.data_ptr(), seed=6,
                                 segment=seg, camera=cam, stream=s.cuda_stream)
            assert st.segments == n
    s.synchronize()
    img = d_rad.cpu().numpy().reshape(cam.image_height, cam.image_width, 3)
    assert img.tobytes() == want_img.tobytes()
