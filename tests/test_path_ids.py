"""The path-id entries: rt_camera_rays_ids, rt_world_hit_ids and rt_shade_ids (and their _device forms).

Each row carries the render's own path id (pixel, sample, segment), and its draws are philox(seed; pixel, sample, segment, slot).
With them a client loop runs any number of samples per pixel, and may compact, permute and refill its batch:

    ids = (pixel, stratum, 0) for the paths in the batch; rays = camera_rays_ids(cam, seed, ids); beta = 1; radiance = 0
    loop: rec = sc.world_hit_ids(rays, ids, seed=seed); sc.shade_ids(rec, ids, rays, beta, radiance, state, seed=seed, camera=cam)
          rows that left: framebuffer[ids.pixel] += radiance; the others stay, new paths fill the free rows
    image = framebuffer * cam.pixel_sample_scale

Checks: the new entries against their twins bit for bit (ids (i, 0, s) / (i, s, .)); every stratum at sqrt_spp 2 and 3 against
rt_render of that one sample, bit for bit; a shuffled, compacting, refilling batch against the per-path values and the full render;
the row rules (segment >= max_depth, inactive rows, out-of-range ids, `reserved`); the device entries on a torch stream."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from test_shade import SCENES, make_scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RT_ERR_INVALID, RT_ERR_NO_DEVICE = -1, -3
NEW_SYMBOLS = ("rt_camera_rays_ids", "rt_camera_rays_ids_device", "rt_world_hit_ids", "rt_world_hit_ids_device", "rt_shade_ids",
               "rt_shade_ids_device")


def camera_at(rt, hs, sqrt_spp):
    """The scene's camera at sqrt_spp^2 samples per pixel."""
    cam = rt.rt_camera.from_buffer_copy(hs.camera)
    cam.sqrt_spp, cam.recip_sqrt_spp, cam.pixel_sample_scale = sqrt_spp, 1.0 / sqrt_spp, 1.0 / (sqrt_spp * sqrt_spp)
    return cam


def make_ids(rt, pixel, sample, segment=0, reserved=None):
    n = len(pixel)
    ids = np.zeros(n, rt.rt_path_id_dtype)
    ids["pixel"], ids["sample"], ids["segment"] = pixel, sample, segment
    ids["reserved"] = np.arange(n, dtype=np.uint32) * np.uint32(2654435761) if reserved is None else reserved
    return ids


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def stratum_loop(rt, sc, cam, seed, sample):
    """One path per pixel at stratum `sample`, rows = pixels, through the _ids entries.  Returns (radiance per pixel, segments, errors)."""
    n = cam.image_width * cam.image_height
    ids = make_ids(rt, np.arange(n), sample)
    reserved = ids["reserved"].copy()
    rays = rt.camera_rays_ids(cam, seed, ids)
    beta, radiance = np.ones((n, 3)), np.zeros((n, 3))
    state = np.full(n, rt.RT_PATH_ALIVE, np.uint8)
    segments = errors = 0
    for seg in range(cam.max_depth):
        live = (state & rt.RT_PATH_ALIVE) != 0
        assert (ids["segment"][live] == seg).all()
        segments += int(live.sum())
        rec, _ = sc.world_hit_ids(rays, ids, t_min=1e-8, t_max=np.where(live, np.inf, np.nan), seed=seed)
        st = sc.shade_ids(rec, ids, rays, beta, radiance, state, seed=seed, camera=cam)
        assert st.segments == n and st.kernel_launches == 1
        errors += st.errors
        if not (state & rt.RT_PATH_ALIVE).any():
            break
    assert np.array_equal(ids["reserved"], reserved) and np.array_equal(ids["pixel"], np.arange(n)) and (ids["sample"] == sample).all()
    return radiance, segments, errors


# ---------------------------------------------------------------- CPU: the ABI and argument checks

def test_symbols_are_exported(rt):
    L = rt.product_lib()
    for name in NEW_SYMBOLS:
        assert name in rt.ABI_SYMBOLS and hasattr(L, name)


def test_path_id_layout_matches_the_header(rt, tmp_path):
    src = tmp_path / "pid.c"
    src.write_text("""
#include <stddef.h>
#include <stdio.h>
#include "rt2025.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu\\n", sizeof(rt_path_id), offsetof(rt_path_id, pixel), offsetof(rt_path_id, sample),
         offsetof(rt_path_id, segment), offsetof(rt_path_id, reserved));
  return 0;
}
""")
    exe = tmp_path / "pid"
    subprocess.check_call(["/usr/bin/gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    dt = rt.rt_path_id_dtype
    assert got == [dt.itemsize] + [dt.fields[f][1] for f in ("pixel", "sample", "segment", "reserved")] == [16, 0, 4, 8, 12]


def test_invalid_arguments_are_refused_before_device_work(rt):
    """Null pointers, flags, an oversized batch, image_width == 0 and sqrt_spp == 0 are refused with RT_ERR_INVALID before anything
    is dereferenced or the device is looked for.  Without a device camera rays return RT_ERR_NO_DEVICE."""
    L = rt.product_lib()
    b = rt.Builder(1)
    hs = b.finish(b.list([b.sphere([0, 0, 0], 1.0, b.lambertian(b.solid(0.5, 0.5, 0.5)))]), width=8, spp=4)
    cam = rt.rt_camera.from_buffer_copy(hs.camera)
    rec = np.zeros(1, rt.rt_hit_record_dtype)
    ray = rt.make_rays([[0.0, 0.0, 5.0]], [[0.0, 0.0, -1.0]])
    ids = make_ids(rt, [0], [0])
    beta, rad, state = np.ones((1, 3)), np.zeros((1, 3)), np.ones(1, np.uint8)
    st = rt.rt_stats()
    fake = C.c_void_p(ray.ctypes.data)  # never dereferenced: the pointers and the batch size are checked first
    err = lambda: L.rt_last_error().decode()  # noqa: E731
    big = 2 ** 32 - 15
    # rt_shade_ids(scene, camera, records, ids, n, seed, flags, rays, beta, radiance, state, stats)
    args = [fake, C.byref(cam), rec.ctypes.data, ids.ctypes.data, 1, 1, 0, ray.ctypes.data, beta.ctypes.data, rad.ctypes.data,
            state.ctypes.data]
    for k in (0, 1, 2, 3, 7, 8, 9, 10):
        a = list(args)
        a[k] = None
        assert L.rt_shade_ids(*a, C.byref(st)) == RT_ERR_INVALID and "null" in err()
        assert L.rt_shade_ids_device(*a, None, C.byref(st)) == RT_ERR_INVALID and "null" in err()
    a = list(args)
    a[6] = 1
    assert L.rt_shade_ids(*a, C.byref(st)) == RT_ERR_INVALID and "flags" in err()
    assert L.rt_shade_ids_device(*a, None, C.byref(st)) == RT_ERR_INVALID and "flags" in err()
    a = list(args)
    a[4] = big
    assert L.rt_shade_ids(*a, C.byref(st)) == RT_ERR_INVALID and "2^32" in err()
    assert L.rt_shade_ids_device(*a, None, C.byref(st)) == RT_ERR_INVALID and "2^32" in err()
    # rt_world_hit_ids(scene, rays, ids, t_max_per_ray, n, t_min, t_max, seed, flags, out, stats)
    out = np.zeros(1, rt.rt_hit_record_dtype)
    args = [fake, ray.ctypes.data, ids.ctypes.data, None, 1, 1e-8, float("inf"), 1, 0, out.ctypes.data]
    for k in (0, 1, 2, 9):
        a = list(args)
        a[k] = None
        assert L.rt_world_hit_ids(*a, C.byref(st)) == RT_ERR_INVALID and "null" in err()
        assert L.rt_world_hit_ids_device(*a, None, C.byref(st)) == RT_ERR_INVALID and "null" in err()
    a = list(args)
    a[4] = big
    assert L.rt_world_hit_ids(*a, C.byref(st)) == RT_ERR_INVALID and "2^32" in err()
    assert L.rt_world_hit_ids_device(*a, None, C.byref(st)) == RT_ERR_INVALID and "2^32" in err()
    # rt_camera_rays_ids(camera, seed, ids, n, out)
    ids4 = make_ids(rt, [0, 5, 63, 1000], [0, 3, 17, 2])
    out = np.zeros(4, rt.rt_ray_dtype)
    for f, extra in ((L.rt_camera_rays_ids, ()), (L.rt_camera_rays_ids_device, (None,))):
        assert f(None, 1, ids4.ctypes.data, 4, out.ctypes.data, *extra) == RT_ERR_INVALID and "null" in err()
        assert f(C.byref(cam), 1, None, 4, out.ctypes.data, *extra) == RT_ERR_INVALID and "null" in err()
        assert f(C.byref(cam), 1, ids4.ctypes.data, 4, None, *extra) == RT_ERR_INVALID and "null" in err()
        assert f(C.byref(cam), 1, ids4.ctypes.data, big, out.ctypes.data, *extra) == RT_ERR_INVALID and "2^32" in err()
        for field in ("image_width", "sqrt_spp"):
            bad = rt.rt_camera.from_buffer_copy(cam)
            setattr(bad, field, 0)
            assert f(C.byref(bad), 1, ids4.ctypes.data, 4, out.ctypes.data, *extra) == RT_ERR_INVALID and field in err()
        if L.rt_device_count() < 1:
            assert f(C.byref(cam), 1, ids4.ctypes.data, 4, out.ctypes.data, *extra) == RT_ERR_NO_DEVICE
        elif not extra:  # (the device entry would write to a host buffer); ids beyond the image or the strata are not refused
            assert f(C.byref(cam), 1, ids4.ctypes.data, 4, out.ctypes.data) == 0


# ---------------------------------------------------------------- GPU

@pytest.mark.gpu
@pytest.mark.parametrize("name", ["book2_final", "final_reduced", "random_graph", "materials", "disney", "obj_mesh"])
def test_same_bits_as_the_fixed_address_entries(gpu, rt, name):
    """Over every segment of a path loop: rt_world_hit_ids with ids (i, 0, s) writes the records of rt_world_hit(segment = s) byte for
    byte; rt_shade_ids with those ids gives rt_shade's rays, beta, radiance and state, and advances ids.segment exactly on the rows that
    leave alive.  rt_camera_rays_ids with (i, s, any) is rt_camera_rays(s) for every stratum."""
    hs = make_scene(rt, name)
    sc = rt.Scene(hs)
    cam = hs.camera
    seed = 23
    n = cam.image_width * cam.image_height
    rng = np.random.default_rng(4)
    for s in range(cam.sqrt_spp ** 2):
        ids = make_ids(rt, np.arange(n), s, rng.integers(0, 2 ** 32, n, dtype=np.uint32))
        assert rt.camera_rays_ids(cam, seed, ids).tobytes() == rt.camera_rays(cam, seed, s).tobytes(), s
    rays = rt.camera_rays(cam, seed, 0)
    beta, radiance = np.ones((n, 3)), np.zeros((n, 3))
    state = np.full(n, rt.RT_PATH_ALIVE, np.uint8)
    media_rows = 0
    for seg in range(cam.max_depth):
        live = (state & rt.RT_PATH_ALIVE) != 0
        t_max = np.where(live, np.inf, np.nan)
        ids = make_ids(rt, np.arange(n), 0, seg)
        rec, st = sc.world_hit(rays, t_min=1e-8, t_max=t_max, seed=seed, segment=seg)
        rec_ids, st_ids = sc.world_hit_ids(rays, ids, t_min=1e-8, t_max=t_max, seed=seed)
        assert rec.tobytes() == rec_ids.tobytes(), f"{name}: records differ in segment {seg}"
        assert (st_ids.segments, st_ids.kernel_launches) == (st.segments, st.kernel_launches) == (n, 2)
        media_rows += int((rec["kind"] == rt.RT_HIT_MEDIUM).sum())
        r2, b2, rad2, s2, ids2 = rays.copy(), beta.copy(), radiance.copy(), state.copy(), ids.copy()
        st = sc.shade(rec, rays, beta, radiance, state, seed=seed, segment=seg, camera=cam)
        st2 = sc.shade_ids(rec, ids2, r2, b2, rad2, s2, seed=seed, camera=cam)
        for a, b_ in ((rays, r2), (beta, b2), (radiance, rad2), (state, s2)):
            assert a.tobytes() == b_.tobytes(), f"{name}: shade differs in segment {seg}"
        assert (st2.segments, st2.errors, st2.kernel_launches) == (st.segments, st.errors, st.kernel_launches)
        went_on = live & ((state & rt.RT_PATH_ALIVE) != 0)
        assert np.array_equal(ids2["segment"], np.where(went_on, seg + 1, seg))
        for f in ("pixel", "sample", "reserved"):
            assert np.array_equal(ids2[f], ids[f])
        if not went_on.any():
            break
    if name in ("book2_final", "final_reduced", "random_graph"):
        assert media_rows > 0, name


@pytest.mark.gpu
@pytest.mark.parametrize("sqrt_spp", [2, 3])
@pytest.mark.parametrize("seed", [3, 0x9E3779B97F4A7C15])
@pytest.mark.parametrize("name", SCENES)
def test_every_stratum_equals_the_render_of_that_sample(gpu, rt, name, seed, sqrt_spp):
    """For every stratum s, the loop with ids (i, s, segment) gives radiance * pixel_sample_scale bit for bit equal to rt_render with
    sample_begin = s, sample_end = s + 1 (one path per pixel: the render's sum has a fixed order), and the render's segments and errors."""
    hs = make_scene(rt, name)
    sc = rt.Scene(hs)
    cam = camera_at(rt, hs, sqrt_spp)
    W, H = cam.image_width, cam.image_height
    for s in range(sqrt_spp * sqrt_spp):
        radiance, segments, errors = stratum_loop(rt, sc, cam, seed, s)
        img = (radiance * cam.pixel_sample_scale).reshape(H, W, 3)
        ref, st = sc.render(camera=cam, seed=seed, sample_begin=s, sample_end=s + 1)
        assert st.paths == W * H
        assert (segments, errors) == (st.segments, st.errors), (s, segments, st.segments, errors, st.errors)
        eq = (bits(img) == bits(ref)).all(axis=2)
        assert eq.all(), f"{name} stratum {s}: {int((~eq).sum())} of {eq.size} pixels are not bit-equal to rt_render"


def compacting_loop(rt, sc, cam, seed, capacity, order, each_iteration=None):
    """All paths (pixel, stratum) of the image in the queue order `order` (indices into pixel * spp + stratum), through one batch
    of `capacity` rows that is compacted and refilled after every segment.  Returns (radiance of each path by path index, framebuffer
    by pixel, segments, errors, the largest number of distinct segments in one launch)."""
    spp = cam.sqrt_spp ** 2
    n_paths = len(order)
    path_rad = np.full((n_paths, 3), np.nan)
    fb = np.zeros((cam.image_width * cam.image_height, 3))
    ids = np.zeros(0, rt.rt_path_id_dtype)
    rays = np.zeros(0, rt.rt_ray_dtype)
    beta, radiance = np.zeros((0, 3)), np.zeros((0, 3))
    head = segments = errors = mixed = 0
    while head < n_paths or len(ids):
        take = order[head:head + capacity - len(ids)]
        head += len(take)
        new_ids = make_ids(rt, take // spp, take % spp)
        ids = np.concatenate([ids, new_ids])
        rays = np.concatenate([rays, rt.camera_rays_ids(cam, seed, new_ids)])
        beta = np.concatenate([beta, np.ones((len(take), 3))])
        radiance = np.concatenate([radiance, np.zeros((len(take), 3))])
        n = len(ids)
        state = np.full(n, rt.RT_PATH_ALIVE, np.uint8)
        mixed = max(mixed, len(np.unique(ids["segment"])))
        reserved = ids["reserved"].copy()
        rec, _ = sc.world_hit_ids(rays, ids, t_min=1e-8, seed=seed)
        st = sc.shade_ids(rec, ids, rays, beta, radiance, state, seed=seed, camera=cam)
        assert st.segments == n and np.array_equal(ids["reserved"], reserved)
        segments += n
        errors += st.errors
        done = (state & rt.RT_PATH_ALIVE) == 0
        if each_iteration is not None:
            each_iteration(n, int(done.sum()))
        path_rad[ids["pixel"][done].astype(np.int64) * spp + ids["sample"][done]] = radiance[done]
        np.add.at(fb, ids["pixel"][done].astype(np.int64), radiance[done])
        keep = ~done
        ids, rays, beta, radiance = ids[keep], rays[keep], beta[keep], radiance[keep]
    return path_rad, fb, segments, errors, mixed


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cornell_glass", "book2_final", "random_graph"])
def test_compaction_permutation_and_refill(gpu, rt, name):
    """One batch smaller than the number of paths holds every stratum in shuffled order; finished rows leave and new ones come in after
    every segment, so rows at different segments share a launch.  Each path's radiance is bit for bit the value the render gives for
    its sample alone, the framebuffer matches the full render, and segments and errors are the render's."""
    hs = make_scene(rt, name)
    sc = rt.Scene(hs)
    cam = camera_at(rt, hs, 2)
    W, H, spp, seed = cam.image_width, cam.image_height, 4, 31
    n_paths = W * H * spp
    order = np.random.default_rng(8).permutation(n_paths)
    sizes = []
    path_rad, fb, segments, errors, mixed = compacting_loop(rt, sc, cam, seed, n_paths // 3 + 17, order,
                                                            lambda n, d: sizes.append((n, d)))
    assert not np.isnan(path_rad).any()
    assert mixed > 1 and any(d and n == n_paths // 3 + 17 for n, d in sizes[:-1])
    for s in range(spp):
        ref_s, _ = sc.render(camera=cam, seed=seed, sample_begin=s, sample_end=s + 1)
        got = (path_rad[np.arange(W * H) * spp + s] * cam.pixel_sample_scale).reshape(H, W, 3)
        eq = (bits(got) == bits(ref_s)).all(axis=2)
        assert eq.all(), f"{name} stratum {s}: {int((~eq).sum())} paths differ from their render"
    ref, st = sc.render(camera=cam, seed=seed)
    img = (fb * cam.pixel_sample_scale).reshape(H, W, 3)
    assert np.allclose(img, ref, rtol=1e-11, atol=1e-13)
    assert (segments, errors) == (st.segments, st.errors) and st.paths == n_paths


@pytest.mark.gpu
def test_row_rules(gpu, rt, orc):
    """A live row at segment >= max_depth ends with RT_PATH_ERROR and nothing else of it changes; inactive rows are untouched, ids
    included; `reserved` is never written; the other rows are as in a batch without those rows."""
    hs = make_scene(rt, "book2_final")
    sc = rt.Scene(hs)
    cam = camera_at(rt, hs, 2)
    n = cam.image_width * cam.image_height
    seed = 12
    rng = np.random.default_rng(3)
    ids = make_ids(rt, rng.permutation(n), rng.integers(0, 4, n), rng.integers(0, cam.max_depth, n),
                   rng.integers(0, 2 ** 32, n, dtype=np.uint32))
    rays = rt.camera_rays_ids(cam, seed, ids)
    rec, _ = sc.world_hit_ids(rays, ids, seed=seed)
    inactive = rng.uniform(size=n) < 0.2
    deep = ~inactive & (rng.uniform(size=n) < 0.2)
    state0 = np.where(inactive, rng.choice([0, 2, 0xFC], n), rt.RT_PATH_ALIVE | rng.choice([0, 0xFC], n)).astype(np.uint8)
    deep_ids = ids.copy()
    deep_ids["segment"][deep] = cam.max_depth + rng.integers(0, 2, deep.sum()) * rng.integers(0, 2 ** 31, deep.sum())

    def run(pid, state):
        r, bt, rad, s, i2 = rays.copy(), np.full((n, 3), 0.5), np.full((n, 3), 0.25), state.copy(), pid.copy()
        for a in (r, bt, rad):
            a.view(np.uint8).reshape(n, -1)[inactive] = 0xA5
        st = sc.shade_ids(rec, i2, r, bt, rad, s, seed=seed, camera=cam)
        return r, bt, rad, s, i2, st

    base = run(ids, np.where(deep, 0, state0).astype(np.uint8))
    got = run(deep_ids, state0)
    r, bt, rad, s, i2, st = got
    assert (s[deep] == rt.RT_PATH_ERROR).all()
    assert r[deep].tobytes() == rays[deep].tobytes() and (bt[deep] == 0.5).all() and (rad[deep] == 0.25).all()
    assert i2[deep].tobytes() == deep_ids[deep].tobytes()
    assert np.array_equal(s[inactive], state0[inactive]) and i2[inactive].tobytes() == ids[inactive].tobytes()
    for a in (r, bt, rad):
        assert (a.view(np.uint8).reshape(n, -1)[inactive] == 0xA5).all()
    assert np.array_equal(i2["reserved"], ids["reserved"])
    rest = ~deep
    for a, b_ in zip(got[:5], base[:5]):
        assert a[rest].tobytes() == b_[rest].tobytes()
    assert st.errors == base[5].errors + int(deep.sum()) == int(((s & rt.RT_PATH_ERROR) != 0)[~inactive].sum())
    assert (s[~inactive & ~deep] & 1).any()


@pytest.mark.gpu
def test_out_of_range_ids_give_the_camera_arithmetic(gpu, rt, orc):
    """Pixels beyond the image and strata >= sqrt_spp^2 are addresses like any other: the ray is Camera::get_ray of (p % W, p / W)
    and stratum (s / sqrt_spp, s % sqrt_spp), bit for bit the oracle's, and the in-image rows of a taller camera."""
    b = rt.Builder(1)
    hs = b.finish(b.list([b.sphere([0, 0, 0], 1.0, b.lambertian(b.solid(0.5, 0.5, 0.5)))]), width=24, aspect=24 / 17, spp=9, vfov=40,
                  look_from=(0.3, 1.1, 7), look_at=(0, 0, 0))
    cam = hs.camera
    W, H = cam.image_width, cam.image_height
    pixel = np.array([0, W * H - 1, W * H, W * H + 5, W * (H + 2) + 3, 2 ** 31, 2 ** 32 - 1] * 3, np.uint32)
    sample = np.array([0] * 7 + [9] * 7 + [2 ** 32 - 1] * 7, np.uint32)
    ids = make_ids(rt, pixel, sample, 2 ** 32 - 1)
    for seed in (0, 2 ** 64 - 1):
        got = rt.camera_rays_ids(cam, seed, ids)
        want = np.concatenate([orc.camera_rays(cam, seed, [(p % W, p // W)], s) for p, s in zip(pixel.tolist(), sample.tolist())])
        assert got.tobytes() == want.tobytes()
        tall = rt.rt_camera.from_buffer_copy(cam)
        tall.image_height = H + 3
        below = np.arange(W * H, W * (H + 3))
        got = rt.camera_rays_ids(cam, seed, make_ids(rt, below, 4))
        assert got.tobytes() == rt.camera_rays(tall, seed, 4)[below].tobytes()


@pytest.mark.gpu
def test_device_entries_on_a_torch_stream(gpu, rt):
    """The compacting loop on device buffers, with torch doing the gathers on the same stream, equals the host-pointer loop."""
    import torch
    hs = make_scene(rt, "random_graph")
    sc = rt.Scene(hs)
    cam = camera_at(rt, hs, 2)
    seed, spp = 6, 4
    n_paths = cam.image_width * cam.image_height * spp
    cap = n_paths // 4
    order = np.arange(n_paths)
    _, want_fb, want_segments, want_errors, _ = compacting_loop(rt, sc, cam, seed, cap, order)
    dev = "cuda"
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    segments = errors = 0
    with torch.cuda.stream(s):
        d_ids = torch.zeros((cap, 4), dtype=torch.int32, device=dev)
        d_rays = torch.empty((cap, 7), dtype=torch.float64, device=dev)
        d_rec = torch.empty((cap, rt.rt_hit_record_dtype.itemsize), dtype=torch.uint8, device=dev)
        d_beta = torch.ones((cap, 3), dtype=torch.float64, device=dev)
        d_rad = torch.zeros((cap, 3), dtype=torch.float64, device=dev)
        d_state = torch.empty(cap, dtype=torch.uint8, device=dev)
        fb = torch.zeros((cam.image_width * cam.image_height, 3), dtype=torch.float64, device=dev)
        live = head = 0
        while head < n_paths or live:
            k = min(cap - live, n_paths - head)
            if k:
                q = torch.arange(head, head + k, device=dev, dtype=torch.int64)
                d_ids[live:live + k, 0] = (q // spp).to(torch.int32)
                d_ids[live:live + k, 1] = (q % spp).to(torch.int32)
                d_ids[live:live + k, 2:] = 0
                rt.camera_rays_ids_device(cam, seed, d_ids[live:].data_ptr(), k, d_rays[live:].data_ptr(), stream=s.cuda_stream)
                d_beta[live:live + k] = 1.0
                d_rad[live:live + k] = 0.0
                head += k
                live += k
            d_state[:live] = rt.RT_PATH_ALIVE
            sc.world_hit_ids_device(d_rays.data_ptr(), d_ids.data_ptr(), live, d_rec.data_ptr(), seed=seed, stream=s.cuda_stream)
            st = sc.shade_ids_device(d_rec.data_ptr(), d_ids.data_ptr(), live, d_rays.data_ptr(), d_beta.data_ptr(), d_rad.data_ptr(),
                                     d_state.data_ptr(), seed=seed, camera=cam, stream=s.cuda_stream)
            assert st.segments == live
            segments += live
            errors += st.errors
            alive = (d_state[:live] & rt.RT_PATH_ALIVE) != 0
            done = ~alive
            fb.index_add_(0, d_ids[:live, 0][done].to(torch.int64), d_rad[:live][done])
            keep = torch.nonzero(alive).squeeze(1)
            n_keep = int(keep.numel())
            for t in (d_ids, d_rays, d_beta, d_rad):
                t[:n_keep] = t[:live][keep]
            live = n_keep
    s.synchronize()
    assert (segments, errors) == (want_segments, want_errors)
    # index_add_ and np.add.at may sum the samples of a pixel in different orders
    assert np.allclose(fb.cpu().numpy(), want_fb, rtol=1e-12, atol=1e-14)
