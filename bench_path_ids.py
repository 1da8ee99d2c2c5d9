#!/usr/bin/env python
"""bench_path_ids.py — a compacting, refilling client path loop on the path-id entries against rt_render, at several samples per
pixel, on device buffers.  One batch of --capacity rows; each iteration:

    refill the free tail with the next (pixel, stratum) ids of the queue, rt_camera_rays_ids_device for them (beta 1, radiance 0);
    rt_world_hit_ids_device(t_min = 1e-8) and rt_shade_ids_device on every row (all rows of the batch are live);
    torch: index_add_ the radiance of the rows that finished into a binary64 framebuffer by pixel, count their error bits, and
    gather the survivors (rays, beta, radiance, ids) to the front of the batch; the survivor count is the one look at the host

until the queue is empty and no row is left; then the framebuffer is scaled by pixel_sample_scale.  Against rt_render_device of the
same camera (binary64 accumulation), on two cases:

  book2_final     800 x 800, sqrt_spp 4, max_depth 40
  cornell_glass   the scene's own camera at sqrt_spp 4

One JSON line per case: both times, paths/s and segments/s (world.hit calls) of both, the loop / render time ratio, the loop's
segments, errors and iterations next to the render's rt_stats, and the image parity in the same run: allclose(rtol=1e-11,
atol=1e-13), max |difference| and the bit-equal pixels (reported, not required: the render sums a pixel's samples with atomics in
no fixed order).  Timing: CUDA events around the whole loop (host loop included) and around rt_render_device, best of --repeats
after one warm-up, the two alternating.  The card's name, power limit and maximum SM clock are read in the same run.

    python bench_path_ids.py [--cases book2_final cornell_glass] [--repeats 3] [--capacity 4194304]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "raytracer-2025_b200"))
import rt2025 as rt  # noqa: E402
from bench_occluded import gpu_description  # noqa: E402


def make_case(name):
    if name == "book2_final":
        hs = rt.named_scene("book2_final", seed=7, params=[800, 16, 40])
    else:
        hs = rt.named_scene("cornell_glass", seed=7)
    cam = rt.rt_camera.from_buffer_copy(hs.camera)
    cam.sqrt_spp, cam.recip_sqrt_spp, cam.pixel_sample_scale = 4, 0.25, 1.0 / 16
    return hs, cam


def path_loop(torch, L, sc, cam, seed, bufs, fb):
    """The loop of the module docstring.  Returns (segments, errors, iterations); the framebuffer sum is left in fb (unscaled)."""
    d_ids, d_rays, d_rec, d_beta, d_rad, d_state = bufs
    cap = d_ids.shape[0]
    spp = cam.sqrt_spp * cam.sqrt_spp
    n_paths = cam.image_width * cam.image_height * spp
    fb.zero_()
    d_errors = torch.zeros((), dtype=torch.int64, device="cuda")
    live = head = segments = iterations = 0
    while head < n_paths or live:
        k = min(cap - live, n_paths - head)
        if k:
            q = torch.arange(head, head + k, device="cuda", dtype=torch.int64)
            d_ids[live:live + k, 0] = (q // spp).to(torch.int32)
            d_ids[live:live + k, 1] = (q % spp).to(torch.int32)
            d_ids[live:live + k, 2] = 0
            _check(L.rt_camera_rays_ids_device(rt.C.byref(cam), seed, d_ids[live:].data_ptr(), k, d_rays[live:].data_ptr(), None), L)
            d_beta[live:live + k] = 1.0
            d_rad[live:live + k] = 0.0
            head += k
            live += k
        d_state[:live] = rt.RT_PATH_ALIVE
        # no stats: the entries would wait for their own events; the errors are counted on the device from the state bits
        _check(L.rt_world_hit_ids_device(sc.h, d_rays.data_ptr(), d_ids.data_ptr(), None, live, 1e-8, float("inf"), seed, 0,
                                         d_rec.data_ptr(), None, None), L)
        _check(L.rt_shade_ids_device(sc.h, rt.C.byref(cam), d_rec.data_ptr(), d_ids.data_ptr(), live, seed, 0, d_rays.data_ptr(),
                                     d_beta.data_ptr(), d_rad.data_ptr(), d_state.data_ptr(), None, None), L)
        segments += live
        iterations += 1
        st = d_state[:live]
        alive = (st & rt.RT_PATH_ALIVE) != 0
        d_errors += ((st & rt.RT_PATH_ERROR) != 0).sum()
        done = ~alive
        fb.index_add_(0, d_ids[:live, 0][done].to(torch.int64), d_rad[:live][done])
        keep = torch.nonzero(alive).squeeze(1)  # the look at the host: the survivor count
        n_keep = int(keep.numel())
        for t in (d_ids, d_rays, d_beta, d_rad):
            t[:n_keep] = t[:live][keep]
        live = n_keep
    return segments, int(d_errors), iterations


def _check(rc, L):
    if rc != 0:
        raise RuntimeError(f"rt2025 error {rc}: {L.rt_last_error().decode()}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", nargs="+", default=["book2_final", "cornell_glass"])
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--capacity", type=int, default=1 << 22, help="rows of the loop's batch")
    ap.add_argument("--seed", type=int, default=1)
    args = ap.parse_args()
    import torch
    L = rt.product_lib()
    if not torch.cuda.is_available() or L.rt_device_count() < 1:
        raise SystemExit("bench_path_ids.py: no CUDA device (the product has no CPU path)")
    gpu = gpu_description(torch, torch.cuda.current_device())
    for name in args.cases:
        hs, cam = make_case(name)
        sc = rt.Scene(hs)
        n_px = cam.image_width * cam.image_height
        n_paths = n_px * cam.sqrt_spp * cam.sqrt_spp
        cap = min(args.capacity, n_paths)
        bufs = (torch.zeros((cap, 4), dtype=torch.int32, device="cuda"), torch.empty((cap, 7), dtype=torch.float64, device="cuda"),
                torch.empty((cap, rt.rt_hit_record_dtype.itemsize), dtype=torch.uint8, device="cuda"),
                torch.empty((cap, 3), dtype=torch.float64, device="cuda"), torch.empty((cap, 3), dtype=torch.float64, device="cuda"),
                torch.empty(cap, dtype=torch.uint8, device="cuda"))
        fb = torch.zeros((n_px, 3), dtype=torch.float64, device="cuda")
        d_accum = torch.empty(n_px * 3, dtype=torch.float64, device="cuda")
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_loop, t_render = [], []
        for rep in range(args.repeats + 1):  # the first round warms both up
            e0.record()
            segments, errors, iterations = path_loop(torch, L, sc, cam, args.seed, bufs, fb)
            e1.record()
            torch.cuda.synchronize()
            if rep:
                t_loop.append(e0.elapsed_time(e1))
            e0.record()
            rst = sc.render_device(d_accum.data_ptr(), camera=cam, seed=args.seed)
            e1.record()
            torch.cuda.synchronize()
            if rep:
                t_render.append(e0.elapsed_time(e1))
        img = (fb * cam.pixel_sample_scale).cpu().numpy().reshape(-1, 3)
        ref = d_accum.cpu().numpy().reshape(-1, 3)
        eq = (img.view(np.int64) == ref.view(np.int64)).all(axis=1)
        lo, lr = min(t_loop), min(t_render)
        line = dict(case=name, width=cam.image_width, height=cam.image_height, sqrt_spp=cam.sqrt_spp, max_depth=cam.max_depth, paths=n_paths,
                    capacity=cap, gpu=gpu, loop_ms=round(lo, 3), render_ms=round(lr, 3), loop_over_render=round(lo / lr, 3),
                    loop_ms_all=[round(t, 3) for t in t_loop], render_ms_all=[round(t, 3) for t in t_render],
                    loop_paths_per_s=round(n_paths / lo * 1e3), render_paths_per_s=round(n_paths / lr * 1e3),
                    loop_segments_per_s=round(segments / lo * 1e3), render_segments_per_s=round(rst.segments / lr * 1e3),
                    segments=segments, render_segments=int(rst.segments), errors=errors, render_errors=int(rst.errors),
                    render_paths=int(rst.paths), iterations=iterations, bit_equal_pixels=int(eq.sum()), pixels=n_px,
                    max_abs_diff=float(np.max(np.abs(img - ref))), parity=bool(np.allclose(img, ref, rtol=1e-11, atol=1e-13)))
        print(json.dumps(line), flush=True)
        sc.close()


if __name__ == "__main__":
    main()
