#!/usr/bin/env python
"""bench_shade.py — a client path loop on the public ray queries against rt_render, one sample per pixel, on device buffers:

    rt_camera_rays_device(sample 0); then per segment: t_max_i = inf for live paths, NaN for finished ones (a torch kernel),
    rt_world_hit_device(t_min = 1e-8), rt_shade_device; until no path is alive or max_depth segments ran

against rt_render_device of the same camera (sqrt_spp = 1, pixel_sample_scale = 1, binary64 accumulation), on two cases:

  book2_final     800 x 800, max_depth 40 (the bench scene at one sample per pixel)
  cornell_glass   the scene's own camera, one sample per pixel

One JSON line per case: both times and paths/s, segments/s (world.hit calls) of both, rt_shade rays/s (rows with a live path over
the rt_shade time alone), the loop / render time ratio, and the image parity in the same run (max |difference|, bit-equal
pixels, the errors of both).  Timing: CUDA events around the whole loop (host loop included: a client has to look at the state to
know when to stop, here after every segment) and around rt_render_device, best of --repeats after one warm-up, the two alternating.
The card's name, power limit and maximum SM clock are read in the same run.

    python bench_shade.py [--cases book2_final cornell_glass] [--repeats 5]
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
        hs = rt.named_scene("book2_final", seed=7, params=[800, 1, 40])
    else:
        hs = rt.named_scene("cornell_glass", seed=7)
    cam = rt.rt_camera.from_buffer_copy(hs.camera)
    cam.sqrt_spp, cam.recip_sqrt_spp, cam.pixel_sample_scale = 1, 1.0, 1.0
    return hs, cam


def client_loop(torch, sc, cam, seed, bufs):
    """The loop on device buffers; returns (segments traced, errors, ms in rt_shade)."""
    n = cam.image_width * cam.image_height
    d_rays, d_rec, d_beta, d_rad, d_state, d_tmax = bufs
    d_beta.fill_(1.0)
    d_rad.zero_()
    d_state.fill_(rt.RT_PATH_ALIVE)
    inf = torch.tensor(float("inf"), dtype=torch.float64, device="cuda")
    nan = torch.tensor(float("nan"), dtype=torch.float64, device="cuda")
    rt.camera_rays_device(cam, seed, 0, d_rays.data_ptr())
    segments = errors = 0
    ms_shade = 0.0
    for seg in range(cam.max_depth):
        live = (d_state & 1) != 0
        n_live = int(live.sum())  # the client's look at the state: one synchronisation per segment
        if n_live == 0:
            break
        segments += n_live
        torch.where(live, inf, nan, out=d_tmax)
        sc.world_hit_device(d_rays.data_ptr(), n, d_rec.data_ptr(), d_tmax.data_ptr(), t_min=1e-8, seed=seed, segment=seg)
        st = sc.shade_device(d_rec.data_ptr(), n, d_rays.data_ptr(), d_beta.data_ptr(), d_rad.data_ptr(), d_state.data_ptr(), seed=seed,
                             segment=seg, camera=cam)
        errors += st.errors
        ms_shade += st.ms_total
    return segments, errors, ms_shade


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", nargs="+", default=["book2_final", "cornell_glass"])
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--seed", type=int, default=1)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available() or rt.product_lib().rt_device_count() < 1:
        raise SystemExit("bench_shade.py: no CUDA device (the product has no CPU path)")
    gpu = gpu_description(torch, torch.cuda.current_device())
    for name in args.cases:
        hs, cam = make_case(name)
        sc = rt.Scene(hs)
        n = cam.image_width * cam.image_height
        bufs = (torch.empty(n * 7, dtype=torch.float64, device="cuda"),
                torch.empty(n * rt.rt_hit_record_dtype.itemsize, dtype=torch.uint8, device="cuda"),
                torch.empty(n * 3, dtype=torch.float64, device="cuda"), torch.empty(n * 3, dtype=torch.float64, device="cuda"),
                torch.empty(n, dtype=torch.uint8, device="cuda"), torch.empty(n, dtype=torch.float64, device="cuda"))
        d_accum = torch.empty(n * 3, dtype=torch.float64, device="cuda")
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_loop, t_render, t_shade = [], [], []
        for rep in range(args.repeats + 1):  # the first round warms both up
            e0.record()
            segments, errors, ms_shade = client_loop(torch, sc, cam, args.seed, bufs)
            e1.record()
            torch.cuda.synchronize()
            if rep:
                t_loop.append(e0.elapsed_time(e1))
                t_shade.append(ms_shade)
            e0.record()
            rst = sc.render_device(d_accum.data_ptr(), camera=cam, seed=args.seed)
            e1.record()
            torch.cuda.synchronize()
            if rep:
                t_render.append(e0.elapsed_time(e1))
        img = bufs[3].cpu().numpy()
        ref = d_accum.cpu().numpy()
        eq = (img.reshape(-1, 3).view(np.int64) == ref.reshape(-1, 3).view(np.int64)).all(axis=1)
        lo, lr, ls = min(t_loop), min(t_render), min(t_shade)
        line = dict(case=name, width=cam.image_width, height=cam.image_height, max_depth=cam.max_depth, paths=n, gpu=gpu,
                    loop_ms=round(lo, 3), render_ms=round(lr, 3), loop_over_render=round(lo / lr, 3),
                    loop_paths_per_s=round(n / lo * 1e3), render_paths_per_s=round(n / lr * 1e3),
                    segments=segments, render_segments=int(rst.segments), loop_segments_per_s=round(segments / lo * 1e3),
                    render_segments_per_s=round(rst.segments / lr * 1e3), shade_ms=round(ls, 3), shade_rays_per_s=round(segments / ls * 1e3),
                    errors=int(errors), render_errors=int(rst.errors), bit_equal_pixels=int(eq.sum()),
                    max_abs_diff=float(np.max(np.abs(img - ref))), parity=bool(np.allclose(img, ref, rtol=1e-11, atol=1e-13)))
        print(json.dumps(line), flush=True)
        sc.close()


if __name__ == "__main__":
    main()
