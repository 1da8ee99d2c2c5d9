#!/usr/bin/env python
"""bench_world_hit.py — the world-hit query (the reference's HitRecord, media sampled) against the closest-hit query on the same
batch, 2^24 rays in HBM, on three cases:

  book2_final      the bench scene (sphere-bounded media: the global mist and the subsurface ball).  Incoherent rays: origins
                   uniform in [0, 555]^3, directions uniform on the sphere, t_max = inf.
  final_reduced    config 4 on the shipped assets (a fog mesh: the general-boundary record pass).  Segments between two uniform
                   points of the box x, z in [-2.5, 2.5], y in [-1.5, 5.5] around the fog mesh: unit direction, per-ray
                   t_max_i = |b - a| (1 - 1e-6) for world hit; closest hit, which has no per-ray bound, runs with t_max = inf.
  tri_soup         1M random triangles in the unit cube (config 5), media-free, incoherent rays as in bench_closest_hit.py, t_max = inf:
                   what the 96-byte record, the 16-byte scratch hit and the second launch cost over closest hit.

One JSON line per case: both rates in Mrays/s and their time ratio, the hit / medium / miss fractions, nodes and primitives per ray
of both queries (RT_OPT_COUNT instantiations), on media-free scenes the device parity of (t, prim_id) with closest hit on every ray,
and the oracle parity on the first `--oracle-rays` rays (mismatches of kind, ids, material or front face; max relative error of t
and p; surface t bit-exact).

    python bench_world_hit.py [--cases book2_final final_reduced tri_soup] [--rays 16777216] [--oracle-rays 100000]

Timing is CUDA events around each _device call (stats.ms_total; both launches for rt_world_hit), best of 5 after 2 warm-ups, the
two queries alternating.  The card's name, power limit and maximum SM clock are read in the same run.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

from bench_closest_hit import make_rays, rt
from bench_occluded import gpu_description
from bench_transmittance import segments

ROOT = os.path.dirname(os.path.abspath(__file__))


def scene_and_rays(torch, name, n):
    if name == "book2_final":
        hs = rt.named_scene("book2_final", seed=7, params=[800, 1000, 40])
        g = torch.Generator(device="cuda").manual_seed(11)
        rays = torch.zeros((n, 7), dtype=torch.float64, device="cuda")
        rays[:, 0:3] = torch.rand((n, 3), generator=g, device="cuda", dtype=torch.float64) * 555.0
        d = torch.randn((n, 3), generator=g, device="cuda", dtype=torch.float64)
        rays[:, 3:6] = d / d.norm(dim=1, keepdim=True)
        rays[:, 6] = torch.rand(n, generator=g, device="cuda", dtype=torch.float64)
        return hs, rays, None, "incoherent: origins in [0,555]^3, uniform directions"
    if name == "final_reduced":
        from scenes_util import final_reduced_scene  # tests/ is on sys.path (main)
        hs = final_reduced_scene(rt, width=1920, spp=256, depth=30)
        rays, t_max = segments(torch, n, 11, [-2.5, -1.5, -2.5], [2.5, 5.5, 2.5])
        return hs, rays, t_max, "segments between uniform points of x,z in [-2.5,2.5], y in [-1.5,5.5] (around the fog mesh)"
    hs = rt.named_scene("tri_soup", seed=5, params=[1_000_000])
    return hs, make_rays(torch, n, "incoherent", 11), None, "incoherent: origins in the unit cube, uniform directions"


def oracle_parity(hs, sample, t_max, got):
    from world_hit_oracle import WorldHitOracle
    want = WorldHitOracle(hs).world_hit(sample, t_max=float("inf") if t_max is None else t_max, seed=1, segment=0)
    ids = np.zeros(len(got), dtype=bool)
    for f in ("kind", "prim_id", "inst_id", "material", "front_face"):
        ids |= got[f] != want[f]
    ok = ~ids & (want["kind"] != rt.RT_HIT_MISS)
    rel_t = np.abs(got["t"][ok] - want["t"][ok]) / np.abs(want["t"][ok])
    pn = np.linalg.norm(want["p"][ok], axis=1)
    rel_p = np.abs(got["p"][ok] - want["p"][ok]).max(axis=1) / np.where(pn > 0, pn, 1.0)
    surf = ok & (want["kind"] == rt.RT_HIT_SURFACE)
    return {"rays": len(got), "id_mismatches": int(ids.sum()), "max_rel_err_t": float(rel_t.max()) if rel_t.size else 0.0,
            "max_rel_err_p": float(rel_p.max()) if rel_p.size else 0.0,
            "surface_t_bit_exact": bool(np.array_equal(got["t"][surf].view(np.int64), want["t"][surf].view(np.int64)))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", nargs="+", default=["book2_final", "final_reduced", "tri_soup"])
    ap.add_argument("--rays", type=int, default=1 << 24)
    ap.add_argument("--oracle-rays", type=int, default=100_000)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: the product has no CPU path")
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    gpu = gpu_description(torch, 0)
    stream = torch.cuda.current_stream().cuda_stream
    n = args.rays
    rec_bytes = rt.rt_hit_record_dtype.itemsize
    for name in args.cases:
        hs, rays, t_max, ray_set = scene_and_rays(torch, name, n)
        t0 = time.perf_counter()
        sc = rt.Scene(hs, device=0)
        t_build = time.perf_counter() - t0
        info = sc.info()
        recs = torch.empty(n * rec_bytes, dtype=torch.uint8, device="cuda")
        hits = torch.empty((n, 3), dtype=torch.float64, device="cuda")  # 24-byte rt_hit records
        t_max_ptr = None if t_max is None else t_max.data_ptr()
        run_wh = lambda flags=0: sc.world_hit_device(rays.data_ptr(), n, recs.data_ptr(), t_max_ptr, seed=1, segment=0, flags=flags,  # noqa: E731
                                                     stream=stream)
        run_ch = lambda flags=0: sc.closest_hit_device(rays.data_ptr(), n, hits.data_ptr(), flags=flags, stream=stream)  # noqa: E731
        ms_wh, ms_ch = float("inf"), float("inf")
        for k in range(7):  # alternating, best of 5 after 2 warm-ups
            torch.cuda.synchronize()
            a = run_wh().ms_total
            b = run_ch().ms_total
            if k >= 2:
                ms_wh, ms_ch = min(ms_wh, a), min(ms_ch, b)
        c_wh, c_ch = run_wh(rt.RT_OPT_COUNT), run_ch(rt.RT_OPT_COUNT)
        torch.cuda.synchronize()
        words = recs.view(torch.int32).view(n, rec_bytes // 4)
        kind = words[:, 18]  # rt_hit_record.kind at byte 72
        fractions = {k: float((kind == v).float().mean().item()) for k, v in
                     (("surface", rt.RT_HIT_SURFACE), ("medium", rt.RT_HIT_MEDIUM), ("miss", rt.RT_HIT_MISS))}
        device_parity = None
        if info.n_media == 0:  # the same (t, prim_id) as closest hit on every ray
            t_rec = recs.view(torch.float64).view(n, rec_bytes // 8)[:, 0]
            same = (t_rec == hits[:, 0]) & (words[:, 20] == hits.view(torch.int32)[:, 2])
            device_parity = {"rays": n, "mismatches": int((~same).sum().item())}
        m = min(args.oracle_rays, n)
        sample = np.ascontiguousarray(rays[:m].cpu().numpy()).view(rt.rt_ray_dtype).reshape(m)
        got = recs[:m * rec_bytes].cpu().numpy().view(rt.rt_hit_record_dtype)
        parity = oracle_parity(hs, sample, None if t_max is None else t_max[:m].cpu().numpy(), got)
        line = {"metric": "world_hit_mrays_per_sec", "value": n / ms_wh / 1e3, "unit": "Mrays/s", "n_gpus": 1, "dtype": "f64",
                "config": {"workload": f"{name} rays={n}", "rays": ray_set, "t_max": "inf" if t_max is None else "per ray", "n_media": info.n_media,
                           "bvh_nodes": info.n_nodes, "node_bytes": info.node_bytes, "scene_create_s": t_build},
                "gpu": gpu, "ms": ms_wh,
                "nodes_per_ray": c_wh.node_visits / n, "prims_per_ray": c_wh.prim_tests / n,
                "fractions": fractions,
                "closest_hit": {"value": n / ms_ch / 1e3, "unit": "Mrays/s", "ms": ms_ch, "t_max": "inf",
                                "nodes_per_ray": c_ch.node_visits / n, "prims_per_ray": c_ch.prim_tests / n},
                "time_ratio_vs_closest_hit": ms_wh / ms_ch,
                "device_parity_vs_closest_hit": device_parity,
                "oracle_parity": parity}
        print(json.dumps(line), flush=True)
        sc.close()
        del sc, rays, t_max, recs, hits, words, kind


if __name__ == "__main__":
    main()
