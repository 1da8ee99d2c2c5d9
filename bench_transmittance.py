#!/usr/bin/env python
"""bench_transmittance.py — the transmittance query (visibility through media) against the occlusion query on the same batch,
2^24 segments in HBM, on two scenes with media:

  book2_final      the bench scene (sphere-bounded media: the global mist and the subsurface ball).  Shadow segments from a
                   uniform in [0, 555]^3 to b uniform on the ceiling light (x in [123, 423], z in [147, 412], y = 554): unit
                   direction, per-ray t_max_i = |b - a| (1 - 1e-6).
  final_reduced    config 4 on the shipped assets (a fog mesh: the general-boundary media pass).  Segments between two uniform
                   points of the box x, z in [-2.5, 2.5], y in [-1.5, 5.5], which holds the fog mesh's bounding box
                   (x, z in [-1.23, 1.23], y in [-0.33, 4.38]) and the geometry around it: unit direction, t_max_i = |b - a| (1 - 1e-6).

One JSON line per scene with the transmittance and the occlusion rate in Mrays/s (their ratio is the cost of the media pass),
the occluded fraction, the mean T of the unoccluded rays, nodes and primitives per ray of both queries, the device parity on every
ray ((T == 0) == occlusion byte, as a mismatch count) and the oracle parity on the first `--oracle-rays` rays (max relative error
of T and the count of mismatched zero patterns).

    python bench_transmittance.py [--scenes book2_final final_reduced] [--rays 16777216] [--oracle-rays 100000]

Timing is CUDA events around each _device call (stats.ms_total; both launches for rt_transmittance), best of 5 after 2 warm-ups,
the two queries alternating.  Node and primitive counts come from the RT_OPT_COUNT instantiations.  The card's name, power limit
and maximum SM clock are read in the same run.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

from bench_closest_hit import rt
from bench_occluded import gpu_description

ROOT = os.path.dirname(os.path.abspath(__file__))


def segments(torch, n, seed, lo, hi, b_lo=None, b_hi=None):
    """a uniform in [lo, hi], b uniform in [b_lo, b_hi] (default: the same box): rays a -> b with unit direction, t_max = |b - a| (1 - 1e-6)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    lo, hi = torch.tensor(lo, dtype=torch.float64, device="cuda"), torch.tensor(hi, dtype=torch.float64, device="cuda")
    b_lo = lo if b_lo is None else torch.tensor(b_lo, dtype=torch.float64, device="cuda")
    b_hi = hi if b_hi is None else torch.tensor(b_hi, dtype=torch.float64, device="cuda")
    a = lo + torch.rand((n, 3), generator=g, device="cuda", dtype=torch.float64) * (hi - lo)
    b = b_lo + torch.rand((n, 3), generator=g, device="cuda", dtype=torch.float64) * (b_hi - b_lo)
    length = (b - a).norm(dim=1)
    rays = torch.zeros((n, 7), dtype=torch.float64, device="cuda")
    rays[:, 0:3] = a
    rays[:, 3:6] = (b - a) / length[:, None]
    rays[:, 6] = torch.rand(n, generator=g, device="cuda", dtype=torch.float64)
    return rays, length * (1.0 - 1e-6)


def scene_and_rays(torch, name, n):
    if name == "book2_final":
        hs = rt.named_scene("book2_final", seed=7, params=[800, 1000, 40])
        rays, t_max = segments(torch, n, 11, [0.0, 0.0, 0.0], [555.0, 555.0, 555.0], [123.0, 554.0, 147.0], [423.0, 554.0, 412.0])
        return hs, rays, t_max, "shadow segments: a in [0,555]^3 -> b on the ceiling light"
    from scenes_util import final_reduced_scene  # tests/ is on sys.path (main)
    hs = final_reduced_scene(rt, width=1920, spp=256, depth=30)
    rays, t_max = segments(torch, n, 11, [-2.5, -1.5, -2.5], [2.5, 5.5, 2.5])
    return hs, rays, t_max, "segments between uniform points of x,z in [-2.5,2.5], y in [-1.5,5.5] (around the fog mesh)"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenes", nargs="+", default=["book2_final", "final_reduced"])
    ap.add_argument("--rays", type=int, default=1 << 24)
    ap.add_argument("--oracle-rays", type=int, default=100_000)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: the product has no CPU path")
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from transmittance_oracle import TransmittanceOracle
    gpu = gpu_description(torch, 0)
    stream = torch.cuda.current_stream().cuda_stream
    n = args.rays
    for name in args.scenes:
        hs, rays, t_max, ray_set = scene_and_rays(torch, name, n)
        t0 = time.perf_counter()
        sc = rt.Scene(hs, device=0)
        t_build = time.perf_counter() - t0
        info = sc.info()
        T = torch.empty(n, dtype=torch.float64, device="cuda")
        occ = torch.empty(n, dtype=torch.uint8, device="cuda")
        run_tr = lambda flags=0: sc.transmittance_device(rays.data_ptr(), n, T.data_ptr(), t_max.data_ptr(), flags=flags, stream=stream)
        run_occ = lambda flags=0: sc.occluded_device(rays.data_ptr(), n, occ.data_ptr(), t_max.data_ptr(), flags=flags, stream=stream)
        ms_tr, ms_occ = float("inf"), float("inf")
        for k in range(7):  # alternating, best of 5 after 2 warm-ups
            torch.cuda.synchronize()
            a = run_tr().ms_total
            b = run_occ().ms_total
            if k >= 2:
                ms_tr, ms_occ = min(ms_tr, a), min(ms_occ, b)
        c_tr, c_occ = run_tr(rt.RT_OPT_COUNT), run_occ(rt.RT_OPT_COUNT)
        torch.cuda.synchronize()
        # device parity on every ray: T == 0 exactly where a surface lies in the interval
        blocked = occ.bool()
        mismatches = int(((T == 0) != blocked).sum().item())
        open_T = T[~blocked]
        # oracle parity on a sample
        m = min(args.oracle_rays, n)
        sample = np.ascontiguousarray(rays[:m].cpu().numpy()).view(rt.rt_ray_dtype).reshape(m)
        want = TransmittanceOracle(hs).transmittance(sample, t_max=t_max[:m].cpu().numpy())
        got = T[:m].cpu().numpy()
        zero_mismatch = int(((got == 0) != (want == 0)).sum())
        nz = (want != 0) & ~np.isnan(want)
        rel = float(np.max(np.abs(got[nz] - want[nz]) / want[nz])) if nz.any() else 0.0
        line = {"metric": "transmittance_mrays_per_sec", "value": n / ms_tr / 1e3, "unit": "Mrays/s", "n_gpus": 1, "dtype": "f64",
                "config": {"workload": f"{name} rays={n}", "rays": ray_set, "t_max": "per ray", "n_media": info.n_media,
                           "bvh_nodes": info.n_nodes, "node_bytes": info.node_bytes, "scene_create_s": t_build},
                "gpu": gpu, "ms": ms_tr,
                "nodes_per_ray": c_tr.node_visits / n, "prims_per_ray": c_tr.prim_tests / n,
                "occluded_fraction": float(blocked.float().mean().item()),
                "mean_T_unoccluded": float(open_T.mean().item()) if open_T.numel() else None,
                "occluded": {"value": n / ms_occ / 1e3, "unit": "Mrays/s", "ms": ms_occ,
                             "nodes_per_ray": c_occ.node_visits / n, "prims_per_ray": c_occ.prim_tests / n},
                "time_ratio_vs_occluded": ms_tr / ms_occ,
                "device_parity": {"rays": n, "mismatches": mismatches},
                "oracle_parity": {"rays": m, "max_rel_err": rel, "zero_pattern_mismatches": zero_mismatch}}
        print(json.dumps(line), flush=True)
        sc.close()
        del sc, rays, t_max, T, occ, blocked, open_T


if __name__ == "__main__":
    main()
