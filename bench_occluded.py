#!/usr/bin/env python
"""bench_occluded.py — the occlusion (any-hit) query against closest hit on the config-5 soups (SURVEY.md §8d): N random
triangles / spheres in the unit cube, 2^24 rays per batch, three ray sets:

  primary     rays from a pinhole at (0.5, 0.5, -2), scalar t_max = inf       (bench_closest_hit.make_rays)
  incoherent  origins uniform in the cube, directions uniform on the sphere, scalar t_max = inf
  shadow      segments between two uniform points a, b of the cube: unit direction, per-ray t_max_i = |b - a| (1 - 1e-6)

One JSON line per (shape, N, ray set) with the occlusion and the closest-hit rate on the same batch in the same process.  For
`shadow` closest hit runs with t_max = inf, which is what a caller without rt_occluded has to do, and compares t on its own.

    python bench_occluded.py [--sizes 1000000 10000000] [--shapes tri_soup sphere_soup] [--rays 16777216]

Rays live in HBM (torch tensors); timing is CUDA events around each _device call (stats.ms_total), best of 5 after 2 warm-ups,
the two queries alternating.  Node and primitive counts per ray come from the RT_OPT_COUNT instantiation of each kernel.  The
parity flag covers the whole batch: the occlusion bytes against (prim_id != RT_NONE and t <= t_max_i) of the closest-hit
output, compared on the device.  The card's name, power limit and maximum SM clock are read in the same run.
"""
import argparse
import json
import subprocess
import time

from bench_closest_hit import make_rays, rt


def gpu_description(torch, device):
    """Name, power limit and maximum SM clock of the card, read-only."""
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(device), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
        name, power, clock = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": power, "clocks_max_sm": clock}
    except Exception:
        return {"name": torch.cuda.get_device_name(device), "power_limit": None, "clocks_max_sm": None}


def shadow_rays(torch, n, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    a = torch.rand((n, 3), generator=g, device="cuda", dtype=torch.float64)
    b = torch.rand((n, 3), generator=g, device="cuda", dtype=torch.float64)
    length = (b - a).norm(dim=1)
    rays = torch.zeros((n, 7), dtype=torch.float64, device="cuda")
    rays[:, 0:3] = a
    rays[:, 3:6] = (b - a) / length[:, None]
    rays[:, 6] = torch.rand(n, generator=g, device="cuda", dtype=torch.float64)
    return rays, length * (1.0 - 1e-6)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[1_000_000, 10_000_000])
    ap.add_argument("--shapes", nargs="+", default=["tri_soup", "sphere_soup"])
    ap.add_argument("--rays", type=int, default=1 << 24)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: the product has no CPU path")
    gpu = gpu_description(torch, 0)
    stream = torch.cuda.current_stream().cuda_stream
    n = args.rays
    for shape in args.shapes:
        for size in args.sizes:
            t0 = time.perf_counter()
            sc = rt.Scene(rt.named_scene(shape, seed=5, params=[size]), device=0)
            t_build = time.perf_counter() - t0
            info = sc.info()
            for kind in ("primary", "incoherent", "shadow"):
                if kind == "shadow":
                    rays, t_max = shadow_rays(torch, n, 11)
                    t_max_ptr = t_max.data_ptr()
                else:
                    rays, t_max, t_max_ptr = make_rays(torch, n, kind, 11), None, None
                occ = torch.empty(n, dtype=torch.uint8, device="cuda")
                hits = torch.empty((n, 3), dtype=torch.float64, device="cuda")  # 24-byte rt_hit records
                run_occ = lambda flags=0: sc.occluded_device(rays.data_ptr(), n, occ.data_ptr(), t_max_ptr, flags=flags, stream=stream)
                run_ch = lambda flags=0: sc.closest_hit_device(rays.data_ptr(), n, hits.data_ptr(), flags=flags, stream=stream)
                ms_occ, ms_ch = float("inf"), float("inf")
                for k in range(7):  # alternating, best of 5 after 2 warm-ups
                    torch.cuda.synchronize()
                    a = run_occ().ms_total
                    b = run_ch().ms_total
                    if k >= 2:
                        ms_occ, ms_ch = min(ms_occ, a), min(ms_ch, b)
                c_occ, c_ch = run_occ(rt.RT_OPT_COUNT), run_ch(rt.RT_OPT_COUNT)
                # the equivalence rt2025.h states, on every ray of the batch
                prim_id = hits.view(torch.int32)[:, 2]
                want = (prim_id != -1) & (hits[:, 0] <= (t_max if t_max is not None else float("inf")))
                got = occ.bool()
                mismatches = int((got != want).sum().item())
                line = {"metric": "occluded_mrays_per_sec", "value": n / ms_occ / 1e3, "unit": "Mrays/s", "n_gpus": 1, "dtype": "f64",
                        "config": {"workload": f"{shape} N={size} rays={n} {kind}", "t_max": "per ray" if t_max is not None else "inf",
                                   "builder": "host binned SAH", "bvh_nodes": info.n_nodes, "node_bytes": info.node_bytes, "scene_create_s": t_build},
                        "gpu": gpu, "ms": ms_occ,
                        "nodes_per_ray": c_occ.node_visits / n, "prims_per_ray": c_occ.prim_tests / n,
                        "occluded_fraction": float(got.float().mean().item()),
                        "closest_hit": {"value": n / ms_ch / 1e3, "unit": "Mrays/s", "ms": ms_ch, "t_max": "inf",
                                        "nodes_per_ray": c_ch.node_visits / n, "prims_per_ray": c_ch.prim_tests / n},
                        "speedup_vs_closest_hit": ms_ch / ms_occ,
                        "parity": {"rays": n, "mismatches": mismatches, "bit_exact": mismatches == 0}}
                print(json.dumps(line), flush=True)
                del rays, t_max, occ, hits, got, want
            sc.close()
            del sc


if __name__ == "__main__":
    main()
