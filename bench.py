#!/usr/bin/env python
"""bench.py — paths/sec on the book-2 final scene (BASELINE.json configs[1]).

    python bench.py --gpus N --steps K --warmup W            # the CUDA core
    python bench.py --impl reference --gpus N --steps K ...  # CPU restatement of the reference

One "step" = one full render of the 800x800 frame at 1000 spp (961 effective, depth 40) =
615,040,000 paths.  With N > 1 (torchrun, one rank per GPU) the frame is cut into interleaved
8x8 pixel tiles, rank r renders tiles with tile_index % N == r, and one NCCL reduce(sum) of the
float framebuffer reassembles it on rank 0: total work is fixed, so scaling is "strong".

--dump-outputs DIR writes the image the last timed step computed to DIR/image.npy, (H, W, 3) after the timed region: the float
framebuffer (on rank 0 the reduced frame), the RgbImage bytes with --single-process, the oracle's partial frame with --impl reference.
Scene and render seeds are fixed, so two builds run with the same arguments can be compared image for image.

Keys beyond the base contract: `roofline` (dominant kernel = extend), `cpu_baseline` (the oracle on
this box's host cores, bounded sample), `e2e` (flatten + upload + render + read-back + 8-bit encode
per step, i.e. what Camera::render does), `clocks`, `gpu_launches`.
"""
import argparse
import ctypes
import importlib.util
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
# torchrun presets OMP_NUM_THREADS=1 for its workers.  The host side here is OpenMP (scene compile, and the CPU
# reference arm, which has to use every host thread and runs on rank 0 alone): size it before libgomp loads.
if int(os.environ.get("WORLD_SIZE", "1")) > 1:
    _cores = os.cpu_count() or 8
    os.environ["OMP_NUM_THREADS"] = str(_cores if "reference" in sys.argv else max(1, _cores // int(os.environ["WORLD_SIZE"])))
_spec = importlib.util.spec_from_file_location("rt2025", os.path.join(ROOT, "raytracer-2025_b200", "rt2025.py"))
rt = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(rt)

SCENE = ("book2_final", 7, [800, 1000, 40])  # name, scene seed, [width, spp, max_depth]
RENDER_SEED = 2025
# algorithmic HBM bytes of the dominant kernel (extend) per unit (= one path segment), DESIGN.md §5:
# ray stream record read (64, path ids included) + hit stream record read (16: the medium scatter point the sampling pass
# left as the incumbent; book2_final has media, so that pass runs first) + hit stream record written (16) + class byte (1)
EXTEND_BYTES_PER_SEGMENT = 64 + 16 + 16 + 1
# SURVEY.md §8(d), whole step: 2 x 64 (path state read + written once) + 2 x 16 (hit record written by extend, read by shade)
# per segment, + 12 per path for the framebuffer add
STEP_BYTES_PER_SEGMENT, STEP_BYTES_PER_PATH = 160, 12


def dump_outputs(out_dir, image):
    """--dump-outputs: the image the last timed step computed, as out_dir/image.npy (float32, or float64 when it was rendered so)."""
    import numpy as np
    image = np.asarray(image)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "image.npy"), image if image.dtype == np.float64 else image.astype(np.float32))


def partition_for_rank(rank, world):
    """rt_render_opts.part_index / part_count of a rank: interleaved 8x8 tiles, tile % world == rank."""
    return rank, max(1, world)


def reduce_framebuffer_and_paths(fb, paths, dst=0):
    """The single collective of the multi-GPU path: sum the float framebuffers on `dst` (partitions
    are disjoint, so the sum is also the gather) and total the path counts."""
    import torch
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.reduce(fb, dst=dst, op=dist.ReduceOp.SUM)
        t = torch.tensor([int(paths)], dtype=torch.int64, device=fb.device)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return int(t.item())
    return int(paths)


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons during the timed region (NVML, 100 ms period)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if not self.nv:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                get = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
                mask = get(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def cpu_baseline(host_scene, target_seconds=12.0):
    """The C++ restatement of the reference (oracle/) on this box's host cores, on a bounded sample:
    the same frame and camera, strata [0, k) of the 961."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import orc
    osc = orc.OracleScene(host_scene)
    cores = orc.lib().orc_num_threads()
    t0 = time.perf_counter()
    _, st = osc.render(seed=RENDER_SEED, sample_begin=0, sample_end=1)
    dt1 = time.perf_counter() - t0
    k = int(max(1, min(16, target_seconds / max(dt1, 1e-3))))
    t0 = time.perf_counter()
    _, st = osc.render(seed=RENDER_SEED, sample_begin=0, sample_end=k)
    dt = time.perf_counter() - t0
    return {"value": st.paths / dt, "unit": "paths/s", "cores": cores, "kind": "port",
            "sample": f"strata [0,{k}) of 961 over the full 800x800 frame: {st.paths} paths in {dt:.2f} s, "
                      f"{st.segments / st.paths:.2f} segments/path",
            "note": "C++ restatement of the reference algorithm (recursive, virtual dispatch, median BVH); "
                    "the Rust crate itself cannot be built here (no rustc/cargo)"}


def closest_hit_metric(torch, peak, sizes=(1_000_000, 10_000_000), n_rays=1 << 24):
    """The second BASELINE metric (config 5), on rank 0 at N=1: BVH closest-hit Mrays/s on the triangle and sphere soups,
    primary and incoherent rays, 2^24 rays resident in HBM, with an id / t parity check against the oracle on a strided
    sample of each batch (bench_closest_hit.py is the same sweep as a program of its own, with more sizes and N > 1)."""
    spec = importlib.util.spec_from_file_location("bench_closest_hit", os.path.join(ROOT, "bench_closest_hit.py"))
    bch = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bch)
    cases = []
    bch.sweep(torch, list(sizes), ["tri_soup", "sphere_soup"], n_rays, 100_000, 1_000_000, False, 1, 0, torch.cuda.current_device(), peak, cases.append)
    head = next(c for c in cases if c["config"]["workload"].startswith("tri_soup N=1000000") and c["config"]["workload"].endswith("incoherent"))
    return {"value": head["value"], "unit": "Mrays/s", "workload": head["config"]["workload"] + ", binary64 primitive tests",
            "note": "`frac` counts every node / primitive fetch as HBM bytes (SURVEY.md 8d, no cache credit); `dram_frac` is the ncu DRAM traffic of the same "
                    "workload over the measured time; parity = ids and t bit-exact against the oracle on a strided sample (sizes the oracle builds in seconds)",
            "cases": [{"workload": c["config"]["workload"], "mrays_per_s": c["value"], "ms": c["ms"], "nodes_per_ray": c["nodes_per_ray"],
                       "prims_per_ray": c["prims_per_ray"], "node_bytes": c["config"]["node_bytes"], "scene_create_s": c["config"]["scene_create_s"],
                       "roofline": c["roofline"], "parity": c.get("parity"), "cpu_baseline": c.get("cpu_baseline")} for c in cases]}


def run_reference(args, rank):
    """--impl reference: the oracle port timed on host cores; rank 0 only."""
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import orc
    name, seed, params = SCENE
    hs = rt.named_scene(name, seed=seed, params=params)
    osc = orc.OracleScene(hs)
    cores = orc.lib().orc_num_threads()
    strata = 2  # per step: 800*800*2 = 1.28 M paths
    for _ in range(args.warmup):
        osc.render(seed=RENDER_SEED, sample_begin=0, sample_end=strata)
    t0 = time.perf_counter()
    paths = 0
    for k in range(args.steps):
        img, st = osc.render(seed=RENDER_SEED, sample_begin=(k * strata) % 960, sample_end=(k * strata) % 960 + strata)
        paths += st.paths
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, img)
    v = paths / dt
    sample = f"{strata} strata of 961 per step over the full 800x800 frame ({paths // max(1, args.steps)} paths/step)"
    print(json.dumps({
        "impl": "reference", "metric": "paths_per_sec", "value": v, "unit": "paths/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / max(1, args.steps) * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "book2_final 800x800 spp=1000 (961 effective) depth=40", "sample": sample},
        "cpu_baseline": {"value": v, "unit": "paths/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "paths/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def run_single_process(args):
    """--single-process: ONE process, N GPUs, through the library's own multi-GPU entry (rt_render_multi_rgb8): one host thread
    per GPU inside the library, partial frames summed on GPU 0 by a kernel that reads the peers' memory over NVLink, 8-bit
    encode on GPU 0, the RgbImage bytes land in a host buffer.  `value`: scenes resident, wall clock around the call (it
    returns when the bytes are on the host); `e2e`: rt_scene_create on every GPU inside the timed region as well."""
    import numpy as np
    import torch
    n = args.gpus
    if torch.cuda.device_count() < n:
        raise SystemExit(f"bench.py --single-process: {n} GPUs requested, {torch.cuda.device_count()} visible")
    name, seed, params = SCENE
    params = [params[0], args.spp, params[2]]
    hs = rt.named_scene(name, seed=seed, params=params)
    cam = hs.camera
    W, H = cam.image_width, cam.image_height
    scenes = [rt.Scene(hs, device=k) for k in range(n)]
    for _ in range(args.warmup):
        rt.render_multi_rgb8(scenes, seed=RENDER_SEED)
    sampler = ClockSampler(0)
    sampler.start()
    for k in range(n):
        torch.cuda.synchronize(k)
    t0 = time.perf_counter()
    paths = launches = 0
    for _ in range(args.steps):
        img, st = rt.render_multi_rgb8(scenes, seed=RENDER_SEED)
        paths += st.paths
        launches += st.kernel_launches
    dt = time.perf_counter() - t0
    sampler.stop_flag = True
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, img)
    for sc in scenes:
        sc.close()
    t0 = time.perf_counter()
    e2e_paths = 0
    for _ in range(args.steps):
        sc2 = [rt.Scene(hs, device=k) for k in range(n)]
        img, st = rt.render_multi_rgb8(sc2, seed=RENDER_SEED)
        e2e_paths += st.paths
        for sc in sc2:
            sc.close()
    e2e_dt = time.perf_counter() - t0
    d = hs.desc.contents
    h2d = n * (d.n_objects * 72 + d.n_children * 4 + d.n_spheres * 64 + d.n_planars * 144 + d.n_transforms * 80 + d.n_media * 16 +
               d.n_materials * 176 + d.n_textures * 80 + d.n_perlins * 9216 + d.n_texels * 4)
    print(json.dumps({
        "metric": "paths_per_sec", "value": paths / dt, "unit": "paths/s", "n_gpus": n, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / max(1, args.steps) * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"book2_final {W}x{H} spp={args.spp} ({cam.sqrt_spp ** 2} effective) depth={cam.max_depth}", "scene_seed": seed,
                   "parallelism": f"single process, rt_render_multi_rgb8 over {n} GPUs (interleaved 8x8 tiles, peer-memory reduce on GPU 0)",
                   "timing": "host wall clock around the call: it returns when the RgbImage bytes are in the host buffer"},
        "clocks": sampler.summary(), "gpu_launches": int(launches),
        "e2e": {"value": e2e_paths / e2e_dt, "unit": "paths/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(W * H * 3),
                "includes": "rt_scene_create on every GPU + rt_render_multi_rgb8"},
        "image_mean_8bit": float(np.mean(img)),
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--spp", type=int, default=1000, help="samples_per_pixel field (default = the config's 1000)")
    ap.add_argument("--single-process", action="store_true",
                    help="one process drives --gpus N through rt_render_multi_rgb8 (the library's own multi-GPU path: peer-memory reduce on GPU 0) "
                         "instead of one torchrun rank per GPU with an NCCL reduce")
    ap.add_argument("--no-closest-hit", action="store_true", help="skip the config-5 closest-hit cases (N=1 only)")
    ap.add_argument("--partition", default="tiles", choices=["tiles", "strata"],
                    help="how N > 1 ranks share the frame: interleaved 8x8 pixel tiles (default) or contiguous stratum ranges of every pixel")
    ap.add_argument("--rank-times", action="store_true", help="print every rank's device time per step to stderr (load-balance diagnosis)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the image the last timed step computed to DIR/image.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if args.single_process:
        run_single_process(args)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU path (use --impl reference for the CPU port)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)

    name, seed, params = SCENE
    params = [params[0], args.spp, params[2]]
    hs = rt.named_scene(name, seed=seed, params=params)
    cam = hs.camera
    W, H = cam.image_width, cam.image_height
    scene = rt.Scene(hs, device=local_rank)
    info = scene.info()
    part_index, part_count = partition_for_rank(rank, world)
    spp_eff = cam.sqrt_spp ** 2
    part_kw = dict(part_index=part_index, part_count=part_count)
    if args.partition == "strata" and world > 1:  # every rank renders all pixels, strata [begin, end) of the sampling grid
        part_kw = dict(sample_begin=rank * spp_eff // world, sample_end=(rank + 1) * spp_eff // world)
    fb = torch.zeros((H, W, 3), dtype=torch.float32, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    stream = torch.cuda.current_stream().cuda_stream

    def step(flags=rt.RT_OPT_STAGE_TIMES):
        flush.zero_()
        st = scene.render_device(fb.data_ptr(), stream=stream, seed=RENDER_SEED, accum_type=rt.RT_ACCUM_F32, flags=flags, **part_kw)
        if args.rank_times:
            print(f"[rank {rank}] render {st.ms_total:.2f} ms, {st.paths} paths, {st.iterations} iterations", file=sys.stderr, flush=True)
        total = reduce_framebuffer_and_paths(fb, st.paths, dst=0)
        return st, total

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    paths = segs = walk_segs = launches = iters = 0
    ms_extend = ms_shade = ms_gen = ms_media = 0.0
    for _ in range(args.steps):
        st, total = step()
        paths += total
        segs += st.segments
        walk_segs += st.walk_segments  # evaluated in registers by k_walk: they never pass through k_extend
        launches += st.kernel_launches + 1  # + the L2 flush fill
        iters += st.iterations
        ms_extend += st.ms_extend
        ms_shade += st.ms_shade
        ms_gen += st.ms_raygen
        ms_media += st.ms_other
    e1.record()
    barrier()
    sampler.stop_flag = True
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, fb.cpu().numpy())
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    extra = torch.tensor([segs, launches], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(extra, op=dist.ReduceOp.SUM)
    ms_total = float(ms.item())
    value = paths / (ms_total * 1e-3)

    # ---- e2e: what Camera::render does per call: flatten/upload the scene, render, reduce, read the
    # frame back to the host, 8-bit encode.  Host buffers in, host image out.
    d = hs.desc.contents
    h2d = (d.n_objects * 72 + d.n_children * 4 + d.n_spheres * 64 + d.n_planars * 144 + d.n_transforms * 80 + d.n_media * 16 +
           d.n_materials * 176 + d.n_textures * 80 + d.n_perlins * 9216 + d.n_texels * 4)
    d2h = W * H * 3  # the RgbImage bytes
    host_rgb = torch.empty((H, W, 3), dtype=torch.uint8).pin_memory()
    rgb_dev = torch.empty((H, W, 3), dtype=torch.uint8, device=dev)
    barrier()
    t0 = time.perf_counter()
    e2e_paths = 0
    for _ in range(args.steps):
        sc2 = rt.Scene(hs, device=local_rank)  # rt_scene_create: compile + BVH build + H2D of the scene
        if world == 1:
            # the host-buffer entry a client of Camera::render calls: render, Color::to_rgb on the device, D2H of the bytes
            o = sc2.render_opts(seed=RENDER_SEED)
            st = rt.rt_stats()
            rc = sc2.L.rt_render_rgb8(sc2.h, ctypes.byref(cam), ctypes.byref(o), host_rgb.data_ptr(), ctypes.byref(st))
            assert rc == 0, sc2.L.rt_last_error()
            e2e_paths += st.paths
        else:
            st = sc2.render_device(fb.data_ptr(), stream=stream, seed=RENDER_SEED, accum_type=rt.RT_ACCUM_F32, **part_kw)
            e2e_paths += reduce_framebuffer_and_paths(fb, st.paths, dst=0)
            if rank == 0:
                # Color::to_rgb where the reduced frame lies, then the D2H of the 8-bit image
                rt.tonemap_device(fb.data_ptr(), W * H, rgb_dev.data_ptr(), cam.toon_map, rt.RT_ACCUM_F32, stream)
                host_rgb.copy_(rgb_dev, non_blocking=False)
        sc2.close()
    barrier()
    e2e_t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_value = e2e_paths / float(e2e_t.item())

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        n_ext_launches = max(1, iters)
        seg_rank0 = segs - walk_segs  # the segments k_extend processed on this rank
        ext_bytes_per_launch = seg_rank0 * EXTEND_BYTES_PER_SEGMENT / n_ext_launches
        ext_ms_per_launch = ms_extend / n_ext_launches
        achieved = ext_bytes_per_launch / (ext_ms_per_launch * 1e-3) / 1e9 if ext_ms_per_launch > 0 else 0.0
        traffic, ncu_issue = None, None
        try:
            prof = json.load(open(os.path.join(ROOT, "profiles", "extend_traffic.json")))
            traffic = prof.get("dram_bytes_per_launch")
            # the figures that describe an issue-bound kernel, from the same ncu capture (not measured live)
            ncu_issue = {"issue_active_pct": prof.get("issue_active_pct"), "active_lanes_per_instruction": prof.get("active_lanes_per_instruction"),
                         "warps_active_pct": prof.get("warps_active_pct"), "source": prof.get("source"), "captured_on_commit": prof.get("commit")}
        except Exception:
            pass
        line = {
            "metric": "paths_per_sec", "value": value, "unit": "paths/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / max(1, args.steps), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"book2_final {W}x{H} spp={args.spp} ({cam.sqrt_spp ** 2} effective) depth={cam.max_depth}",
                       "scene_seed": seed, "prims": info.n_prims, "bvh_nodes": info.n_nodes, "media": info.n_media,
                       "paths_per_step": paths // max(1, args.steps), "segments_per_path": float(extra[0].item()) / max(1, paths),
                       "parallelism": f"{args.partition}{world}" if world > 1 else "single",
                       "l2": "flushed between steps (256 MiB fill); the ray/throughput/hit streams of up to 2^27 paths in flight (249 B per path, 33 GB) exceed the 126 MB L2, the 0.7 MB scene is cache-resident by design"},
            "clocks": sampler.summary(),
            "e2e": {"value": e2e_value, "unit": "paths/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "includes": ("rt_scene_create (compile + SAH build + upload of the host description) then rt_render_rgb8 into a host buffer (render, 8-bit encode on the device, D2H)"
                                 if world == 1 else
                                 "per rank rt_scene_create + rt_render_device, one NCCL reduce, rt_tonemap_device + D2H of the RgbImage bytes on rank 0")},
            "gpu_launches": int(extra[1].item()),
            "roofline": {"bound": "hbm", "kernel": "k_extend", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "bytes_per_segment": EXTEND_BYTES_PER_SEGMENT, "segments_per_launch": seg_rank0 / n_ext_launches,
                         "walk_segment_share": walk_segs / max(1, segs),
                         "ms_per_launch": ext_ms_per_launch, "ncu": ncu_issue,
                         # the whole step by SURVEY.md 8(d)'s formula (all stages, loose by design for a cache-resident scene)
                         "step": {"bytes_per_segment": STEP_BYTES_PER_SEGMENT, "bytes_per_path": STEP_BYTES_PER_PATH,
                                  "achieved": (float(extra[0].item()) * STEP_BYTES_PER_SEGMENT + paths * STEP_BYTES_PER_PATH) / (ms_total * 1e-3) / 1e9 / world,
                                  "frac": (float(extra[0].item()) * STEP_BYTES_PER_SEGMENT + paths * STEP_BYTES_PER_PATH) / (ms_total * 1e-3) / 1e9 / world / peak,
                                  "unit": "GB/s per GPU"},
                         "stage_ms_per_step": {"generate": ms_gen / args.steps, "extend": ms_extend / args.steps,
                                               "media_bin": ms_media / args.steps, "shade": ms_shade / args.steps},
                         "note": "configs 1-3 keep the scene in L1/L2: the binding limit is SM issue rate under divergence, "
                                 "not HBM (SURVEY.md §8d); see profiles/ for issue utilisation"},
        }
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline(hs)
            if not args.no_closest_hit:
                try:
                    scene.close()
                    del fb, flush
                    torch.cuda.empty_cache()
                    line["closest_hit"] = closest_hit_metric(torch, peak)
                except Exception as e:  # the headline line must not depend on the secondary metric
                    line["closest_hit"] = {"error": repr(e)}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
