#!/usr/bin/env python
"""bench.py — BASELINE.json's headline metric on its config: Mrays/s incoherent closest-hit,
synthetic 1M-triangle random-soup mesh, 16M-ray batch of diffuse bounce rays (config 3).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pass of the closest-hit path over one 16,777,216-ray batch; the any-hit, host-buffer and
path-traced legs time K passes (frames) of their own as well.
  value  : rays already resident in HBM, K launches timed with CUDA events on the launching
           stream (rrt_intersect_device), max over ranks.
  e2e    : the same batch through the host-buffer C-ABI call a Rust `impl Primitive` binds
           (rrt_intersect): pinned host rays -> H2D -> kernel -> D2H hits inside the timed region.
  N > 1  : the path shards by rays/pixels with no exchange; every rank holds the scene and traces
           its own 16M-ray batch (weak scaling, no data-path collective).
`--impl reference` times the CPU restatement of the reference's own BVH path (oracle/, all host
threads) on bounded samples of the same workload — the Rust reference cannot be built here.
`--dump-outputs DIR` writes, on rank 0, what the last timed step of each leg returned, as DIR/<name>.npy:
a fixed, seeded sample of the rays (hits: prim_id with -1 for a miss, t, u, v; any-hit: occluded) and of
the pixels of each path-traced frame (RGB).  The inputs are seeded, so two builds can be compared array
for array (the films to rounding: they are summed with f64 atomics).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

N_TRIS = 1 << 20
N_RAYS = 1 << 24
METRIC = "Mrays/s incoherent closest-hit"
UNIT = "Mrays/s"
# Algorithmic bytes per ray (SURVEY.md §8d / DESIGN.md §5): fp32 record sizes ray 32 B + hit 16 B
# + 32 B per node visited + 36 B per triangle tested, with the mean node / triangle counts measured
# by the oracle on the Tier-F HLBVH (max_prims_in_node 4, near-first order, true closest-hit
# culling) on this exact workload — a property of the workload, not of the GPU kernel.
NV_C3 = 122.98
NT_C3 = 20.02
BYTES_PER_RAY = 32 + 16 + 32 * NV_C3 + 36 * NT_C3
# --dump-outputs: rays and pixels kept per array (38 MiB of .npy files in all)
DUMP_RAYS = 1 << 19
DUMP_PIXELS = 1 << 18
DUMP_SEED = 20261020
DUMP_LIMIT_BYTES = 64 << 20


def sample_rows(n, k):
    """The same min(n, k) row indices of an n-row output on every run, increasing."""
    if n <= k:
        return np.arange(n)
    return np.sort(np.random.default_rng(DUMP_SEED).choice(n, k, replace=False))


def write_dump(directory, arrays):
    out = Path(directory)
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"bench.py: --dump-outputs would write {total} bytes (limit {DUMP_LIMIT_BYTES})")
    out.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(out / f"{name}.npy", a)


def workload_config(n_gpus, n_rays=N_RAYS):
    return {
        "workload": "config 3: synthetic 1M-triangle random-soup mesh (v0~U[0,1]^3, edges U[-0.01,0.01]^3, seed 3), "
                    "16,777,216 incoherent cosine-weighted bounce rays per batch (seed 4+rank), t_max=inf, closest hit",
        "n_triangles": N_TRIS,
        "rays_per_step_per_gpu": n_rays,
        "max_prims_in_node": 4,
        "tier": "F (true closest hit, ties -> lowest prim id)",
        "l2_policy": "inputs larger than L2: 1 GiB of rays + 0.5 GiB of hits stream per step (126 MB L2)",
        "parallelism": f"ray-sharded x{n_gpus}, scene replicated, no data-path collective",
    }


class ClockSampler:
    """Samples SM clock + throttle reasons through NVML while the timed region runs."""

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4),
            "hw_power_brake": getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80),
        }
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(0.05)

    def __enter__(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thr:
            self._thr.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml_unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def measured_peak():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        try:
            return float(json.loads(f.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic():
    """dram bytes per launch of the dominant kernel from the committed ncu summary, or None."""
    f = ROOT / "profiles" / "traffic.json"
    if f.exists():
        try:
            return float(json.loads(f.read_text())["closest_hit_dram_bytes_per_launch_16M"])
        except Exception:
            return None
    return None


def cpu_oracle_rate(p, idx, rays_sample, threads=None):
    """Times the CPU restatement (oracle, Tier F) on `rays_sample`; returns (Mrays/s, threads, stats)."""
    sys.path.insert(0, str(ROOT / "tests"))
    import oracle_lib as O
    threads = threads or O.hardware_threads()
    scene = O.soup_scene(p, idx, O.TIER_F, 4)
    scene.intersect(rays_sample[: min(len(rays_sample), 1 << 16)], nthreads=threads)  # warm
    t0 = time.perf_counter()
    r = scene.intersect(rays_sample, nthreads=threads)
    dt = time.perf_counter() - t0
    return len(rays_sample) / dt / 1e6, threads, r["stats"], scene


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU algorithm (restated in oracle/, see its header)
    with every host thread, on bounded samples of config 3.  Rank 0 only."""
    if rank != 0:
        return
    sys.path.insert(0, str(ROOT / "tests"))
    import oracle_lib as O
    from rs_ray_toy_b200 import synth
    threads = O.hardware_threads()
    p, idx = synth.soup_triangles(N_TRIS)
    scene = O.soup_scene(p, idx, O.TIER_F, 4)
    probe = synth.bounce_rays(p, idx, 1 << 17, seed=synth.SEED_C3_RAYS)
    t0 = time.perf_counter()
    scene.intersect(probe, nthreads=threads)
    rate = len(probe) / (time.perf_counter() - t0)
    steps_total = args.steps + args.warmup
    per_step = int(min(N_RAYS, max(1 << 16, rate * 120.0 / max(1, steps_total))))  # whole run ~2 min
    rays = synth.bounce_rays(p, idx, per_step, seed=synth.SEED_C3_RAYS)
    for _ in range(args.warmup):
        scene.intersect(rays, nthreads=threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        scene.intersect(rays, nthreads=threads)
    dt = time.perf_counter() - t0
    value = per_step * args.steps / dt / 1e6
    sample = f"{per_step} rays per step of the 16,777,216-ray batch (same generator and seed), full 1M-triangle scene"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "CPU restatement (C++ f64, oracle/) of bvh.rs HLBVH + traversal with Q1/Q2/Q3 fixed; the Rust "
                "reference needs a nightly toolchain and un-vendored crates and cannot be built in this image",
    }
    print(json.dumps(line), flush=True)


PT_CONFIGS = {
    "c4": "config 4: 100,000 spheres r=0.5 (16 sphere entries: 8 Plastic rough 0.05-0.5, 8 Metal copper rough 0.01-0.3, "
          "x 6,250 instances, centres U[-50,50]^3 seed 5), 1 distant + 1 point light, Path max_depth 5 rr_threshold 1, "
          "Halton nsamp 65 (64 rendered, Q10), 1920x1080, box filter 0.5, double-Gauss lens camera",
    "c5": "config 5: 4,194,304-triangle random soup (edge 0.006, seed 6; half Matte, half Plastic), 1 point + 1 distant "
          "light, Path max_depth 5, Halton nsamp 257 (256 rendered), 3840x2160, box filter 0.5, double-Gauss lens camera",
}


def path_traced(args, ctx, rank, world, local_rank, barrier, config, dump):
    """Second half of BASELINE.json's metric: one path-traced frame, its 16x16 sample tiles dealt
    t % world == rank over the ranks (scene replicated), films summed onto rank 0 over NCCL.
    Strong scaling: the frame is fixed, value = camera samples of the whole frame / max-over-ranks time.
    A sample of the last timed frame's pixels goes into `dump` unless it is None."""
    import tempfile
    import torch
    import torch.distributed as dist
    from rs_ray_toy_b200 import parallel, synth
    from rs_ray_toy_b200.render import Render
    t_setup = time.perf_counter()
    if config == "c4":
        d = tempfile.mkdtemp(prefix=f"rrt_c4_{rank}_")
        path = synth.scene_c4(d)
        r = Render.load(ctx, path, seed=1)
        keep = None
    else:
        keep, r = synth.scene_c5_api(ctx, commit=(lambda a: parallel.commit_replicated(a, 4)) if world > 1 else None)
    setup_s = time.perf_counter() - t_setup
    frames = args.steps

    def frame():
        r.clear()
        r.run(tile_mod=world, tile_rank=rank)
        if world > 1:
            parallel.gather_film(r, world, rank, dst=0)

    # one untimed warm-up frame (config 5: 2.1 G camera samples, about 3 s on one B200); its wall time is reported beside the
    # timed one (`warmup_frame_ms`: the first frame of a renderer also sizes the traversal kernels' sort workspace)
    t_w = time.perf_counter()
    frame()
    warm_s = time.perf_counter() - t_w
    launches0 = ctx.launch_count
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(frames):
        frame()
    e1.record()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0   # rrt_render_run returns when the device finished: host clock = device time
    t = torch.tensor([dt], dtype=torch.float64, device="cuda")
    st = r.stats()
    counts = torch.tensor([st["samples"], st["camera_rays"], st["extension_rays"], st["shadow_rays"], st["bounces"]],
                          dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(counts, op=dist.ReduceOp.SUM)
    dt = float(t.item())
    samples, cam, ext, sh, bnc = [float(x) for x in counts.tolist()]
    out = None
    if rank == 0:
        img = r.film()
        if dump is not None:
            pix = sample_rows(img.shape[0] * img.shape[1], DUMP_PIXELS)
            dump[f"path_{config}_pixel_index"] = pix.astype(np.float64)
            dump[f"path_{config}_rgb"] = img.reshape(-1, 3)[pix]
        out = {
            "metric": "Msamples/s path-traced", "unit": "Msamples/s", "value": samples / (dt / frames) / 1e6,
            "ms_per_frame": dt / frames * 1e3, "frames": frames, "warmup_frame_ms": warm_s * 1e3, "n_gpus": world, "scaling": "strong",
            "config": {"workload": PT_CONFIGS[config], "parallelism": f"16x16 sample tiles dealt t % {world} == rank, "
                       "scene replicated (one rank builds the tree, the others receive it), one NCCL gather of the ranks' own tiles per frame"},
            "samples_per_frame": samples, "camera_rays": cam, "extension_rays": ext, "shadow_rays": sh,
            "rays_per_sample": (ext + sh) / max(samples, 1.0), "mean_bounces": bnc / max(cam, 1.0),
            "Mrays_per_s": (ext + sh) / (dt / frames) / 1e6, "setup_s": setup_s,
            "gpu_launches": int(ctx.launch_count - launches0),
            "image_mean_rgb": [float(x) for x in img.mean(axis=(0, 1))],
            "dtype": "f64 shading and film, fp32 box culling",
        }
        # ---- end to end: the call a consumer makes — rrt_render_clear + rrt_render_run + rrt_render_read_film into host
        # memory (scene and lens resident; down: the 4-f64-per-pixel film, converted to RGB on the host).  N = 1 only:
        # with more ranks the frame above already ends in the NCCL film reduce.
        if world == 1 and not args.no_e2e:
            t0 = time.perf_counter()
            r.clear()
            r.run()
            img_e2e = r.film()
            e2e_s = time.perf_counter() - t0
            out["e2e"] = {"value": samples / e2e_s / 1e6, "unit": "Msamples/s", "h2d_bytes_per_step": int(((img.shape[1] + 15) // 16) * ((img.shape[0] + 15) // 16) * 4),   # the tile list
                          "d2h_bytes_per_step": int(img.shape[0] * img.shape[1] * 4 * 8),
                          "api": "rrt_render_clear + rrt_render_run + rrt_render_read_film (host RGB film)",
                          # the film is summed with f64 atomics, whose order differs from run to run: equal to rounding
                          "same_image": bool(np.allclose(img_e2e, img, rtol=1e-9, atol=1e-12)),
                          "max_rel_difference": float(np.max(np.abs(img_e2e - img) / np.maximum(np.abs(img), 1e-12)))}
        if world == 1 and not args.no_cpu_baseline:
            sys.path.insert(0, str(ROOT / "tests"))
            import oracle_lib as O
            if config == "c4":
                import oracle_scene as S
                crop = (880, 460, 1040, 620)   # centred 160x160 pixels, full spp
                ls = S.load(path)
                t0 = time.perf_counter()
                ref = ls.render(seed=1, crop=crop)
                cdt = time.perf_counter() - t0   # includes the camera's exit-pupil set-up (a few seconds)
                prim_bytes = 16   # sphere: centre + radius (SURVEY.md §8d)
                what = "centred 160x160-pixel crop of the frame at full spp"
            else:
                import scenes
                crop = (1888, 1048, 1952, 1112)   # centred 64x64 pixels, full spp (256): 1 Mi camera samples
                t0 = time.perf_counter()
                ref = scenes.oracle_c5(1 << 22, 0.006, 3840, 2160, 257, crop=crop)
                cdt = time.perf_counter() - t0   # includes the oracle's HLBVH build over 4 Mi triangles and the exit-pupil set-up
                prim_bytes = 36   # triangle: 9 x fp32
                what = "centred 64x64-pixel crop of the frame at full spp"
            rs = ref["stats"]
            n_s = rs["camera_rays"] + rs["zero_weight"]
            gpu_crop = img[crop[1]:crop[3], crop[0]:crop[2]]
            ref_crop = ref["rgb"][crop[1]:crop[3], crop[0]:crop[2]]
            rmse = float(np.sqrt(np.mean((gpu_crop - ref_crop) ** 2)) / max(np.sqrt(np.mean(ref_crop ** 2)), 1e-300))
            nv = (rs["closest_nodes"] + rs["any_nodes"]) / max(n_s, 1)
            nt = (rs["closest_prims"] + rs["any_prims"]) / max(n_s, 1)
            rays_ps = (rs["extension_rays"] + rs["shadow_rays"]) / max(n_s, 1)
            bbar = rs["bounces"] / max(n_s, 1)
            # SURVEY.md §8d: sum over a sample's rays of (32 + 16|1 + 32 Nv + S_prim Nt) + film 16 + 2*96*B
            bytes_ps = (32 + 16) * rs["extension_rays"] / max(n_s, 1) + (32 + 1) * rs["shadow_rays"] / max(n_s, 1) + \
                32 * nv + prim_bytes * nt + 16 + 2 * 96 * bbar
            peak, peak_src = measured_peak()
            out["cpu_baseline"] = {"value": n_s / cdt / 1e6, "unit": "Msamples/s", "cores": O.hardware_threads(), "kind": "port",
                                   "sample": f"{what} ({n_s} camera samples), oracle Tier F, one thread per tile; the time "
                                             "includes the oracle's tree build and the camera's exit-pupil set-up",
                                   "seconds": cdt, "crop_rel_rmse_gpu_vs_oracle": rmse}
            out["roofline"] = {"bound": "hbm", "unit": "GB/s", "algorithmic_bytes_per_sample": bytes_ps,
                               "nodes_visited_per_sample_oracle": nv, "prims_tested_per_sample_oracle": nt,
                               "rays_per_sample_oracle": rays_ps, "bounces_per_sample_oracle": bbar,
                               "achieved": out["value"] * 1e6 * bytes_ps / 1e9, "peak": peak, "peak_source": peak_src,
                               "frac": out["value"] * 1e6 * bytes_ps / 1e9 / peak, "traffic": None}
    r.close()
    del keep
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--rays", type=int, default=N_RAYS, help=argparse.SUPPRESS)
    ap.add_argument("--path-config", default="both", choices=["both", "c4", "c5", "none"],
                    help="second half of the metric: path-traced Msamples/s on config 4 (1080p, 64 spp) and config 5 "
                         "(4K, 256 spp, the multi-GPU configuration)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write a fixed sample of what the last timed step of each leg computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs: use it with --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    dump = {} if args.dump_outputs and rank == 0 else None
    if args.impl == "reference":
        run_reference(args, rank, world)
        return 0
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    from rs_ray_toy_b200 import synth
    from rs_ray_toy_b200.aggregate import HIT_DTYPE, RAY_DTYPE, Context, pack_rays, soup_aggregate

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — this framework has no CPU path")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    n_rays = args.rays

    ctx = Context(local_rank)
    p, idx = synth.soup_triangles(N_TRIS)
    agg = soup_aggregate(ctx, p, idx, 4)
    stats = agg.stats()
    rays_np = synth.bounce_rays(p, idx, n_rays, seed=synth.SEED_C3_RAYS + rank)
    h_rays = ctx.pinned_empty(n_rays, RAY_DTYPE)
    h_rays[:] = pack_rays(rays_np)
    h_hits = ctx.pinned_empty(n_rays, HIT_DTYPE)
    del rays_np

    d_rays = torch.empty(n_rays * 8, dtype=torch.float64, device="cuda")
    d_hits = torch.empty(n_rays * 4, dtype=torch.float64, device="cuda")
    d_rays.copy_(torch.from_numpy(h_rays.view(np.float64)), non_blocking=False)
    stream = torch.cuda.current_stream()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_device():
        agg.intersect_device(n_rays, d_rays.data_ptr(), d_hits.data_ptr(), stream.cuda_stream)

    # ---- device-resident timing: K launches, CUDA events on the launching stream ----
    for _ in range(args.warmup):
        step_device()
    barrier()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    launches0 = ctx.launch_count
    with ClockSampler(local_rank) as clocks:
        ev[0].record(stream)
        for i in range(args.steps):
            step_device()
            ev[i + 1].record(stream)
        barrier()
    launches = ctx.launch_count - launches0
    per_launch_ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(args.steps)]
    total_ms = ev[0].elapsed_time(ev[-1])
    t = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms_max = float(t.item())
    value = n_rays * world * args.steps / (total_ms_max * 1e-3) / 1e6
    n_hit = int((d_hits.view(torch.int64)[0::4] & 0xFFFFFFFF != 0xFFFFFFFF).sum().item())
    if dump is not None:
        rows = sample_rows(n_rays, DUMP_RAYS)
        d_rows = torch.from_numpy(rows).cuda()
        h = d_hits.view(n_rays, 4)[d_rows].cpu().numpy().view(HIT_DTYPE).reshape(-1)
        dump["ray_index"] = rows.astype(np.float64)
        dump["closest_hit_prim_id"] = np.where(h["prim_id"] == 0xFFFFFFFF, -1.0, h["prim_id"].astype(np.float64))
        for f in ("t", "u", "v"):
            dump[f"closest_hit_{f}"] = np.ascontiguousarray(h[f])

    # ---- the other half of a1/a2: any-hit (BVHAccel::intersect_p) on the same batch, device resident ----
    d_occ = torch.empty(n_rays, dtype=torch.uint8, device="cuda")
    for _ in range(args.warmup):
        agg.intersect_p_device(n_rays, d_rays.data_ptr(), d_occ.data_ptr(), stream.cuda_stream)
    barrier()
    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a0.record(stream)
    for _ in range(args.steps):
        agg.intersect_p_device(n_rays, d_rays.data_ptr(), d_occ.data_ptr(), stream.cuda_stream)
    a1.record(stream)
    barrier()
    t = torch.tensor([a0.elapsed_time(a1)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    any_value = n_rays * world * args.steps / (float(t.item()) * 1e-3) / 1e6
    n_occ = int(d_occ.sum(dtype=torch.int64).item())
    if n_occ != n_hit:
        raise SystemExit(f"bench.py: any-hit and closest-hit disagree on which rays hit ({n_occ} vs {n_hit})")
    if dump is not None:
        dump["any_hit_occluded"] = d_occ[d_rows].float().cpu().numpy()
    del d_occ

    # ---- end to end: host buffers through rrt_intersect (H2D + kernel + D2H per step) ----
    for _ in range(2):
        agg.intersect(h_rays, out=h_hits)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        agg.intersect(h_rays, out=h_hits)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = n_rays * world * args.steps / float(t.item()) / 1e6
    e2e_hit = int((h_hits["prim_id"] != 0xFFFFFFFF).sum())
    if e2e_hit != n_hit:
        raise SystemExit(f"bench.py: host path and device path disagree ({e2e_hit} vs {n_hit} hits)")

    # free the ray batch before the frame renders
    del d_rays, d_hits
    torch.cuda.empty_cache()
    del agg
    pt = pt5 = None
    if args.path_config in ("both", "c4"):
        pt = path_traced(args, ctx, rank, world, local_rank, barrier, "c4", dump)
    if args.path_config in ("both", "c5"):
        pt5 = path_traced(args, ctx, rank, world, local_rank, barrier, "c5", dump)
    if dump is not None:
        write_dump(args.dump_outputs, dump)

    if rank == 0:
        peak, peak_src = measured_peak()
        kernel_ms = float(np.mean(per_launch_ms))
        achieved = n_rays * BYTES_PER_RAY / (kernel_ms * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64 deciding arithmetic (Moller-Trumbore / quadratic), fp32 box culling", "data": "synthetic",
            "config": workload_config(world, n_rays),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": n_rays * 64, "d2h_bytes_per_step": n_rays * 32,
                    "api": "rrt_intersect (pinned host rays -> hits), chunks of 128 Ki .. 1 Mi rays (tapered at both ends of the batch) on 4 streams"},
            "launches_per_step": launches / args.steps,
            "gpu_launches": int(launches),
            "clocks": clocks.summary(),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": ncu_traffic(), "peak_source": peak_src, "kernel": "trace_kernel<closest> (+4 ray-sort launches per step, inside the timed region)",
                         "kernel_ms": kernel_ms, "algorithmic_bytes_per_ray": BYTES_PER_RAY,
                         "nodes_visited_per_ray_oracle": NV_C3, "prims_tested_per_ray_oracle": NT_C3,
                         "compulsory_dram_bytes_per_ray": 64 + 32 + stats["device_bytes"] / n_rays},
            "hit_fraction": n_hit / n_rays,
            "any_hit": {"metric": "Mrays/s incoherent any-hit (intersect_p)", "value": any_value, "unit": UNIT,
                        "note": "same batch and scene through rrt_intersect_p_device, t_max = inf; occluded count equals the closest-hit count"},
            "scene": stats,
        }
        line["path_traced"] = pt
        line["path_traced_4k"] = pt5
        if not args.no_cpu_baseline and world == 1:
            n_sample = 1 << 22
            sample = synth.bounce_rays(p, idx, n_sample, seed=synth.SEED_C3_RAYS)
            rate, threads, st, _ = cpu_oracle_rate(p, idx, sample)
            # size-check: ~10-30 s of CPU work; one more pass if the first was very short
            line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
                                    "sample": f"first {n_sample} rays of the batch generator (seed 4), full 1M-triangle scene, "
                                              "oracle Tier F (C++ f64 restatement, std::thread x cores)",
                                    "nodes_visited_per_ray": float(st[1]) / float(st[0]),
                                    "prims_tested_per_ray": float(st[2]) / float(st[0])}
        else:
            line["cpu_baseline"] = None
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
