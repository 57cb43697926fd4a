"""The surface records of the intersect API against the hits alone, on config 3 (1 Mi-triangle soup, 16 Mi bounce rays,
bench.py's generator): the device-resident entries (rrt_intersect_device, rrt_intersect_surface_device) timed with CUDA
events and the host entries (rrt_intersect, rrt_intersect_surface, pinned buffers) with a host clock around a
synchronised call, each pair alternated step by step in one process after a warm-up.  Adds the card's name and power
limit, the bytes each leg moves, and whether every record's hit equals the hit-only call's.  Writes one JSON line
(stdout, and --out).

--profile: a separate run that takes each kernel's own time with torch.profiler over a few device-entry calls.
Not part of the product or the tests."""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))


def gpu_identity() -> dict:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    name, power = (r.stdout.splitlines()[0].split(",") + ["?"])[:2] if r.returncode == 0 and r.stdout else ("?", "?")
    return {"name": name.strip(), "power_limit": power.strip()}


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--rays", type=int, default=1 << 24)
    ap.add_argument("--tris", type=int, default=1 << 20)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--profile", action="store_true", help="kernel times with torch.profiler instead of the timed legs")
    ap.add_argument("--no-host", action="store_true", help="device legs only")
    ap.add_argument("--out", type=Path)
    args = ap.parse_args()
    if args.steps < 10 and not args.profile:
        raise SystemExit("--steps must be at least 10")

    import torch

    from rs_ray_toy_b200 import synth
    from rs_ray_toy_b200.aggregate import HIT_DTYPE, RAY_DTYPE, SURFACE_DTYPE, Context, pack_rays, soup_aggregate

    if not torch.cuda.is_available():
        raise SystemExit("bench_surface.py: no CUDA device")
    n = args.rays
    ident = gpu_identity()
    ctx = Context(0)
    p, idx = synth.soup_triangles(args.tris)
    agg = soup_aggregate(ctx, p, idx, 4)
    h_rays = ctx.pinned_empty(n, RAY_DTYPE)
    h_rays[:] = pack_rays(synth.bounce_rays(p, idx, n, seed=synth.SEED_C3_RAYS))
    d_rays = torch.from_numpy(h_rays.view(np.float64)).cuda()
    d_hits = torch.empty(n * 4, dtype=torch.float64, device="cuda")
    d_surf = torch.empty(n * 42, dtype=torch.float64, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    dev = {
        "hit_device": lambda: agg.intersect_device(n, d_rays.data_ptr(), d_hits.data_ptr(), stream),
        "surface_device": lambda: agg.intersect_surface_device(n, d_rays.data_ptr(), d_surf.data_ptr(), stream),
    }
    for _ in range(args.warmup):
        for fn in dev.values():
            fn()
    torch.cuda.synchronize()

    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                for fn in dev.values():
                    fn()
            torch.cuda.synchronize()
        kernels = {}
        for e in prof.key_averages():
            if e.device_type.name == "CUDA" and e.count:
                t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
                kernels[e.key] = {"calls": e.count, "us_per_call": t / e.count}
        surf = [v["us_per_call"] for k, v in kernels.items() if "surface_kernel" in k]
        line = {"tool": "bench_surface", "mode": "profile", "gpu": ident, "rays": n, "triangles": args.tris,
                "kernels": kernels,
                "surface_kernel_ms": surf[0] / 1e3 if surf else None,
                "surface_kernel_bytes": n * (336 + 64 + 32),
                "surface_kernel_GBps": n * (336 + 64 + 32) / (surf[0] * 1e-6) / 1e9 if surf else None}
    else:
        times = {k: [] for k in dev}
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        for _ in range(args.steps):
            for k, fn in dev.items():
                ev[0].record()
                fn()
                ev[1].record()
                ev[1].synchronize()
                times[k].append(ev[0].elapsed_time(ev[1]) * 1e-3)
        hits = d_hits.cpu().numpy().view(np.uint64).reshape(n, 4)
        recs = d_surf.cpu().numpy().view(np.uint64).reshape(n, 42)
        identical = bool(np.array_equal(recs[:, :4], hits))
        if not args.no_host:
            h_hits = ctx.pinned_empty(n, HIT_DTYPE)
            h_surf = ctx.pinned_empty(n, SURFACE_DTYPE)
            host = {"hit_host": lambda: agg.intersect(h_rays, out=h_hits),
                    "surface_host": lambda: agg.intersect_surface(h_rays, out=h_surf)}
            for _ in range(args.warmup):
                for fn in host.values():
                    fn()
            for k in host:
                times[k] = []
            for _ in range(args.steps):
                for k, fn in host.items():
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    fn()
                    torch.cuda.synchronize()
                    times[k].append(time.perf_counter() - t0)
            identical = identical and bool(np.array_equal(np.frombuffer(h_hits, np.uint64).reshape(n, 4), hits)) and \
                bool(np.array_equal(np.frombuffer(h_surf, np.uint64).reshape(n, 42), recs))

        def rate(k):
            t = np.array(times[k])
            return {"Mrays_s_median": n / float(np.median(t)) / 1e6, "ms_min": float(t.min() * 1e3),
                    "ms_median": float(np.median(t) * 1e3), "ms_max": float(t.max() * 1e3)}

        res = {k: rate(k) for k in times}
        line = {
            "tool": "bench_surface", "mode": "timed", "gpu": ident, "rays": n, "triangles": args.tris, "steps": args.steps,
            "warmup": args.warmup,
            "timing": "device legs: CUDA events around each call; host legs: host clock around a synchronised call; "
                      "the two legs of each pair alternated per step",
            "legs": res,
            "bytes_per_step": {"hit_device": {"written": n * 32}, "surface_device": {"written": n * (32 + 336)},
                               "hit_host": {"h2d": n * 64, "d2h": n * 32}, "surface_host": {"h2d": n * 64, "d2h": n * 336}},
            "surface_device_extra_ms": res["surface_device"]["ms_median"] - res["hit_device"]["ms_median"],
            "hit_fraction": float(((recs[:, 0] & 0xFFFFFFFF) != 0xFFFFFFFF).mean()),
            "identical": identical,
        }
        if "surface_host" in res:
            line["surface_host_d2h_GBps"] = n * 336 / (res["surface_host"]["ms_median"] * 1e-3) / 1e9
    text = json.dumps(line)
    print(text)
    if args.out:
        args.out.parent.mkdir(parents=True, exist_ok=True)
        args.out.write_text(text + "\n")
    return 0 if line.get("identical", True) else 1


if __name__ == "__main__":
    sys.exit(main())
