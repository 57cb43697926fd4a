"""fp32 rays against f64 rays through the aggregate API on config 3 (1 Mi-triangle soup, 16 Mi bounce rays): the f64
host entry (rrt_intersect, bench.py's `e2e`), the fp32 host entry (rrt_intersect_f32), and both device-resident
entries (rrt_intersect_device, rrt_intersect_f32_device), timed step by step in alternation in one process, pinned
host buffers, after a warm-up.  Adds the card's name and power limit, the link's per-direction rate
(tools/pcie_probe.py) and whether every fp32 hit is the rounded f64 hit of the same run.  Writes one JSON line
(stdout, and --out).  Not part of the product or the tests.

RRT_HOST_TRACE=1 in the environment prints the host pipeline's per-chunk timeline on stderr (csrc/capi.cpp)."""
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
sys.path.insert(0, str(ROOT / "tools"))


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
    ap.add_argument("--no-link-probe", action="store_true")
    ap.add_argument("--out", type=Path)
    args = ap.parse_args()
    if args.steps < 10:
        raise SystemExit("--steps must be at least 10")

    import torch

    from rs_ray_toy_b200 import synth
    from rs_ray_toy_b200.aggregate import (HIT_DTYPE, HIT_F32_DTYPE, RAY_DTYPE, RAY_F32_DTYPE, Context, pack_rays_f32,
                                           promote_rays_f32, soup_aggregate)

    if not torch.cuda.is_available():
        raise SystemExit("bench_rays_f32.py: no CUDA device")
    n = args.rays
    ident = gpu_identity()
    link = None
    if not args.no_link_probe:
        import pcie_probe
        r = pcie_probe.measure()
        link = {"h2d_GBps": (1 << 30) / r["h2d_1GiB_ms"] / 1e6, "d2h_GBps": (1 << 29) / r["d2h_0.5GiB_ms"] / 1e6,
                "both_1GiB_up_0.5GiB_down_ms": r["both_ms"]}

    ctx = Context(0)
    p, idx = synth.soup_triangles(args.tris)
    agg = soup_aggregate(ctx, p, idx, 4)
    r32 = synth.bounce_rays(p, idx, n, seed=synth.SEED_C3_RAYS).astype(np.float32)
    h_r32 = ctx.pinned_empty(n, RAY_F32_DTYPE)
    pack_rays_f32(r32, out=h_r32)
    h_r64 = ctx.pinned_empty(n, RAY_DTYPE)
    h_r64[:] = promote_rays_f32(h_r32)        # the same rays, so the two answers can be compared
    del r32
    h_h32 = ctx.pinned_empty(n, HIT_F32_DTYPE)
    h_h64 = ctx.pinned_empty(n, HIT_DTYPE)
    d_r32 = torch.from_numpy(h_r32.view(np.float32)).cuda()
    d_r64 = torch.from_numpy(h_r64.view(np.float64)).cuda()
    d_h32 = torch.empty(n * 4, dtype=torch.float32, device="cuda")
    d_h64 = torch.empty(n * 4, dtype=torch.float64, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream

    legs = {
        "f64_host": lambda: agg.intersect(h_r64, out=h_h64),
        "f32_host": lambda: agg.intersect_f32(h_r32, out=h_h32),
        "f64_device": lambda: agg.intersect_device(n, d_r64.data_ptr(), d_h64.data_ptr(), stream),
        "f32_device": lambda: agg.intersect_f32_device(n, d_r32.data_ptr(), d_h32.data_ptr(), stream),
    }
    for _ in range(args.warmup):
        for fn in legs.values():
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in legs}
    for _ in range(args.steps):
        for k, fn in legs.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            times[k].append(time.perf_counter() - t0)

    want = h_h64.copy()
    same_host = bool(np.array_equal(h_h32["prim_id"], want["prim_id"]) and all(
        np.array_equal(h_h32[f].view(np.uint32), want[f].astype(np.float32).view(np.uint32)) for f in ("t", "u", "v")))
    dev32 = d_h32.cpu().numpy().view(HIT_F32_DTYPE).reshape(-1)
    dev64 = d_h64.cpu().numpy().view(HIT_DTYPE).reshape(-1)
    same_dev = bool(np.array_equal(dev32, h_h32) and np.array_equal(dev64, want))

    def rate(k):
        t = np.array(times[k])
        return {"Mrays_s_median": n / float(np.median(t)) / 1e6, "Mrays_s_mean": n * t.size / float(t.sum()) / 1e6,
                "ms_min": float(t.min() * 1e3), "ms_median": float(np.median(t) * 1e3), "ms_max": float(t.max() * 1e3)}

    res = {k: rate(k) for k in legs}
    line = {
        "tool": "bench_rays_f32", "gpu": ident, "rays": n, "triangles": args.tris, "steps": args.steps,
        "warmup": args.warmup, "timing": "host clock around each call, device synchronised before and after; legs alternated per step",
        "legs": res,
        "bytes_per_step": {"f64_host": {"h2d": n * 64, "d2h": n * 32}, "f32_host": {"h2d": n * 32, "d2h": n * 16},
                           "f64_device": {"h2d": 0, "d2h": 0}, "f32_device": {"h2d": 0, "d2h": 0}},
        "f32_host_over_f64_host": res["f32_host"]["Mrays_s_median"] / res["f64_host"]["Mrays_s_median"],
        "f32_device_over_f64_device": res["f32_device"]["Mrays_s_median"] / res["f64_device"]["Mrays_s_median"],
        "link_probe": link,
        "hit_fraction": float((h_h32["prim_id"] != 0xFFFFFFFF).mean()),
        "identical": same_host and same_dev,
    }
    text = json.dumps(line)
    print(text)
    if args.out:
        args.out.parent.mkdir(parents=True, exist_ok=True)
        args.out.write_text(text + "\n")
    return 0 if line["identical"] else 1


if __name__ == "__main__":
    sys.exit(main())
