"""Benchmark of rrt_scene_update_mesh (GPU box): wall time per update of the device entry, the host entry, a fresh
RRT_BUILD_DEVICE_LBVH commit and a fresh RRT_BUILD_FAST commit of the same geometry, on config 3's 1 Mi-triangle soup and
config 5's 4 Mi-triangle soup (every vertex displaced by a seeded float32 offset, so the records stay PrimRec48); where the
device entry's time goes (RRT_BUILD_TIMING laps); and closest-hit Mrays/s on config 3's 16 Mi bounce rays through the
updated scene's device-built tree against the SBVH tree of a fresh RRT_BUILD_FAST commit.  The variants alternate
round by round.  Writes one JSON document (--out)."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import numpy as np
import torch

from rs_ray_toy_b200 import capi, synth
from rs_ray_toy_b200.aggregate import Context, pack_rays, soup_aggregate


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def frames(p, k, seed):
    return [(p.astype(np.float32) + np.random.default_rng(seed + f).normal(0, 2e-3, p.shape).astype(np.float32))
            .astype(np.float64) for f in range(k)]


def laps_of(fn):
    """RRT_BUILD_TIMING lines the library writes to stderr during fn()."""
    os.environ["RRT_BUILD_TIMING"] = "1"
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+") as f:
        os.dup2(f.fileno(), 2)
        try:
            fn()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["RRT_BUILD_TIMING"]
        f.seek(0)
        return [line.rstrip() for line in f if line.startswith("RRT_BUILD_TIMING")]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r3_mesh_update_bench.json"))
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    ctx = Context(0)
    doc = {"gpu": card(), "rounds": args.rounds, "scenes": []}
    for name, n_tris, edge, seed in (("config 3", 1 << 20, 0.01, synth.SEED_C3_SOUP),
                                     ("config 5", 1 << 22, 0.006, synth.SEED_C5_SOUP)):
        p, idx = synth.soup_triangles(n_tris, edge, seed)
        fs = frames(p, args.rounds + 1, 1000)
        d_fs = [torch.from_numpy(f).cuda() for f in fs]
        dev = soup_aggregate(ctx, p, idx)
        host = soup_aggregate(ctx, p, idx)
        stream = torch.cuda.current_stream().cuda_stream
        torch.cuda.synchronize()
        # the first update of each scene makes the device image: timed on its own
        t0 = time.perf_counter()
        dev.update_mesh_device(0, 0, p.shape[0], d_fs[0].data_ptr(), stream=stream)
        first_dev = time.perf_counter() - t0
        t0 = time.perf_counter()
        host.update_mesh(0, fs[0])
        first_host = time.perf_counter() - t0
        times = {"device entry": [], "host entry": [], "fresh DEVICE_LBVH commit": [], "fresh FAST commit": []}
        for r in range(1, args.rounds + 1):
            t0 = time.perf_counter()
            dev.update_mesh_device(0, 0, p.shape[0], d_fs[r].data_ptr(), stream=stream)
            times["device entry"].append(time.perf_counter() - t0)
            t0 = time.perf_counter()
            host.update_mesh(0, fs[r])
            times["host entry"].append(time.perf_counter() - t0)
            for label, flags in (("fresh DEVICE_LBVH commit", capi.RRT_BUILD_DEVICE_LBVH), ("fresh FAST commit", capi.RRT_BUILD_FAST)):
                t0 = time.perf_counter()
                a = soup_aggregate(ctx, fs[r], idx, 4, flags)
                times[label].append(time.perf_counter() - t0)
                a.close()
        same = bool((dev.export_tree()[280:] == host.export_tree()[280:]).all())
        laps = laps_of(lambda: dev.update_mesh_device(0, 0, p.shape[0], d_fs[1].data_ptr(), stream=stream))
        entry = {"scene": name, "n_tris": n_tris,
                 "first_update_s": {"device entry": round(first_dev, 4), "host entry": round(first_host, 4)},
                 "update_s": {k: {"median": round(float(np.median(v)), 4), "min": round(min(v), 4), "max": round(max(v), 4)}
                              for k, v in times.items()},
                 "device_and_host_entry_same_tree_and_records": same,
                 "device_entry_laps": laps}
        if name == "config 3":
            n_rays = 1 << 24
            pf = fs[args.rounds]
            rays = pack_rays(synth.bounce_rays(pf, idx, n_rays, seed=synth.SEED_C3_RAYS))
            d_rays = torch.from_numpy(rays.view(np.float64)).cuda()
            d_hits = torch.empty(n_rays * 4, dtype=torch.float64, device="cuda")
            sbvh = soup_aggregate(ctx, pf, idx, 4, capi.RRT_BUILD_FAST)
            rates = {}
            for rep in range(2):                                   # alternate the two trees
                for label, agg in (("updated (device LBVH tree)", host), ("fresh FAST commit (SBVH tree)", sbvh)):
                    s = torch.cuda.current_stream()
                    for _ in range(2):
                        agg.intersect_device(n_rays, d_rays.data_ptr(), d_hits.data_ptr(), s.cuda_stream)
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(s)
                    for _ in range(5):
                        agg.intersect_device(n_rays, d_rays.data_ptr(), d_hits.data_ptr(), s.cuda_stream)
                    e1.record(s)
                    torch.cuda.synchronize()
                    rates.setdefault(label, []).append(round(n_rays * 5 / e0.elapsed_time(e1) / 1e3, 1))
            entry["closest_hit_Mrays_per_s_16Mi_bounce_rays"] = rates
            sbvh.close()
            del d_rays, d_hits
        print(json.dumps(entry), flush=True)
        doc["scenes"].append(entry)
        dev.close()
        host.close()
        del d_fs
        torch.cuda.empty_cache()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(doc, indent=1) + "\n")


if __name__ == "__main__":
    main()
