import sys, time
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from rs_ray_toy_b200 import capi, synth
from rs_ray_toy_b200.aggregate import Context, soup_aggregate
ctx = Context(0)
p, idx = synth.soup_triangles(1 << 22, 0.006, synth.SEED_C5_SOUP)
for flags in (capi.RRT_BUILD_DEVICE_LBVH, capi.RRT_BUILD_DEVICE_LBVH, capi.RRT_BUILD_FAST):
    t0 = time.perf_counter()
    agg = soup_aggregate(ctx, p, idx, 4, flags)
    print("commit total (incl. add_mesh)", flags, round(time.perf_counter() - t0, 3), agg.stats()["build_usec"], flush=True)
    del agg
