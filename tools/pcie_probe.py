"""What the host link gives (GPU box): pinned H2D alone, D2H alone, both at once — the ceiling of bench.py's `e2e`
(1 GiB of rays up + 0.5 GiB of hits down per 16 Mi-ray batch).  Not part of the product or the tests.
`measure()` returns the same numbers for other tools (tools/bench_rays_f32.py)."""
import torch


def measure(reps=5) -> dict:
    dev = torch.device("cuda:0")
    up_h = torch.empty(1 << 30, dtype=torch.uint8).pin_memory()
    dn_h = torch.empty(1 << 29, dtype=torch.uint8).pin_memory()
    up_d = torch.empty(1 << 30, dtype=torch.uint8, device=dev)
    dn_d = torch.empty(1 << 29, dtype=torch.uint8, device=dev)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()

    def timed(fn):
        best = 1e9
        for _ in range(reps):
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            s1.synchronize(); s2.synchronize()
            b.record()
            torch.cuda.synchronize()
            best = min(best, a.elapsed_time(b))
        return best

    def h2d():
        with torch.cuda.stream(s1):
            up_d.copy_(up_h, non_blocking=True)

    def d2h():
        with torch.cuda.stream(s2):
            dn_h.copy_(dn_d, non_blocking=True)

    def both():
        h2d(); d2h()

    def chunked(n=16):
        c, e = (1 << 30) // n, (1 << 29) // n
        for k in range(n):
            with torch.cuda.stream(s1 if k % 2 == 0 else s2):
                up_d[k * c:(k + 1) * c].copy_(up_h[k * c:(k + 1) * c], non_blocking=True)
                dn_h[k * e:(k + 1) * e].copy_(dn_d[k * e:(k + 1) * e], non_blocking=True)

    return {"h2d_1GiB_ms": timed(h2d), "d2h_0.5GiB_ms": timed(d2h), "both_ms": timed(both), "chunked_16_ms": timed(chunked)}


if __name__ == "__main__":
    r = measure()
    t = r["h2d_1GiB_ms"]; print(f"H2D 1 GiB alone: {t:.2f} ms = {1.0737 / t * 1e3:.1f} GB/s")
    t = r["d2h_0.5GiB_ms"]; print(f"D2H 0.5 GiB alone: {t:.2f} ms = {0.5369 / t * 1e3:.1f} GB/s")
    t = r["both_ms"]; print(f"both at once: {t:.2f} ms -> {16.777 / t * 1e3:.0f} Mrays/s ceiling for a 16 Mi-ray batch")
    t = r["chunked_16_ms"]; print(f"16 chunks on 2 streams: {t:.2f} ms -> {16.777 / t * 1e3:.0f} Mrays/s")
