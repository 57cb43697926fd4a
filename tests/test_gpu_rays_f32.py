"""-m gpu: the fp32 entry points (rrt_intersect_f32 and relatives, include/rrt.h) against their definition.  An fp32
call answers bit for bit what the f64 call answers on the same rays promoted exactly to f64 (time = 0), with t, u and v
then rounded to nearest fp32; any-hit flags are the f64 call's byte for byte.  Both tiers, every shape kind, the host
pipeline's chunking, caller-owned device buffers on streams of their own, concurrent callers and the error codes."""
import ctypes as C
import threading

import numpy as np
import pytest

import golden_cases
import scenes
from rs_ray_toy_b200 import capi, synth
from rs_ray_toy_b200 import transform as T
from rs_ray_toy_b200.aggregate import (HIT_F32_DTYPE, GpuAggregate, pack_rays_f32, promote_rays_f32)

pytestmark = pytest.mark.gpu
CHUNK = 1 << 20  # rays per host pipeline slot (csrc/capi.cpp)


def _same_f32(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return bool(((a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))).all())


def _expect(agg, r32):
    """What the fp32 calls must answer: the f64 calls on the promoted rays, rounded."""
    r64 = promote_rays_f32(r32)
    return agg.intersect(r64), agg.intersect_p(r64)


def _assert_f32_answers(h32, h64):
    assert h32.dtype == HIT_F32_DTYPE and h32.shape == h64.shape
    assert np.array_equal(h32["prim_id"], h64["prim_id"])
    for f in ("t", "u", "v"):
        assert _same_f32(h32[f], h64[f].astype(np.float32)), f


def _check(agg, r32):
    h64, occ64 = _expect(agg, r32)
    h32 = agg.intersect_f32(r32)
    _assert_f32_answers(h32, h64)
    occ32 = agg.intersect_p_f32(r32)
    assert np.array_equal(occ32, occ64)
    return h32, occ32


def _partial_spheres_and_field(ctx):
    """Config 4's sphere field plus spheres clipped in z and phi, placed through scaled and rotated instances."""
    rng = np.random.default_rng(12)
    a = GpuAggregate(ctx)
    m, inv = scenes.sphere_instances(20000, extent=15.0)
    a.add_sphere(radius=0.5, instances=(m, inv))
    for k in range(24):
        radius = float(rng.uniform(0.5, 1.5))
        z_min, z_max = sorted((float(rng.uniform(-radius, 0.2 * radius)), float(rng.uniform(0.3 * radius, radius))))
        ms, invs = zip(*[T.make_to_world(rng.uniform(-12, 12, 3), rng.normal(0, 1, 3), float(rng.uniform(0, 360)),
                                         tuple(rng.uniform(0.6, 1.6, 3))) for _ in range(3)])
        a.add_sphere(radius=radius, z_min=z_min, z_max=z_max, phi_max=float(rng.uniform(60, 330)),
                     instances=(np.array(ms), np.array(invs)))
    return a.commit()


def test_config3_soup_at_a_million_rays(ctx):
    p, idx = scenes.soup(1 << 20)
    agg = scenes.gpu_soup(ctx, p, idx)
    rays = synth.bounce_rays(p, idx, (1 << 20) + 4321, seed=61).astype(np.float32)
    rays[::5, 6] = np.random.default_rng(4).uniform(0.01, 0.5, rays[::5].shape[0]).astype(np.float32)
    h32, occ = _check(agg, rays)
    hit = h32["prim_id"] != capi.RRT_NO_HIT
    assert 0.3 < hit.mean() < 1.0
    assert np.array_equal(occ.astype(bool), hit)


def test_instanced_cubes_c2_golden(ctx):
    agg, rays = golden_cases.build_gpu(ctx, "cubes_c2_small")
    h32, _ = _check(agg, rays.astype(np.float32))
    assert (h32["prim_id"] != capi.RRT_NO_HIT).sum() > 1000
    _check(agg, golden_cases.shadow_rays("cubes_c2_small", rays).astype(np.float32))


def test_sphere_field_with_partial_spheres_c4(ctx):
    agg = _partial_spheres_and_field(ctx)
    rng = np.random.default_rng(8)
    n = 200000
    o = rng.uniform(-18, 18, (n, 3))
    d = rng.uniform(-12, 12, (n, 3)) - o
    d /= np.linalg.norm(d, axis=1)[:, None]
    rays = np.concatenate([o, d, np.full((n, 1), np.inf)], axis=1).astype(np.float32)
    rays[: n // 4, 6] = rng.uniform(2.0, 20.0, n // 4)
    h32, _ = _check(agg, rays)
    hit = h32["prim_id"] != capi.RRT_NO_HIT
    assert hit.sum() > n // 10
    # rays leaving the surfaces, from fp32 hit points: the self-hit floor on both sides of the shell
    pts = (rays[hit, 0:3].astype(np.float64) + rays[hit, 3:6].astype(np.float64) * h32["t"][hit, None]).astype(np.float32)
    sec = np.concatenate([pts, synth.random_unit_vectors(pts.shape[0], rng).astype(np.float32),
                          np.full((pts.shape[0], 1), np.inf, np.float32)], axis=1)
    _check(agg, sec)


@pytest.mark.parametrize("kind", ["soup", "cubes"])
def test_literal_tier(ctx, kind):
    a = GpuAggregate(ctx)
    if kind == "soup":
        p, idx = scenes.soup(3000, edge=0.02)
        a.add_triangles(a.add_mesh(p, idx), 0)
        rays = synth.bounce_rays(p, idx, 20000, seed=17)
    else:
        m, inv = scenes.cube_instances(300, extent=20.0)
        a.add_triangles(a.add_mesh(synth.CUBE_P, synth.CUBE_VI, synth.CUBE_N, synth.CUBE_NI), 0, instances=(m, inv))
        rays = synth.camera_like_rays(20000, (0.0, 0.0, -60.0), 20.0)
    a.commit(4, capi.RRT_BUILD_LITERAL)
    h32, _ = _check(a, rays.astype(np.float32))
    assert (h32["prim_id"] != capi.RRT_NO_HIT).sum() > 1000


def test_edge_cases(ctx):
    p, idx = scenes.soup(5000)
    agg = scenes.gpu_soup(ctx, p, idx)
    rng = np.random.default_rng(5)
    assert agg.intersect_f32(np.zeros((0, 7), np.float32)).shape == (0,)
    assert agg.intersect_p_f32(np.zeros((0, 7), np.float32)).shape == (0,)
    for n in (1, 31, 4097, CHUNK + 3, 2 * CHUNK + CHUNK // 3):   # one ray .. several chunks, never a multiple of one
        rays = synth.bounce_rays(p, idx, n, seed=300 + n).astype(np.float32)
        pick = rng.integers(0, 3, n)
        rays[:, 6] = np.where(pick == 0, 0.0, np.where(pick == 1, rng.uniform(0.001, 0.3, n), np.inf))
        _check(agg, rays)
    rays = np.zeros((600, 7), np.float32)
    rays[:, 6] = np.inf
    rays[:300, 0:3] = rng.uniform(0, 1, (300, 3))                    # axis-parallel
    ax = rng.integers(0, 3, 300)
    rays[np.arange(300), 3 + ax] = rng.choice([-1.0, 1.0], 300)
    rays[300:, 0:3] = rng.uniform(-0.2, 1.2, (300, 3))
    rays[300:, 3:6] = synth.random_unit_vectors(300, rng)
    h32, _ = _check(agg, rays)
    assert (h32["prim_id"][:300] != capi.RRT_NO_HIT).sum() > 10
    away = np.zeros((5000, 7), np.float32)                           # all misses
    away[:, 0:3] = rng.uniform(2, 3, (5000, 3))
    away[:, 3] = 1.0
    away[:, 6] = np.inf
    h32, occ = _check(agg, away)
    assert (h32["prim_id"] == capi.RRT_NO_HIT).all() and not occ.any()


def test_device_entries_on_torch_tensors_and_streams(ctx):
    import torch
    p, idx = scenes.soup(30000)
    agg = scenes.gpu_soup(ctx, p, idx)
    s = torch.cuda.Stream()
    for n in (50000, 3, 150000):          # the stream's scratch grows, and is reused at a smaller size
        rays = synth.bounce_rays(p, idx, n, seed=9 + n).astype(np.float32)
        h64, occ64 = _expect(agg, rays)
        d_rays = torch.from_numpy(pack_rays_f32(rays).view(np.float32).reshape(-1).copy()).cuda()
        d_hits = torch.zeros(n * 4, dtype=torch.float32, device="cuda")
        d_occ = torch.zeros(n, dtype=torch.uint8, device="cuda")
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            agg.intersect_f32_device(n, d_rays.data_ptr(), d_hits.data_ptr(), s.cuda_stream)
            agg.intersect_p_f32_device(n, d_rays.data_ptr(), d_occ.data_ptr(), s.cuda_stream)
        s.synchronize()
        _assert_f32_answers(d_hits.cpu().numpy().view(HIT_F32_DTYPE).reshape(-1), h64)
        assert np.array_equal(d_occ.cpu().numpy(), occ64)
    # more streams than the scene keeps scratch for: the extra ones share, ordered by an event
    rays = synth.bounce_rays(p, idx, 40000, seed=99).astype(np.float32)
    h64, _ = _expect(agg, rays)
    d_rays = torch.from_numpy(pack_rays_f32(rays).view(np.float32).reshape(-1).copy()).cuda()
    streams = [torch.cuda.Stream() for _ in range(12)]
    outs = [torch.zeros(40000 * 4, dtype=torch.float32, device="cuda") for _ in streams]
    torch.cuda.synchronize()
    for st, out in zip(streams, outs):
        agg.intersect_f32_device(40000, d_rays.data_ptr(), out.data_ptr(), st.cuda_stream)
    torch.cuda.synchronize()
    for out in outs:
        _assert_f32_answers(out.cpu().numpy().view(HIT_F32_DTYPE).reshape(-1), h64)


def test_concurrent_host_threads_share_one_aggregate(ctx):
    import torch
    p, idx = scenes.soup(20000)
    agg = scenes.gpu_soup(ctx, p, idx)
    batches = [synth.bounce_rays(p, idx, 30000, seed=200 + k).astype(np.float32) for k in range(4)]
    expect = [_expect(agg, b) for b in batches]
    got, occ, dev = [None] * 4, [None] * 4, [None] * 4
    d_rays = [torch.from_numpy(pack_rays_f32(b).view(np.float32).reshape(-1).copy()).cuda() for b in batches]
    torch.cuda.synchronize()

    def work(k):
        st = torch.cuda.Stream()
        out = torch.zeros(30000 * 4, dtype=torch.float32, device="cuda")
        for _ in range(3):
            got[k] = agg.intersect_f32(batches[k])
            occ[k] = agg.intersect_p_f32(batches[k])
            agg.intersect_f32_device(30000, d_rays[k].data_ptr(), out.data_ptr(), st.cuda_stream)
        st.synchronize()
        dev[k] = out.cpu().numpy().view(HIT_F32_DTYPE).reshape(-1)

    th = [threading.Thread(target=work, args=(k,)) for k in range(4)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    for k in range(4):
        _assert_f32_answers(got[k], expect[k][0])
        _assert_f32_answers(dev[k], expect[k][0])
        assert np.array_equal(occ[k], expect[k][1])


def test_errors_are_the_f64_entries(ctx):
    import torch
    L = capi.lib()
    a = GpuAggregate(ctx)
    buf = torch.zeros(64, dtype=torch.float32, device="cuda")
    ptr = C.c_void_p(buf.data_ptr())
    # not committed
    assert L.rrt_intersect_f32(a.h, 4, None, None) == L.rrt_intersect(a.h, 4, None, None) == capi.RRT_ERR_INVALID
    assert L.rrt_intersect_p_f32(a.h, 4, None, None) == L.rrt_intersect_p(a.h, 4, None, None) == capi.RRT_ERR_INVALID
    assert L.rrt_intersect_f32_device(a.h, 4, ptr, ptr, None) == L.rrt_intersect_device(a.h, 4, ptr, ptr, None) == capi.RRT_ERR_INVALID
    assert L.rrt_intersect_p_f32_device(a.h, 4, ptr, ptr, None) == capi.RRT_ERR_INVALID
    with pytest.raises(capi.RrtError) as e:
        a.intersect_f32(np.zeros((4, 7), np.float32))
    assert e.value.status == capi.RRT_ERR_INVALID and "not committed" in str(e.value)
    p, idx = scenes.soup(100)
    a.add_triangles(a.add_mesh(p, idx), 0)
    a.commit()
    # null buffers
    for fn, ref in ((L.rrt_intersect_f32, L.rrt_intersect), (L.rrt_intersect_p_f32, L.rrt_intersect_p)):
        assert fn(a.h, 4, None, None) == ref(a.h, 4, None, None) == capi.RRT_ERR_INVALID
    for fn, ref in ((L.rrt_intersect_f32_device, L.rrt_intersect_device), (L.rrt_intersect_p_f32_device, L.rrt_intersect_p_device)):
        assert fn(a.h, 4, None, ptr, None) == ref(a.h, 4, None, ptr, None) == capi.RRT_ERR_INVALID
        assert fn(a.h, 4, ptr, None, None) == ref(a.h, 4, ptr, None, None) == capi.RRT_ERR_INVALID
        # n = 0 is a no-op, buffers or not
        assert fn(a.h, 0, None, None, None) == ref(a.h, 0, None, None, None) == capi.RRT_OK
        # 2^32 rays or more: refused before any memory is touched
        assert fn(a.h, 1 << 32, ptr, ptr, None) == ref(a.h, 1 << 32, ptr, ptr, None) == capi.RRT_ERR_INVALID
    assert L.rrt_intersect_f32(a.h, 0, None, None) == capi.RRT_OK
    # the vector loads need 16-byte aligned records
    odd = C.c_void_p(buf.data_ptr() + 4)
    assert L.rrt_intersect_f32_device(a.h, 1, odd, ptr, None) == capi.RRT_ERR_INVALID
    assert L.rrt_intersect_f32_device(a.h, 1, ptr, odd, None) == capi.RRT_ERR_INVALID
    assert L.rrt_last_error()
    torch.cuda.synchronize()
