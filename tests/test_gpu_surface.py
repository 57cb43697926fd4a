"""-m gpu: rrt_intersect_surface / rrt_intersect_surface_device (include/rrt.h) against the oracle's SurfaceInteraction
(tests/surface_oracle.py).  A record's `hit` is rrt_intersect's record byte for byte; every other field is a function of the
hit, so where the hit equals the oracle's bit for bit the triangle fields must too.  Hits on rotated instances differ
from the oracle's in the last bits (the walk runs in world space on baked vertices, the oracle in instance space), and
the sphere fields go through the device's atan2 / acos / sin: those rows are held to a relative tolerance per vector."""
import ctypes as C
import threading

import numpy as np
import pytest

import oracle_lib as O
import scenes
import surface_oracle as SO
from rs_ray_toy_b200 import capi, synth
from rs_ray_toy_b200 import transform as T
from rs_ray_toy_b200.aggregate import SURFACE_DTYPE, GpuAggregate, pack_rays

pytestmark = pytest.mark.gpu
SURF_CHUNK = 1 << 18  # rays per host pipeline slot of the surface calls (csrc/capi.cpp)
# rrt_surface after its hit, as the surface oracle lays it out: (name, first double, width)
VECTORS = [("p", 0, 3), ("wo", 3, 3), ("n", 6, 3), ("uv", 9, 2), ("dpdu", 11, 3), ("dpdv", 14, 3), ("dndu", 17, 3),
           ("dndv", 20, 3), ("sh_n", 23, 3), ("sh_dpdu", 26, 3), ("sh_dpdv", 29, 3), ("sh_dndu", 32, 3), ("sh_dndv", 35, 3)]


def _si(rec):
    """The 38 doubles after the hit, [n, 38]."""
    return np.ascontiguousarray(rec).view(np.float64).reshape(-1, 42)[:, 4:]


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def _close(a, b, tol):
    """Per vector: |a - b| <= tol * max(|a|, |b|) (both zero passes)."""
    ok = np.ones(a.shape[0], bool)
    for _, k, w in VECTORS:
        x, y = a[:, k:k + w], b[:, k:k + w]
        ok &= np.linalg.norm(x - y, axis=1) <= tol * np.maximum(np.linalg.norm(x, axis=1), np.linalg.norm(y, axis=1))
    return ok


def _check(rec, hits, ref, exact=True, tol_same=1e-12, tol_moved=1e-9, hit_uv=True, label=""):
    """rec: rrt_surface records; hits: rrt_intersect on the same rays; ref: SurfaceOracle.intersect_si.  exact: the fields of a row
    whose hit equals the oracle's must be bit-equal (triangles), else within tol_same (spheres).  hit_uv = False: the
    hits carry no (u, v) to compare (the literal tier's sphere hits, whose rrt_hit has u = v = 0)."""
    assert rec.dtype == SURFACE_DTYPE
    assert rec["hit"].tobytes() == hits.tobytes()
    h = rec["hit"]
    hit = h["prim_id"] != capi.RRT_NO_HIT
    assert np.array_equal(np.where(hit, h["prim_id"].astype(np.int64), -1), ref["prim"])
    si, rsi = _si(rec), ref["si"]
    assert not _bits(si[~hit]).any()                      # misses: +0.0 everywhere but the hit
    fields = ((h["t"], ref["t"]), (h["u"], ref["uv"][:, 0]), (h["v"], ref["uv"][:, 1]))[:3 if hit_uv else 1]
    same = hit.copy()
    for got, want in fields:
        same &= _bits(got) == _bits(want)
    moved = hit & ~same
    # a hit that differs from the oracle's does so by rounding only
    for got, want in fields:
        assert (np.abs(got[moved] - want[moved]) <= 1e-9 * np.maximum(np.abs(want[moved]), 1.0)).all()
    equal = (_bits(si) == _bits(rsi)).all(axis=1)
    if exact:
        assert equal[same].all(), (label, np.flatnonzero(same & ~equal)[:5])
    else:
        assert _close(si[same], rsi[same], tol_same).all(), label
    assert _close(si[moved], rsi[moved], tol_moved).all(), label
    print(f"{label}: {hit.sum()} hits of {hit.size}, hit equal to the oracle's {same.sum()}, "
          f"records bit-equal to the oracle's {(equal & hit).sum()}")
    return hit


# ---- scenes ----------------------------------------------------------------------------------------------------------
MESH_KINDS = ["n_uv", "n_only", "uv_no_uvi", "bare", "degenerate_uv", "zero_normal"]


def _mesh(kind, k=12, seed=3):
    """A bumpy k x k grid with the attributes `kind` names.  Returns (gpu kwargs, oracle kwargs)."""
    rng = np.random.default_rng(seed)
    x, y = np.meshgrid(np.linspace(-1, 1, k), np.linspace(-1, 1, k))
    p = np.stack([x.ravel(), y.ravel(), 0.15 * np.sin(3 * x.ravel()) * np.cos(2 * y.ravel())], axis=1)
    q = np.arange(k * k).reshape(k, k)
    a, b, c, d = q[:-1, :-1].ravel(), q[:-1, 1:].ravel(), q[1:, :-1].ravel(), q[1:, 1:].ravel()
    vi = np.concatenate([np.stack([a, b, d], 1), np.stack([a, d, c], 1)]).astype(np.uint32)
    n = np.array([0.0, 0.0, 1.0]) + rng.normal(0, 0.3, (k * k, 3))
    uv = np.stack([0.7 * x.ravel() + 0.1 * y.ravel(), 1.3 * y.ravel() - 0.2 * x.ravel()], axis=1)
    g = {"p": p, "vi": vi}
    if kind == "n_uv":
        g.update(n=n, ni=vi, uv=uv, uvi=vi)
    elif kind == "n_only":
        g.update(n=n, ni=vi)
    elif kind == "degenerate_uv":      # every uv on one line: |det| < 1e-8, the coordinate_system fallbacks
        t = x.ravel() + y.ravel()
        g.update(n=n, ni=vi, uv=np.stack([t, 2 * t], 1), uvi=vi)
    elif kind == "zero_normal":        # the interpolated normal has zero length: the geometric normal stands in
        g.update(n=np.zeros((k * k, 3)), ni=vi, uv=uv, uvi=vi)
    o = dict(g)
    if kind == "uv_no_uvi":
        # the reference reads uv indices [0, 0, 0] when a mesh has uvs but no uv indices (triangle.rs:88-98); the C API
        # takes uvs together with their indices, so the library is given those indices explicitly
        g.update(uv=uv, uvi=np.zeros_like(vi))
        o.update(uv=uv)
    return g, o


def _placements():
    """Rotated, non-uniformly scaled, mirrored (det < 0); each one apart from the bare mesh at the origin."""
    return [T.make_to_world((3.0, 0.5, 0.0), (1.0, 2.0, 0.5), 37.0),
            T.make_to_world((-3.0, 0.0, 0.5), (0.3, -1.0, 0.2), 75.0, (1.6, 0.6, 1.1)),
            T.make_to_world((0.0, 3.0, -0.5), (0.0, 0.0, 1.0), 20.0, (-1.2, 0.9, 1.0))]


def _mesh_scenes(ctx, kind, tier=O.TIER_F, build=capi.RRT_BUILD_FAST):
    g, o = _mesh(kind)
    a = GpuAggregate(ctx)
    s = SO.SurfaceOracle(tier)
    mesh = a.add_mesh(**g)
    a.add_triangles(mesh, 0)
    om = s.add_mesh(**o)
    g0 = s.add_geo_triangles(om)
    nt = g["vi"].shape[0]
    s.add_prims(g0, nt, -1)
    xs = _placements()
    a.add_triangles(mesh, 0, instances=(np.array([m for m, _ in xs]), np.array([i for _, i in xs])))
    for m, inv in xs:
        s.add_prims(g0, nt, s.add_xform(m, inv))
    a.commit(4, build)
    s.build(4)
    return a, s


def _rays_at(n, seed, extent=4.0, eye=(1.0, -2.0, 9.0)):
    """Camera-like rays over the scene, some of them missing it, and bounce rays leaving surfaces."""
    rng = np.random.default_rng(seed)
    cam = synth.camera_like_rays(n, eye, extent, seed=seed)
    return cam, rng


def _bounce(rec, rng, k):
    h = rec["hit"]
    hit = h["prim_id"] != capi.RRT_NO_HIT
    p = rec["p"][hit][:k]
    nrm = rec["n"][hit][:k]
    d = synth.random_unit_vectors(p.shape[0], rng)
    return np.concatenate([p + 1e-6 * nrm * np.sign((d * nrm).sum(1))[:, None], d, np.full((p.shape[0], 1), np.inf)], 1)


# ---- 1. triangles -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", MESH_KINDS)
def test_triangle_attribute_matrix(ctx, kind):
    a, s = _mesh_scenes(ctx, kind)
    cam, rng = _rays_at(60000, seed=40 + MESH_KINDS.index(kind))
    rec = a.intersect_surface(cam)
    hit = _check(rec, a.intersect(cam), s.intersect_si(cam), label=f"{kind} camera")
    assert hit.sum() > 5000 and (~hit).sum() > 1000
    sec = _bounce(rec, rng, 40000)
    _check(a.intersect_surface(sec), a.intersect(sec), s.intersect_si(sec), label=f"{kind} bounce")
    if kind == "n_uv":   # the vertex normals make a shading frame of their own (the shading normal stays the geometric
        # one, flipped towards it: set_shading_geometry with orientation_is_authoritative, interaction.rs:186-202)
        assert (np.abs(rec["sh_dpdu"][hit] - rec["dpdu"][hit]).sum(1) > 1e-6).mean() > 0.9
        assert (np.abs(rec["sh_dndu"][hit]).sum(1) > 0).mean() > 0.9


# ---- 2. spheres -------------------------------------------------------------------------------------------------------
def _sphere_scenes(ctx, tier=O.TIER_F, clipped=True, build=capi.RRT_BUILD_FAST):
    rng = np.random.default_rng(21)
    a = GpuAggregate(ctx)
    s = SO.SurfaceOracle(tier)
    for k in range(12):   # full spheres with their own obj_to_world: rotated, scaled, some mirrored
        sc = rng.uniform(0.6, 1.5, 3)
        if k % 4 == 3:
            sc[0] = -sc[0]
        sc = tuple(float(v) for v in sc)
        xf = T.make_to_world(rng.uniform(-8, 8, 3), rng.normal(0, 1, 3), float(rng.uniform(0, 360)), sc)
        r = float(rng.uniform(0.5, 1.5))
        a.add_sphere(radius=r, obj_to_world=xf)
        s.add_prims(s.add_geo_sphere(s.add_sphere(xf[0], xf[1], r)), 1, -1)
    for k in range(16):   # spheres placed through instances, clipped in z and phi
        r = float(rng.uniform(0.5, 1.5))
        z0, z1 = (sorted((float(rng.uniform(-r, 0.2 * r)), float(rng.uniform(0.3 * r, r)))) if clipped and k % 2
                  else (-r, r))
        phi = float(rng.uniform(60, 330)) if clipped and k % 3 else 360.0
        xs = [T.make_to_world(rng.uniform(-8, 8, 3), rng.normal(0, 1, 3), float(rng.uniform(0, 360)),
                              tuple(rng.uniform(0.6, 1.6, 3) * (-1.0 if j == 1 else 1.0))) for j in range(3)]
        a.add_sphere(radius=r, z_min=z0, z_max=z1, phi_max=phi,
                     instances=(np.array([m for m, _ in xs]), np.array([i for _, i in xs])))
        g = s.add_geo_sphere(s.add_sphere(None, None, r, z0, z1, phi))
        for m, inv in xs:
            s.add_prims(g, 1, s.add_xform(m, inv))
    a.commit(4, build)
    s.build(4)
    return a, s


def test_spheres_own_transforms_instances_and_clipping(ctx):
    a, s = _sphere_scenes(ctx)
    rng = np.random.default_rng(5)
    n = 120000
    o = rng.uniform(-14, 14, (n, 3))
    d = rng.uniform(-9, 9, (n, 3)) - o
    d /= np.linalg.norm(d, axis=1)[:, None]
    rays = np.concatenate([o, d, np.full((n, 1), np.inf)], axis=1)
    rays[: n // 4, 6] = rng.uniform(2.0, 20.0, n // 4)
    rec = a.intersect_surface(rays)
    hit = _check(rec, a.intersect(rays), s.intersect_si(rays), exact=False, label="spheres")
    assert hit.sum() > n // 20
    sec = _bounce(rec, rng, 60000)   # leaving the shells, inside and out: far roots of clipped spheres
    _check(a.intersect_surface(sec), a.intersect(sec), s.intersect_si(sec), exact=False, label="spheres bounce")


# ---- 3. config 3 at a million rays through the device entry ----------------------------------------------------------
def test_config3_soup_device_entry(ctx):
    import torch
    p, idx = scenes.soup(1 << 20)
    agg = scenes.gpu_soup(ctx, p, idx)
    n = 1 << 20
    rays = pack_rays(synth.bounce_rays(p, idx, n, seed=71))
    d_rays = torch.from_numpy(rays.view(np.float64).reshape(-1).copy()).cuda()
    d_hits = torch.zeros(n * 4, dtype=torch.float64, device="cuda")
    d_surf = torch.zeros(n * 42, dtype=torch.float64, device="cuda")
    agg.intersect_device(n, d_rays.data_ptr(), d_hits.data_ptr())
    before = ctx.launch_count
    agg.intersect_surface_device(n, d_rays.data_ptr(), d_surf.data_ptr())
    launched = ctx.launch_count - before
    torch.cuda.synchronize()
    rec = d_surf.cpu().numpy().view(SURFACE_DTYPE)
    hits = d_hits.cpu().numpy().view(np.uint8)
    assert rec["hit"].tobytes() == hits.tobytes()
    before = ctx.launch_count
    agg.intersect_device(n, d_rays.data_ptr(), d_hits.data_ptr())
    assert launched == ctx.launch_count - before + 1       # the walk's launches and the surface pass
    sl = slice(300000, 300000 + (1 << 16))
    raw = np.stack([rays["o"][:, 0], rays["o"][:, 1], rays["o"][:, 2], rays["d"][:, 0], rays["d"][:, 1], rays["d"][:, 2],
                    rays["t_max"]], axis=1)[sl]
    ref = SO.soup(p, idx).intersect_si(raw)
    hit = _check(rec[sl], rec[sl]["hit"], ref, label="config 3 slice")
    assert hit.mean() > 0.3
    same = _bits(rec[sl]["hit"]["t"])[hit] == _bits(ref["t"])[hit]
    assert same.all()                                     # bare triangles: the walk's t is the oracle's


# ---- 4. build paths ---------------------------------------------------------------------------------------------------
def test_build_paths_give_identical_records(ctx):
    cam, _ = _rays_at(40000, seed=8)
    out = []
    for build in (capi.RRT_BUILD_FAST, capi.RRT_BUILD_DEVICE_LBVH):
        a, _ = _mesh_scenes(ctx, "n_uv", build=build)
        out.append(a.intersect_surface(cam))
        if build == capi.RRT_BUILD_FAST:
            blob = a.export_tree()
    g, _ = _mesh("n_uv")
    b = GpuAggregate(ctx)
    mesh = b.add_mesh(**g)
    b.add_triangles(mesh, 0)
    xs = _placements()
    b.add_triangles(mesh, 0, instances=(np.array([m for m, _ in xs]), np.array([i for _, i in xs])))
    b.commit_from_tree(blob)
    out.append(b.intersect_surface(cam))
    assert out[0].tobytes() == out[1].tobytes() == out[2].tobytes()
    sa, _ = _sphere_scenes(ctx, build=capi.RRT_BUILD_FAST)
    sb, _ = _sphere_scenes(ctx, build=capi.RRT_BUILD_DEVICE_LBVH)
    rng = np.random.default_rng(2)
    rays = np.concatenate([rng.uniform(-12, 12, (40000, 3)), synth.random_unit_vectors(40000, rng),
                           np.full((40000, 1), np.inf)], axis=1)
    assert sa.intersect_surface(rays).tobytes() == sb.intersect_surface(rays).tobytes()


# ---- 5. Tier L --------------------------------------------------------------------------------------------------------
def test_literal_tier(ctx):
    m, inv = scenes.cube_instances(200, extent=12.0)
    a = scenes.gpu_cubes(ctx, m, inv, build_flags=capi.RRT_BUILD_LITERAL)
    s = SO.cubes(m, inv, tier=O.TIER_L)
    rays = synth.camera_like_rays(40000, (0.0, 0.0, -40.0), 12.0)
    rec = a.intersect_surface(rays)
    hit = _check(rec, a.intersect(rays), s.intersect_si(rays), label="literal cubes")
    assert hit.sum() > 5000
    ms, invs = scenes.sphere_instances(500, extent=10.0)
    a = scenes.gpu_spheres(ctx, ms, invs, build_flags=capi.RRT_BUILD_LITERAL)
    s = SO.spheres(ms, invs, tier=O.TIER_L)
    rays = synth.camera_like_rays(40000, (0.0, 0.0, -30.0), 10.0, seed=3)
    rec = a.intersect_surface(rays)
    hit = _check(rec, a.intersect(rays), s.intersect_si(rays), exact=False, hit_uv=False, label="literal spheres")
    assert (rec["uv"][hit] > 0).any(axis=1).all()   # the record has the sphere's (u, v) although its rrt_hit has none
    assert hit.sum() > 2000


# ---- 6. moved instances -----------------------------------------------------------------------------------------------
def test_update_instances_refreshes_the_tables(ctx):
    m0, inv0 = scenes.cube_instances(300, extent=8.0)
    agg = scenes.gpu_cubes(ctx, m0, inv0)
    rng = np.random.default_rng(16)
    rays = np.concatenate([rng.uniform(-12, 12, (60000, 3)), synth.random_unit_vectors(60000, rng),
                           np.full((60000, 1), np.inf)], axis=1)
    _check(agg.intersect_surface(rays), agg.intersect(rays), SO.cubes(m0, inv0).intersect_si(rays),
           label="cubes before")
    m1, inv1 = scenes.cube_instances(300, extent=8.0, seed=991)
    k = 120
    agg.update_instances(0, m1[:k], inv1[:k])
    m_new, inv_new = np.concatenate([m1[:k], m0[k:]]), np.concatenate([inv1[:k], inv0[k:]])
    _check(agg.intersect_surface(rays), agg.intersect(rays), SO.cubes(m_new, inv_new).intersect_si(rays),
           label="cubes after")


# ---- 7. host entry ----------------------------------------------------------------------------------------------------
def _device_records(agg, rays, stream=0):
    import torch
    r = pack_rays(rays)
    n = r.shape[0]
    d_rays = torch.from_numpy(r.view(np.float64).reshape(-1).copy()).cuda()
    d_surf = torch.zeros(n * 42, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    agg.intersect_surface_device(n, d_rays.data_ptr(), d_surf.data_ptr(), stream)
    torch.cuda.synchronize()
    return d_surf.cpu().numpy().view(SURFACE_DTYPE)


def test_host_entry_chunking_and_buffers(ctx):
    a, _ = _mesh_scenes(ctx, "n_uv")
    assert a.intersect_surface(np.zeros((0, 7))).shape == (0,)
    for n in (1, SURF_CHUNK - 1, SURF_CHUNK, SURF_CHUNK + 1, 3 * SURF_CHUNK + 12345):
        rays, _ = _rays_at(n, seed=n % 1000)
        dev = _device_records(a, rays)
        plain = a.intersect_surface(rays)
        assert plain.tobytes() == dev.tobytes(), n
        assert plain["hit"].tobytes() == a.intersect(rays).tobytes()
        if n > SURF_CHUNK:
            pinned = ctx.pinned_empty(n, SURFACE_DTYPE)
            a.intersect_surface(rays, out=pinned)
            assert pinned.tobytes() == dev.tobytes(), n


# ---- 8. concurrency ---------------------------------------------------------------------------------------------------
def test_torch_streams_beyond_the_scratch_slots(ctx):
    import torch
    a, _ = _mesh_scenes(ctx, "n_only")
    rays, _ = _rays_at(30000, seed=77)
    want = a.intersect_surface(rays).tobytes()
    d_rays = torch.from_numpy(pack_rays(rays).view(np.float64).reshape(-1).copy()).cuda()
    streams = [torch.cuda.Stream() for _ in range(12)]
    outs = [torch.zeros(30000 * 42, dtype=torch.float64, device="cuda") for _ in streams]
    torch.cuda.synchronize()
    for rep in range(2):   # the second round grows nothing and reuses every stream's (or the shared) scratch
        for st, out in zip(streams, outs):
            a.intersect_surface_device(30000, d_rays.data_ptr(), out.data_ptr(), st.cuda_stream)
    torch.cuda.synchronize()
    for out in outs:
        assert out.cpu().numpy().tobytes() == want


def test_concurrent_host_threads_on_one_scene(ctx):
    import torch
    a, _ = _sphere_scenes(ctx)
    rng = np.random.default_rng(31)
    batches = [np.concatenate([rng.uniform(-12, 12, (30000, 3)), synth.random_unit_vectors(30000, rng),
                               np.full((30000, 1), np.inf)], axis=1) for _ in range(4)]
    want = [a.intersect_surface(b).tobytes() for b in batches]
    d_rays = [torch.from_numpy(pack_rays(b).view(np.float64).reshape(-1).copy()).cuda() for b in batches]
    torch.cuda.synchronize()
    got, dev = [None] * 4, [None] * 4

    def work(k):
        st = torch.cuda.Stream()
        out = torch.zeros(30000 * 42, dtype=torch.float64, device="cuda")
        for _ in range(3):
            got[k] = a.intersect_surface(batches[k]).tobytes()
            a.intersect_surface_device(30000, d_rays[k].data_ptr(), out.data_ptr(), st.cuda_stream)
        st.synchronize()
        dev[k] = out.cpu().numpy().tobytes()

    th = [threading.Thread(target=work, args=(k,)) for k in range(4)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert got == want and dev == want


# ---- 9. errors --------------------------------------------------------------------------------------------------------
def test_errors_are_the_intersect_entries(ctx):
    import torch
    L = capi.lib()
    a = GpuAggregate(ctx)
    buf = torch.zeros(64, dtype=torch.float64, device="cuda")
    ptr = C.c_void_p(buf.data_ptr())
    assert L.rrt_intersect_surface(a.h, 4, None, None) == L.rrt_intersect(a.h, 4, None, None) == capi.RRT_ERR_INVALID
    assert L.rrt_intersect_surface_device(a.h, 4, ptr, ptr, None) == L.rrt_intersect_device(a.h, 4, ptr, ptr, None) \
        == capi.RRT_ERR_INVALID
    with pytest.raises(capi.RrtError) as e:
        a.intersect_surface(np.zeros((4, 7)))
    assert e.value.status == capi.RRT_ERR_INVALID and "not committed" in str(e.value)
    p, idx = scenes.soup(100)
    a.add_triangles(a.add_mesh(p, idx), 0)
    a.commit()
    assert L.rrt_intersect_surface(a.h, 4, None, None) == L.rrt_intersect(a.h, 4, None, None) == capi.RRT_ERR_INVALID
    fn, ref = L.rrt_intersect_surface_device, L.rrt_intersect_device
    assert fn(a.h, 4, None, ptr, None) == ref(a.h, 4, None, ptr, None) == capi.RRT_ERR_INVALID
    assert fn(a.h, 4, ptr, None, None) == ref(a.h, 4, ptr, None, None) == capi.RRT_ERR_INVALID
    assert fn(a.h, 0, None, None, None) == ref(a.h, 0, None, None, None) == capi.RRT_OK
    assert L.rrt_intersect_surface(a.h, 0, None, None) == L.rrt_intersect(a.h, 0, None, None) == capi.RRT_OK
    assert fn(a.h, 1 << 32, ptr, ptr, None) == ref(a.h, 1 << 32, ptr, ptr, None) == capi.RRT_ERR_INVALID
    assert L.rrt_last_error()
    torch.cuda.synchronize()
