"""rrt_scene_update_mesh / rrt_scene_update_mesh_device: after an update every call answers like a fresh scene given the
new vertices and committed with RRT_BUILD_DEVICE_LBVH ("H" below), bit for bit, and the exported aggregate is H's but
for the two timing fields of its statistics."""
import numpy as np
import pytest

import oracle_lib as O
import scenes
import surface_oracle as SO
from rs_ray_toy_b200 import capi, synth
from rs_ray_toy_b200 import render as R
from rs_ray_toy_b200 import transform as T
from rs_ray_toy_b200.aggregate import GpuAggregate
from rs_ray_toy_b200.render import Render
from test_gpu_surface import _check

pytestmark = pytest.mark.gpu
LBVH = capi.RRT_BUILD_DEVICE_LBVH
# BlobHeader: magic, version, AggView (152 B), then AggregateStats; build_usec is its 5th word, tree_device_usec its 9th
TIMING_WORDS = (16 + 152 + 8 * 4, 16 + 152 + 8 * 8)


def _blob(agg):
    b = agg.export_tree().copy()
    for at in TIMING_WORDS:
        b[at:at + 8] = 0
    return b


def _same_aggregate(a, h):
    ba, bh = _blob(a), _blob(h)
    assert ba.size == bh.size and (ba == bh).all(), np.flatnonzero(ba != bh)[:8] if ba.size == bh.size else (ba.size, bh.size)
    sa, sh = a.stats(), h.stats()
    sa.pop("build_usec"), sh.pop("build_usec")
    assert sa == sh
    ia, ih = a.build_info(), h.build_info()
    ia.pop("tree_device_usec"), ih.pop("tree_device_usec")
    assert ia == ih and ia["device_lbvh"]


def _same_answers(a, h, rays):
    assert a.intersect(rays).tobytes() == h.intersect(rays).tobytes()
    assert a.intersect_p(rays).tobytes() == h.intersect_p(rays).tobytes()
    r32 = rays.astype(np.float32)
    assert a.intersect_f32(r32).tobytes() == h.intersect_f32(r32).tobytes()
    assert (a.world_bound() == h.world_bound()).all()
    assert a.num_prims == h.num_prims


def _soup_scene(ctx, p, idx, flags):
    a = GpuAggregate(ctx)
    mesh = a.add_mesh(p, idx)
    a.add_triangles(mesh, 0)
    return a.commit(4, flags), mesh


def _displaced_f32(p, seed, scale=2e-3):
    """p moved by a seeded float32 offset, in float32: every coordinate stays an fp32 value (PrimRec48)."""
    off = np.random.default_rng(seed).normal(0.0, scale, p.shape).astype(np.float32)
    return (p.astype(np.float32) + off).astype(np.float64), off


def _assert_oracle(hits, ref):
    c = scenes.compare_closest(hits, ref["prim"], ref["t"], 1e-6, 1e-5)
    assert c["mismatch_excl_ties"] == 0 and c["t_bad"] == 0, c
    return c


# ---- 1. and 2. a bare soup through both entries ------------------------------------------------------------------------
def test_bare_soup_host_and_device_entries(ctx):
    import torch
    p, idx = scenes.soup(1 << 18)
    a, mesh = _soup_scene(ctx, p, idx, capi.RRT_BUILD_FAST)
    assert not a.build_info()["device_lbvh"]
    p1, off = _displaced_f32(p, seed=5)
    a.update_mesh(mesh, p1)
    rays = synth.bounce_rays(p1, idx, 1 << 20, seed=17)
    c = _assert_oracle(a.intersect(rays), scenes.oracle_soup(p1, idx).intersect(rays))
    assert c["hits"] > (1 << 18)
    h, _ = _soup_scene(ctx, p1, idx, LBVH)
    _same_answers(a, h, rays)
    _same_aggregate(a, h)
    assert a.stats()["wide_records"] == 0
    blob1 = _blob(a)

    # the same update from a tensor that torch writes on a side stream, passed with that stream
    b, mesh_b = _soup_scene(ctx, p, idx, capi.RRT_BUILD_FAST)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        d_p = (torch.from_numpy(p.astype(np.float32)).cuda() + torch.from_numpy(off).cuda()).double().contiguous()
        b.update_mesh_device(mesh_b, 0, p.shape[0], d_p.data_ptr(), stream=side.cuda_stream)
    assert (_blob(b) == blob1).all()
    # a middle range only
    lo, hi = p.shape[0] // 3, 2 * p.shape[0] // 3
    p2 = p1.copy()
    p2[lo:hi], _ = _displaced_f32(p1[lo:hi], seed=6, scale=5e-3)
    d_mid = torch.from_numpy(p2[lo:hi].copy()).cuda()
    torch.cuda.synchronize()
    b.update_mesh_device(mesh_b, lo, hi - lo, d_mid.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
    h2, _ = _soup_scene(ctx, p2, idx, LBVH)
    rays2 = synth.bounce_rays(p2, idx, 1 << 20, seed=18)
    _same_answers(b, h2, rays2)
    _same_aggregate(b, h2)


# ---- 3. a mixed scene: soup, instanced cubes, full and clipped spheres -----------------------------------------------------
def _mixed(ctx, cube_p, flags, oracle=False):
    p, idx = scenes.soup(20000, edge=0.02, seed=31)
    p = p * 16.0 - 8.0                                 # (powers of two: still fp32 values)
    m, inv = scenes.cube_instances(300, extent=8.0)
    sm, sinv = scenes.sphere_instances(40, extent=8.0, seed=9)
    a = GpuAggregate(ctx)
    soup = a.add_mesh(p, idx)
    a.add_triangles(soup, 0)
    cube = a.add_mesh(cube_p, synth.CUBE_VI, synth.CUBE_N, synth.CUBE_NI)
    a.add_triangles(cube, 0, instances=(m, inv))
    a.add_sphere(radius=0.75, obj_to_world=T.make_to_world((2.0, -1.0, 0.5)))
    a.add_sphere(radius=0.5, instances=(sm[:20], sinv[:20]))
    a.add_sphere(radius=0.6, z_min=-0.2, z_max=0.45, phi_max=250.0, instances=(sm[20:], sinv[20:]))
    a.commit(4, flags)
    if not oracle:
        return a, cube
    s = O.OracleScene(O.TIER_F)
    g = s.add_geo_triangles(s.add_mesh(p, idx))
    s.add_prims(g, idx.shape[0], -1)
    gc = s.add_geo_triangles(s.add_mesh(cube_p, synth.CUBE_VI, synth.CUBE_N, synth.CUBE_NI))
    for i in range(m.shape[0]):
        s.add_prims(gc, 12, s.add_xform(m[i], inv[i]))
    xf = T.make_to_world((2.0, -1.0, 0.5))
    s.add_prims(s.add_geo_sphere(s.add_sphere(xf[0], xf[1], 0.75)), 1, -1)
    g1 = s.add_geo_sphere(s.add_sphere(None, None, 0.5))
    for i in range(20):
        s.add_prims(g1, 1, s.add_xform(sm[i], sinv[i]))
    g2 = s.add_geo_sphere(s.add_sphere(None, None, 0.6, -0.2, 0.45, 250.0))
    for i in range(20, 40):
        s.add_prims(g2, 1, s.add_xform(sm[i], sinv[i]))
    s.build(4)
    return a, cube, s


def test_mixed_scene_moves_every_instance_and_no_sphere(ctx):
    a, cube = _mixed(ctx, synth.CUBE_P, capi.RRT_BUILD_FAST)
    rng = np.random.default_rng(3)
    rays = np.concatenate([rng.uniform(-12, 12, (1 << 20, 3)), synth.random_unit_vectors(1 << 20, rng),
                           np.full((1 << 20, 1), np.inf)], axis=1)
    before = a.intersect(rays)
    cube_p = (synth.CUBE_P * np.array([0.75, 1.25, 0.5])).astype(np.float32).astype(np.float64)
    a.update_mesh(cube, cube_p)
    h, _, s = _mixed(ctx, cube_p, LBVH, oracle=True)
    after = a.intersect(rays)
    _assert_oracle(after, s.intersect(rays))
    _same_answers(a, h, rays)
    _same_aggregate(a, h)
    # all 300 cubes moved: prim ids 20000 .. 23599
    moved = (after["prim_id"] != before["prim_id"]) & (after["prim_id"] >= 20000) & (after["prim_id"] < 23600)
    assert len(np.unique((after["prim_id"][moved] - 20000) // 12)) > 200


# ---- 4. record and node formats follow the vertices ---------------------------------------------------------------------
def test_record_format_flips_both_ways(ctx):
    p, idx = scenes.soup(30000, seed=44)
    a, mesh = _soup_scene(ctx, p, idx, LBVH)
    rays = synth.bounce_rays(p, idx, 200000, seed=4)
    f64 = p + np.random.default_rng(1).uniform(-1e-9, 1e-9, p.shape)     # not fp32 values: PrimRec96
    back, _ = _displaced_f32(p, seed=2)
    for step, q in enumerate((f64, back)):
        a.update_mesh(mesh, q)
        h, _ = _soup_scene(ctx, q, idx, LBVH)
        assert a.stats()["wide_records"] == h.stats()["wide_records"] == (1 if step == 0 else 0)
        assert a.build_info()["node_bytes"] == h.build_info()["node_bytes"]
        _same_answers(a, h, rays)
        _same_aggregate(a, h)


# ---- 5. vertex normals and the surface records --------------------------------------------------------------------------
def _normal_mesh(z_scale, normal_seed, k=48):
    x, y = np.meshgrid(np.linspace(-1, 1, k), np.linspace(-1, 1, k))
    p = np.stack([x.ravel(), y.ravel(), z_scale * np.sin(3 * x.ravel()) * np.cos(2 * y.ravel())], axis=1)
    q = np.arange(k * k).reshape(k, k)
    a, b, c, d = q[:-1, :-1].ravel(), q[:-1, 1:].ravel(), q[1:, :-1].ravel(), q[1:, 1:].ravel()
    vi = np.concatenate([np.stack([a, b, d], 1), np.stack([a, d, c], 1)]).astype(np.uint32)
    n = np.array([0.0, 0.0, 1.0]) + np.random.default_rng(normal_seed).normal(0, 0.3, (k * k, 3))
    uv = np.stack([0.5 * x.ravel() + 0.5, 0.5 * y.ravel() + 0.5], axis=1)
    return dict(p=p, vi=vi, n=n, ni=vi, uv=uv, uvi=vi)


def _placed(ctx, g, flags, with_oracle=False):
    xs = [T.make_to_world((3.0, 0.5, 0.0), (1.0, 2.0, 0.5), 37.0),
          T.make_to_world((-3.0, 0.0, 0.5), (0.3, -1.0, 0.2), 75.0, (1.6, 0.6, 1.1))]
    a = GpuAggregate(ctx)
    mesh = a.add_mesh(**g)
    a.add_triangles(mesh, 0)
    a.add_triangles(mesh, 0, instances=(np.array([m for m, _ in xs]), np.array([i for _, i in xs])))
    a.commit(4, flags)
    if not with_oracle:
        return a, mesh
    s = SO.SurfaceOracle(O.TIER_F)
    g0 = s.add_geo_triangles(s.add_mesh(**g))
    nt = g["vi"].shape[0]
    s.add_prims(g0, nt, -1)
    for m, inv in xs:
        s.add_prims(g0, nt, s.add_xform(m, inv))
    s.build(4)
    return a, mesh, s


def test_positions_and_normals_update_the_surface_records(ctx):
    g0, g1 = _normal_mesh(0.15, 1), _normal_mesh(0.3, 2)
    a, mesh = _placed(ctx, g0, capi.RRT_BUILD_FAST)
    rays = synth.camera_like_rays(200000, (0.5, -2.0, 9.0), 5.0, seed=9)
    a.intersect_surface(rays)                      # the surface tables exist before the update
    a.update_mesh(mesh, g1["p"], normals=g1["n"])
    h, _, s = _placed(ctx, g1, LBVH, with_oracle=True)
    rec = a.intersect_surface(rays)
    assert rec.tobytes() == h.intersect_surface(rays).tobytes()
    assert (a.world_bound() == h.world_bound()).all()
    _same_aggregate(a, h)
    hit = _check(rec, a.intersect(rays), s.intersect_si(rays), label="updated grid")
    assert hit.sum() > 10000
    # the shading frame comes from the new vertex normals
    assert (np.abs(rec["sh_dndu"][hit]).sum(1) > 0).mean() > 0.9


# ---- 6. an animation through the device entry -----------------------------------------------------------------------------
def test_ten_frames_of_device_updates(ctx):
    import torch
    p, idx = scenes.soup(1 << 16, seed=12)
    a, mesh = _soup_scene(ctx, p, idx, capi.RRT_BUILD_FAST)
    base = torch.from_numpy(p.astype(np.float32)).cuda()
    d_p = torch.empty(p.shape, dtype=torch.float64, device="cuda")
    free = {}
    for frame in range(1, 11):
        q = torch.from_numpy(np.random.default_rng(100 + frame).normal(0, 2e-3, p.shape).astype(np.float32)).cuda()
        d_p.copy_(base + q)
        a.update_mesh_device(mesh, 0, p.shape[0], d_p.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
        pf = d_p.cpu().numpy()
        rays = synth.bounce_rays(pf, idx, 100000, seed=frame)
        hits = a.intersect(rays)
        torch.cuda.synchronize()
        free[frame] = torch.cuda.mem_get_info()[0]
        h, _ = _soup_scene(ctx, pf, idx, LBVH)
        assert hits.tobytes() == h.intersect(rays).tobytes(), frame
        _same_aggregate(a, h)
        h.close()
    assert free[10] == free[2], free


# ---- 7. replication and a later instance update ---------------------------------------------------------------------------
def test_export_and_instance_update_after_a_mesh_update(ctx):
    p, idx = scenes.soup(40000, seed=8)
    a, mesh = _soup_scene(ctx, p, idx, capi.RRT_BUILD_FAST)
    p1, _ = _displaced_f32(p, seed=9)
    a.update_mesh(mesh, p1)
    b = GpuAggregate(ctx)
    b.add_triangles(b.add_mesh(p1, idx), 0)
    b.commit_from_tree(a.export_tree())
    rays = synth.bounce_rays(p1, idx, 200000, seed=3)
    _same_answers(a, b, rays)
    # instanced cubes: the mesh moves, then the instances; the instance update re-bakes from the new vertices
    m0, inv0 = scenes.cube_instances(300, extent=8.0)
    c = scenes.gpu_cubes(ctx, m0, inv0)
    cube_p = (synth.CUBE_P * 0.625).astype(np.float64)
    c.update_mesh(0, cube_p)
    m1, inv1 = scenes.cube_instances(300, extent=8.0, seed=991)
    c.update_instances(0, m1[:120], inv1[:120])
    mn, invn = np.concatenate([m1[:120], m0[120:]]), np.concatenate([inv1[:120], inv0[120:]])
    h = GpuAggregate(ctx)
    h.add_triangles(h.add_mesh(cube_p, synth.CUBE_VI, synth.CUBE_N, synth.CUBE_NI), 0, instances=(mn, invn))
    h.commit(4, LBVH)
    rng = np.random.default_rng(16)
    rays = np.concatenate([rng.uniform(-12, 12, (200000, 3)), synth.random_unit_vectors(200000, rng),
                           np.full((200000, 1), np.inf)], axis=1)
    _same_answers(c, h, rays)
    _same_aggregate(c, h)
    # and a mesh update after the instance update
    cube_p2 = (synth.CUBE_P * 0.875).astype(np.float64)
    c.update_mesh(0, cube_p2)
    h2 = GpuAggregate(ctx)
    h2.add_triangles(h2.add_mesh(cube_p2, synth.CUBE_VI, synth.CUBE_N, synth.CUBE_NI), 0, instances=(mn, invn))
    h2.commit(4, LBVH)
    _same_answers(c, h2, rays)
    _same_aggregate(c, h2)


# ---- 8. scenes a device commit gives the host SAH tree ----------------------------------------------------------------------
def _deep_soup():
    """5000 copies of one tiny triangle + one per Morton bit: a radix tree deeper than the traversal stack
    (test_gpu_parity.test_device_lbvh_duplicates_and_a_tree_too_deep_for_the_stack)."""
    tri = np.array([[0.0, 0.0, 0.0], [1e-3, 0.0, 0.0], [0.0, 1e-3, 0.0]]) * 1e-9
    pts = [np.zeros(3)]
    for j in range(21):
        for axis in range(3):
            q = np.zeros(3)
            q[axis] = 2.0 ** j / 2.0 ** 21
            pts.append(q)
    p = np.concatenate([np.tile(tri, (5000, 1))] + [tri + q * 0.5 for q in pts])
    return p, np.arange(len(p), dtype=np.uint32).reshape(-1, 3)


def test_small_and_too_deep_scenes_fall_back_like_a_commit(ctx):
    p, idx = scenes.soup(12)
    a, mesh = _soup_scene(ctx, p, idx, capi.RRT_BUILD_FAST)
    p1, _ = _displaced_f32(p, seed=3)
    a.update_mesh(mesh, p1)
    h, _ = _soup_scene(ctx, p1, idx, LBVH)
    rays = synth.bounce_rays(p1, idx, 20000, seed=3)
    _assert_oracle(a.intersect(rays), scenes.oracle_soup(p1, idx).intersect(rays))
    assert a.build_info() == h.build_info() and a.build_info()["tree_device_usec"] == 0
    _same_answers(a, h, rays)
    _same_aggregate(a, h)
    # a scene that the device can build first, then moved into one with a radix tree too deep for the stack
    pd, idx = _deep_soup()
    p0, _ = scenes.soup(idx.shape[0], seed=5)
    a, mesh = _soup_scene(ctx, p0, idx, capi.RRT_BUILD_FAST)
    a.update_mesh(mesh, p0[::-1].copy())                       # a device-built update first
    assert a.build_info()["tree_device_usec"] > 0
    a.update_mesh(mesh, pd)
    h, _ = _soup_scene(ctx, pd, idx, LBVH)
    assert a.build_info() == h.build_info() and a.build_info()["tree_device_usec"] == 0
    rng = np.random.default_rng(12)
    o = np.concatenate([rng.uniform(-0.1, 0.6, (4000, 2)), np.full((4000, 1), 1.0)], axis=1)
    rays = np.concatenate([o, np.tile([0.0, 0.0, -1.0], (4000, 1)), np.full((4000, 1), np.inf)], axis=1)
    rays[:500, 0:2] = 2e-13
    _assert_oracle(a.intersect(rays), scenes.oracle_soup(pd, idx).intersect(rays))
    _same_answers(a, h, rays)
    _same_aggregate(a, h)


# ---- 9. refused calls leave the scene as it was --------------------------------------------------------------------------
def test_errors_leave_the_scene_unchanged(ctx):
    import torch
    L = capi.lib()
    p, idx = scenes.soup(5000, seed=2)
    a, mesh = _soup_scene(ctx, p, idx, capi.RRT_BUILD_FAST)
    rays = synth.bounce_rays(p, idx, 50000, seed=2)
    before, blob = a.intersect(rays), a.export_tree()
    nv = p.shape[0]
    p1, _ = _displaced_f32(p, seed=1)

    def status(call):
        with pytest.raises(capi.RrtError) as e:
            call()
        return e.value.status

    d = torch.from_numpy(p1).cuda()
    assert L.rrt_scene_update_mesh(a.h, mesh, 0, 3, None, 0, 0, None) == capi.RRT_ERR_INVALID
    assert L.rrt_scene_update_mesh(a.h, mesh, 0, 0, None, 0, 3, None) == capi.RRT_ERR_INVALID
    assert L.rrt_scene_update_mesh_device(a.h, mesh, 0, 3, None, 0, 0, None, None) == capi.RRT_ERR_INVALID
    assert L.rrt_scene_update_mesh(None, mesh, 0, 3, p1.ctypes.data, 0, 0, None) == capi.RRT_ERR_INVALID
    assert status(lambda: a.update_mesh(mesh + 1, p1)) == capi.RRT_ERR_INVALID                  # unknown mesh
    assert status(lambda: a.update_mesh(mesh, p1, first_vertex=1)) == capi.RRT_ERR_INVALID      # past the end
    assert status(lambda: a.update_mesh_device(mesh, 1, nv, d.data_ptr())) == capi.RRT_ERR_INVALID
    assert status(lambda: a.update_mesh(mesh, p1[:3], normals=np.ones((3, 3)))) == capi.RRT_ERR_INVALID  # no normals
    assert a.update_mesh(mesh, np.zeros((0, 3))) is a                                          # zero counts
    assert L.rrt_scene_update_mesh_device(a.h, mesh, 0, 0, None, 0, 0, None, None) == capi.RRT_OK
    assert a.intersect(rays).tobytes() == before.tobytes() and (a.export_tree() == blob).all()
    assert not a.build_info()["device_lbvh"]                                                     # nothing rebuilt
    # normals: range past the end
    g = _normal_mesh(0.1, 3, k=8)
    b, mb = _placed(ctx, g, capi.RRT_BUILD_FAST)
    assert status(lambda: b.update_mesh(mb, g["p"][:1], normals=g["n"], first_normal=1)) == capi.RRT_ERR_INVALID
    # uncommitted scene
    u = GpuAggregate(ctx)
    mu = u.add_mesh(p, idx)
    u.add_triangles(mu, 0)
    assert status(lambda: u.update_mesh(mu, p1)) == capi.RRT_ERR_INVALID
    # the literal tier
    m, inv = scenes.cube_instances(50, extent=8.0)
    lit = scenes.gpu_cubes(ctx, m, inv, build_flags=capi.RRT_BUILD_LITERAL)
    assert status(lambda: lit.update_mesh(0, synth.CUBE_P)) == capi.RRT_ERR_UNSUPPORTED
    # a live integrator blocks the update; destroying it unblocks
    desc = synth.default_render_desc(16, 16, 1, cam_pos=(0.5, 0.5, -2.5), cam_look=(0.5, 0.5, 0.5), focus_distance=3.0)
    r = Render.create(a, [R.matte()], [R.point_light()], desc, synth.DGAUSS_LENS)
    assert status(lambda: a.update_mesh(mesh, p1)) == capi.RRT_ERR_INVALID
    assert status(lambda: a.update_mesh_device(mesh, 0, nv, d.data_ptr())) == capi.RRT_ERR_INVALID
    assert a.intersect(rays).tobytes() == before.tobytes() and (a.export_tree() == blob).all()
    r.close()
    a.update_mesh_device(mesh, 0, nv, d.data_ptr())
    h, _ = _soup_scene(ctx, p1, idx, LBVH)
    _same_answers(a, h, synth.bounce_rays(p1, idx, 50000, seed=2))
