"""Host-side mirror of the reference's aggregate seam over the C ABI (include/rrt.h).

`GpuAggregate` stands where `BVHAccel` stands behind `Scene.aggregate: Arc<dyn Primitive>`
(src/scene.rs:17, src/bvh.rs:116-121): it is assembled like `make_aggregate`
(src/renderprocess.rs:1178-1304) assembles the primitive list, committed like
`BVHAccel::new(prims, max_prims_in_node, split)` (src/bvh.rs:307-311), and answers
`intersect` / `intersect_p` / `world_bound` (src/primitives.rs:14-17, src/geometry.rs:94-96)
for whole batches of rays.  Every call goes to librrt_sm100.so; nothing is computed here.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import capi

RAY_DTYPE = np.dtype([("o", "<f8", 3), ("d", "<f8", 3), ("t_max", "<f8"), ("time", "<f8")])  # rrt_ray, 64 B
HIT_DTYPE = np.dtype([("prim_id", "<u4"), ("reserved", "<u4"), ("t", "<f8"), ("u", "<f8"), ("v", "<f8")])  # rrt_hit, 32 B
assert RAY_DTYPE.itemsize == 64 and HIT_DTYPE.itemsize == 32
# rrt_ray_f32 (32 B) / rrt_hit_f32 (16 B): fp32 rays promoted exactly to f64 on the device, hits rounded to nearest
RAY_F32_DTYPE = np.dtype([("o", "<f4", 3), ("t_max", "<f4"), ("d", "<f4", 3), ("reserved", "<u4")])
HIT_F32_DTYPE = np.dtype([("prim_id", "<u4"), ("t", "<f4"), ("u", "<f4"), ("v", "<f4")])
assert RAY_F32_DTYPE.itemsize == 32 and HIT_F32_DTYPE.itemsize == 16


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def pack_rays(rays) -> np.ndarray:
    """[n,7] (o, d, t_max) or [n,8] (…, time) f64 -> rrt_ray records (geometry.rs:73-79)."""
    if isinstance(rays, np.ndarray) and rays.dtype == RAY_DTYPE:
        return np.ascontiguousarray(rays)
    a = np.asarray(rays, dtype=np.float64)
    if a.ndim != 2 or a.shape[1] not in (7, 8):
        raise ValueError("rays must be [n,7] (o,d,t_max) or [n,8] (o,d,t_max,time)")
    out = np.zeros((a.shape[0], 8), dtype=np.float64)
    out[:, : a.shape[1]] = a
    return out.view(RAY_DTYPE).reshape(-1)


def pack_rays_f32(rays, out=None) -> np.ndarray:
    """[n,7] float32 (o, d, t_max) -> rrt_ray_f32 records, into `out` when given (e.g. a `Context.pinned_empty` array).
    f64 input is refused rather than rounded: what the fp32 entries answer for is the fp32 ray."""
    if isinstance(rays, np.ndarray) and rays.dtype == RAY_F32_DTYPE:
        if out is None:
            return np.ascontiguousarray(rays)
        out[:] = rays
        return out
    a = np.asarray(rays)
    if a.dtype != np.float32:
        raise TypeError(f"fp32 rays must be float32, got {a.dtype} (round them with .astype(np.float32) if that is meant)")
    if a.ndim != 2 or a.shape[1] != 7:
        raise ValueError("fp32 rays must be [n,7] (o, d, t_max)")
    r = np.empty(a.shape[0], dtype=RAY_F32_DTYPE) if out is None else out
    if r.shape != (a.shape[0],) or r.dtype != RAY_F32_DTYPE:
        raise ValueError("out must be an rrt_ray_f32 array of the batch's length")
    r["o"] = a[:, 0:3]
    r["d"] = a[:, 3:6]
    r["t_max"] = a[:, 6]
    r["reserved"] = 0
    return r


def promote_rays_f32(rays) -> np.ndarray:
    """The rrt_ray records an fp32 batch stands for (exact promotion, time = 0): the f64 call with these answers what
    the fp32 call answers, before rounding."""
    r = pack_rays_f32(rays)
    out = np.zeros(r.shape[0], dtype=RAY_DTYPE)
    out["o"] = r["o"]
    out["d"] = r["d"]
    out["t_max"] = r["t_max"]
    return out


class Context:
    """One CUDA device (rrt_ctx)."""

    def __init__(self, device: int = 0):
        self.L = capi.lib()
        h = C.c_void_p()
        capi.check(self.L.rrt_create(int(device), C.byref(h)))
        self.h = h
        self.device = int(device)

    def close(self):
        if getattr(self, "h", None):
            self.L.rrt_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def launch_count(self) -> int:
        return int(self.L.rrt_launch_count(self.h))

    def pinned_empty(self, n: int, dtype) -> np.ndarray:
        """A page-locked host array (cudaHostAlloc) for ray / hit batches."""
        dtype = np.dtype(dtype)
        nbytes = max(1, int(n) * dtype.itemsize)
        p = C.c_void_p()
        capi.check(self.L.rrt_host_alloc(self.h, nbytes, C.byref(p)))
        buf = (C.c_char * nbytes).from_address(p.value)
        arr = np.frombuffer(buf, dtype=dtype, count=int(n))
        self._pinned = getattr(self, "_pinned", [])
        self._pinned.append(p)
        return arr


class GpuAggregate:
    """The GPU stand-in for `BVHAccel` (src/bvh.rs:116-121)."""

    def __init__(self, ctx: Context):
        self.ctx = ctx
        self.L = ctx.L
        h = C.c_void_p()
        capi.check(self.L.rrt_scene_begin(ctx.h, C.byref(h)))
        self.h = h
        self.committed = False

    def close(self):
        if getattr(self, "h", None):
            self.L.rrt_scene_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- make_aggregate (renderprocess.rs:1178-1304) -------------------------------------
    def add_mesh(self, p, vi, n=None, ni=None, uv=None, uvi=None) -> int:
        """`create_triangle_mesh` (shape/triangle.rs:131-165); indices are 0-based."""
        p = np.ascontiguousarray(p, dtype=np.float64).reshape(-1, 3)
        vi = np.ascontiguousarray(vi, dtype=np.uint32).reshape(-1, 3)
        n = None if n is None else np.ascontiguousarray(n, dtype=np.float64).reshape(-1, 3)
        ni = None if ni is None else np.ascontiguousarray(ni, dtype=np.uint32).reshape(-1, 3)
        uv = None if uv is None else np.ascontiguousarray(uv, dtype=np.float64).reshape(-1, 2)
        uvi = None if uvi is None else np.ascontiguousarray(uvi, dtype=np.uint32).reshape(-1, 3)
        mesh = C.c_uint32()
        capi.check(self.L.rrt_scene_add_mesh(self.h, p.shape[0], _ptr(p), vi.shape[0], _ptr(vi),
                                             0 if n is None else n.shape[0], _ptr(n), _ptr(ni),
                                             0 if uv is None else uv.shape[0], _ptr(uv), _ptr(uvi), C.byref(mesh)))
        return mesh.value

    @staticmethod
    def _instances(instances):
        if instances is None:
            return 0, None, None
        m, inv = instances
        m = np.ascontiguousarray(m, dtype=np.float64).reshape(-1, 16)
        inv = np.ascontiguousarray(inv, dtype=np.float64).reshape(-1, 16)
        if m.shape != inv.shape:
            raise ValueError("instance matrices and inverses differ in shape")
        return m.shape[0], m, inv

    def add_triangles(self, mesh: int, material: int = 0, instances=None):
        """One GeometricPrimitive per triangle, bare or once per instance (renderprocess.rs:1228-1282)."""
        k, m, inv = self._instances(instances)
        capi.check(self.L.rrt_scene_add_triangles(self.h, mesh, material, k, _ptr(m), _ptr(inv)))

    def add_sphere(self, radius=1.0, z_min=None, z_max=None, phi_max=360.0, obj_to_world=None, material: int = 0,
                   instances=None):
        """`Sphere::new` + GeometricPrimitive (+ instances) (renderprocess.rs:1187-1227)."""
        z_min = -radius if z_min is None else z_min
        z_max = radius if z_max is None else z_max
        om = oi = None
        if obj_to_world is not None:
            om = np.ascontiguousarray(obj_to_world[0], dtype=np.float64).reshape(16)
            oi = np.ascontiguousarray(obj_to_world[1], dtype=np.float64).reshape(16)
        k, m, inv = self._instances(instances)
        capi.check(self.L.rrt_scene_add_sphere(self.h, _ptr(om), _ptr(oi), radius, z_min, z_max, phi_max, material, k,
                                               _ptr(m), _ptr(inv)))

    def commit(self, max_prims_in_node: int = 4, build_flags: int = capi.RRT_BUILD_FAST):
        """`BVHAccel::new(prims, max_prims_in_node, split_method)` (bvh.rs:307-363)."""
        capi.check(self.L.rrt_scene_commit(self.h, max_prims_in_node, build_flags))
        self.committed = True
        return self

    def update_instances(self, first: int, m: np.ndarray, inv: np.ndarray):
        """rrt_scene_update_instances: new transforms for instances [first, first + len(m)), tree made anew on the device."""
        m = np.ascontiguousarray(m, dtype=np.float64).reshape(-1, 16)
        inv = np.ascontiguousarray(inv, dtype=np.float64).reshape(-1, 16)
        capi.check(self.L.rrt_scene_update_instances(self.h, first, m.shape[0], _ptr(m), _ptr(inv)))
        return self

    def export_tree(self) -> np.ndarray:
        """rrt_scene_export_tree: the committed aggregate (tree + records + tables) as one uint8 blob."""
        n = C.c_uint64()
        capi.check(self.L.rrt_scene_export_tree(self.h, None, 0, C.byref(n)))
        blob = np.empty(n.value, dtype=np.uint8)
        capi.check(self.L.rrt_scene_export_tree(self.h, blob.ctypes.data, blob.size, C.byref(n)))
        return blob

    def commit_from_tree(self, blob: np.ndarray):
        """rrt_scene_commit_from_tree: commit with a tree another rank built over the same primitives."""
        b = np.ascontiguousarray(blob, dtype=np.uint8)
        capi.check(self.L.rrt_scene_commit_from_tree(self.h, b.ctypes.data, b.size))
        self.committed = True
        return self

    @property
    def num_prims(self) -> int:
        n = C.c_uint32()
        capi.check(self.L.rrt_scene_num_prims(self.h, C.byref(n)))
        return n.value

    def world_bound(self) -> np.ndarray:
        """`Primitive::world_bound` (bvh.rs:177-182) -> [p_min, p_max]."""
        out = np.zeros(6)
        capi.check(self.L.rrt_world_bound(self.h, _ptr(out)))
        return out

    def stats(self) -> dict:
        out = np.zeros(8, dtype=np.uint64)
        capi.check(self.L.rrt_scene_stats(self.h, _ptr(out)))
        keys = ["n_nodes", "n_leaves", "max_depth", "device_bytes", "build_usec", "n_records", "wide_records", "n_prims"]
        return {k: int(v) for k, v in zip(keys, out)}

    def build_info(self) -> dict:
        """How the tree was built (rrt_scene_build_info)."""
        out = np.zeros(4, dtype=np.uint64)
        capi.check(self.L.rrt_scene_build_info(self.h, _ptr(out)))
        return {"tree_device_usec": int(out[0]), "node_bytes": int(out[1]), "device_lbvh": bool(out[2])}

    # ---- Primitive / IntersectP over batches, HOST buffers ----------------------------------
    def intersect(self, rays, out=None) -> np.ndarray:
        """`Scene::intersect` (scene.rs:69-72) for a batch: returns rrt_hit records."""
        r = pack_rays(rays)
        hits = np.empty(r.shape[0], dtype=HIT_DTYPE) if out is None else out
        capi.check(self.L.rrt_intersect(self.h, r.shape[0], _ptr(r), _ptr(hits)))
        return hits

    def intersect_p(self, rays, out=None) -> np.ndarray:
        """`Scene::intersect_p` (scene.rs:75-80) for a batch: returns 0/1 bytes."""
        r = pack_rays(rays)
        occ = np.empty(r.shape[0], dtype=np.uint8) if out is None else out
        capi.check(self.L.rrt_intersect_p(self.h, r.shape[0], _ptr(r), _ptr(occ)))
        return occ

    # ---- the same over fp32 rays (rrt_ray_f32) and compact hits (rrt_hit_f32), HOST buffers ------------------
    # For the link's full rate pass records in page-locked memory: rays packed with pack_rays_f32(a, out=...) and `out`,
    # both from Context.pinned_empty (pageable buffers work, through a staging copy of the driver's).
    def intersect_f32(self, rays, out=None) -> np.ndarray:
        """`Scene::intersect` for an fp32 batch: [n,7] float32 or rrt_ray_f32 records in, HIT_F32_DTYPE records out."""
        r = pack_rays_f32(rays)
        hits = np.empty(r.shape[0], dtype=HIT_F32_DTYPE) if out is None else out
        capi.check(self.L.rrt_intersect_f32(self.h, r.shape[0], _ptr(r), _ptr(hits)))
        return hits

    def intersect_p_f32(self, rays, out=None) -> np.ndarray:
        """`Scene::intersect_p` for an fp32 batch: returns 0/1 bytes."""
        r = pack_rays_f32(rays)
        occ = np.empty(r.shape[0], dtype=np.uint8) if out is None else out
        capi.check(self.L.rrt_intersect_p_f32(self.h, r.shape[0], _ptr(r), _ptr(occ)))
        return occ

    # ---- same, DEVICE buffers (raw pointers; torch tensors' data_ptr()) ---------------------
    def intersect_device(self, n: int, d_rays: int, d_hits: int, stream: int = 0):
        capi.check(self.L.rrt_intersect_device(self.h, n, C.c_void_p(d_rays), C.c_void_p(d_hits), C.c_void_p(stream)))

    def intersect_p_device(self, n: int, d_rays: int, d_occluded: int, stream: int = 0):
        capi.check(self.L.rrt_intersect_p_device(self.h, n, C.c_void_p(d_rays), C.c_void_p(d_occluded),
                                                 C.c_void_p(stream)))

    def intersect_f32_device(self, n: int, d_rays: int, d_hits: int, stream: int = 0):
        """rrt_intersect_f32_device: n rrt_ray_f32 (32 B each) -> n rrt_hit_f32 (16 B each), 16-byte aligned device
        buffers, asynchronous on `stream`."""
        capi.check(self.L.rrt_intersect_f32_device(self.h, n, C.c_void_p(d_rays), C.c_void_p(d_hits), C.c_void_p(stream)))

    def intersect_p_f32_device(self, n: int, d_rays: int, d_occluded: int, stream: int = 0):
        capi.check(self.L.rrt_intersect_p_f32_device(self.h, n, C.c_void_p(d_rays), C.c_void_p(d_occluded),
                                                     C.c_void_p(stream)))


def lbvh_host_probe(bounds6: np.ndarray, max_prims_in_node: int = 4):
    """rrt_lbvh_host_probe: the device LBVH builder's per-element code run on the host (CPU tests).
    Returns (nodes as [n_nodes, 16] uint32 words of Node64, order, info {nodes, max_depth, leaves})."""
    L = capi.lib()
    b = np.ascontiguousarray(bounds6, dtype=np.float64).reshape(-1, 6)
    n = b.shape[0]
    words = np.zeros((max(n, 1), 16), dtype=np.uint32)
    order = np.zeros(n, dtype=np.uint32)
    info = np.zeros(3, dtype=np.uint32)
    cnt = C.c_uint32()
    capi.check(L.rrt_lbvh_host_probe(n, _ptr(b), max_prims_in_node, words.shape[0], C.byref(cnt), _ptr(words), _ptr(order), _ptr(info)))
    return words[: cnt.value], order, {"nodes": int(info[0]), "max_depth": int(info[1]), "leaves": int(info[2])}


def rays_f32_host_probe(rays, hits):
    """rrt_rays_f32_host_probe: the library's fp32 format conversions run on the host (CPU tests).
    rays: RAY_F32_DTYPE records -> RAY_DTYPE as the walk sees them; hits: HIT_DTYPE -> HIT_F32_DTYPE."""
    L = capi.lib()
    r = np.ascontiguousarray(rays, dtype=RAY_F32_DTYPE)
    h = np.ascontiguousarray(hits, dtype=HIT_DTYPE)
    promoted = np.zeros(r.shape[0], dtype=RAY_DTYPE)
    compact = np.zeros(h.shape[0], dtype=HIT_F32_DTYPE)
    capi.check(L.rrt_rays_f32_host_probe(r.shape[0], _ptr(r), _ptr(promoted), h.shape[0], _ptr(h), _ptr(compact)))
    return promoted, compact


def soup_aggregate(ctx: Context, p, idx, max_prims_in_node: int = 4, build_flags: int = capi.RRT_BUILD_FAST) -> GpuAggregate:
    """A bare (non-instanced) triangle mesh as one aggregate — configs 3 and 5."""
    agg = GpuAggregate(ctx)
    mesh = agg.add_mesh(p, idx)
    agg.add_triangles(mesh, 0)
    return agg.commit(max_prims_in_node, build_flags)
