"""ctypes wrapper of tests/cpp/surface_oracle.cpp: the CPU oracle's scenes with every SurfaceInteraction field of a hit.

TEST INFRASTRUCTURE: tests/test_gpu_surface.py checks rrt_intersect_surface against it.  The library is compiled on
first use from that file and the oracle's shape and BVH sources, with the oracle's flags, into the temporary directory
(keyed by the sources' contents, so a changed source gets a library of its own)."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import shutil
import subprocess
import tempfile
from pathlib import Path

import numpy as np

import oracle_lib as O

ROOT = Path(__file__).resolve().parent.parent
SOURCES = [ROOT / "tests" / "cpp" / "surface_oracle.cpp"] + [ROOT / "oracle" / f for f in ("rt_geom.cpp", "rt_shapes.cpp",
                                                                                            "rt_bvh.cpp")]
# oracle/Makefile's flags: no contraction, no fast math (Rust/LLVM never fuses a*b+c for f64)
CXXFLAGS = ["-O3", "-march=x86-64-v3", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-pthread", "-shared"]

_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    h = hashlib.sha1(" ".join(CXXFLAGS).encode())
    for p in SOURCES + sorted((ROOT / "oracle").glob("*.hpp")):
        h.update(p.read_bytes())
    path = Path(tempfile.gettempdir()) / f"rrt_surface_oracle_{os.getuid()}_{h.hexdigest()[:12]}.so"
    if not path.exists():
        gxx = shutil.which("g++") or "/opt/gcc/bin/g++"
        tmp = path.with_suffix(f".tmp{os.getpid()}")
        subprocess.run([gxx, *CXXFLAGS, "-I", str(ROOT / "oracle"), "-o", str(tmp), *map(str, SOURCES)], check=True,
                       capture_output=True)
        os.replace(tmp, path)
    L = C.CDLL(str(path))
    vp, u32, i32, u64, dbl = C.c_void_p, C.c_uint32, C.c_int32, C.c_uint64, C.c_double
    L.sor_last_error.restype = C.c_char_p
    L.sor_scene_new.restype = vp
    L.sor_scene_new.argtypes = [u32]
    L.sor_scene_free.argtypes = [vp]
    L.sor_add_mesh.restype = i32
    L.sor_add_mesh.argtypes = [vp, u32, vp, u32, vp, u32, vp, vp, u32, vp, vp]
    L.sor_add_sphere.restype = i32
    L.sor_add_sphere.argtypes = [vp, vp, vp, dbl, dbl, dbl, dbl]
    L.sor_add_geo_triangles.restype = i32
    L.sor_add_geo_triangles.argtypes = [vp, i32]
    L.sor_add_geo_sphere.restype = i32
    L.sor_add_geo_sphere.argtypes = [vp, i32]
    L.sor_add_xform.restype = i32
    L.sor_add_xform.argtypes = [vp, vp, vp]
    L.sor_add_prims.argtypes = [vp, i32, i32, i32]
    L.sor_build.restype = i32
    L.sor_build.argtypes = [vp, u32]
    L.sor_intersect_si.restype = i32
    L.sor_intersect_si.argtypes = [vp, u64, vp, vp, vp, vp, vp, i32]
    _lib = L
    return L


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _f64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a if shape is None else a.reshape(shape)


class SurfaceOracle:
    """What `make_aggregate` assembles (as oracle_lib.OracleScene), answering with whole SurfaceInteractions."""

    def __init__(self, tier: int = O.TIER_F):
        self.L = lib()
        self.h = self.L.sor_scene_new(tier)
        self._keep = []

    def __del__(self):
        try:
            if self.h:
                self.L.sor_scene_free(self.h)
                self.h = None
        except Exception:
            pass

    def add_mesh(self, p, vi, n=None, ni=None, uv=None, uvi=None) -> int:
        p, vi = _f64(p), np.ascontiguousarray(vi, dtype=np.uint32)
        n = None if n is None else _f64(n)
        ni = None if ni is None else np.ascontiguousarray(ni, dtype=np.uint32)
        uv = None if uv is None else _f64(uv)
        uvi = None if uvi is None else np.ascontiguousarray(uvi, dtype=np.uint32)
        return self.L.sor_add_mesh(self.h, p.shape[0], _ptr(p), vi.shape[0], _ptr(vi), 0 if n is None else n.shape[0],
                                   _ptr(n), _ptr(ni), 0 if uv is None else uv.shape[0], _ptr(uv), _ptr(uvi))

    def add_sphere(self, m=None, inv=None, radius=1.0, z_min=None, z_max=None, phi_max=360.0) -> int:
        m = _f64(np.eye(4) if m is None else m, 16)
        inv = _f64(np.eye(4) if inv is None else inv, 16)
        z_min = -radius if z_min is None else z_min
        z_max = radius if z_max is None else z_max
        return self.L.sor_add_sphere(self.h, _ptr(m), _ptr(inv), radius, z_min, z_max, phi_max)

    def add_geo_triangles(self, mesh: int) -> int:
        return self.L.sor_add_geo_triangles(self.h, mesh)

    def add_geo_sphere(self, sphere: int) -> int:
        return self.L.sor_add_geo_sphere(self.h, sphere)

    def add_xform(self, m, inv) -> int:
        m, inv = _f64(m, 16), _f64(inv, 16)
        return self.L.sor_add_xform(self.h, _ptr(m), _ptr(inv))

    def add_prims(self, first_geo: int, count: int, xf: int = -1):
        self.L.sor_add_prims(self.h, first_geo, count, xf)

    def build(self, max_prims_in_node: int = 4):
        if self.L.sor_build(self.h, max_prims_in_node) != 0:
            raise RuntimeError(self.L.sor_last_error().decode())
        return self

    def intersect_si(self, rays, nthreads=None):
        """{"prim", "t", "uv", "si"}: si is [n, 38] in rrt_surface's order after its hit (zeros for a miss)."""
        rays = _f64(rays)
        n = rays.shape[0]
        prim = np.empty(n, dtype=np.int32)
        t = np.empty(n)
        uv = np.empty((n, 2))
        si = np.empty((n, 38))
        nthreads = O.hardware_threads() if nthreads is None else nthreads
        if self.L.sor_intersect_si(self.h, n, _ptr(rays), _ptr(prim), _ptr(t), _ptr(uv), _ptr(si), nthreads) != 0:
            raise RuntimeError(self.L.sor_last_error().decode())
        return {"prim": prim, "t": t, "uv": uv, "si": si}


# the scenes of tests/scenes.py, on this oracle
def soup(p, idx, tier=O.TIER_F, max_prims=4):
    s = SurfaceOracle(tier)
    s.add_prims(s.add_geo_triangles(s.add_mesh(p, idx)), idx.shape[0], -1)
    return s.build(max_prims)


def cubes(m, inv, tier=O.TIER_F, max_prims=4):
    from rs_ray_toy_b200 import synth
    s = SurfaceOracle(tier)
    g0 = s.add_geo_triangles(s.add_mesh(synth.CUBE_P, synth.CUBE_VI, synth.CUBE_N, synth.CUBE_NI))
    for i in range(m.shape[0]):
        s.add_prims(g0, 12, s.add_xform(m[i], inv[i]))
    return s.build(max_prims)


def spheres(m, inv, radius=0.5, tier=O.TIER_F, max_prims=4):
    s = SurfaceOracle(tier)
    g = s.add_geo_sphere(s.add_sphere(None, None, radius))
    for i in range(m.shape[0]):
        s.add_prims(g, 1, s.add_xform(m[i], inv[i]))
    return s.build(max_prims)
