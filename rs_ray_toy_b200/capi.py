"""ctypes binding of librrt_sm100.so (include/rrt.h).

This is the only way Python reaches the CUDA core; there is no CPU path.  Loading fails
loudly when the library is missing, and `Context()` fails loudly when there is no sm_100 GPU.
"""
from __future__ import annotations

import ctypes as C
import re
from pathlib import Path

PKG = Path(__file__).resolve().parent
import os
# RRT_LIB selects an experiment build of the same library (tools/sweep.py); default = the product
LIB_PATH = Path(os.environ["RRT_LIB"]) if os.environ.get("RRT_LIB") else PKG / "librrt_sm100.so"
HEADER = PKG.parent / "include" / "rrt.h"
TEST_HEADER = PKG.parent / "include" / "rrt_test.h"   # host-only probes for the CPU tests, not for bindings

RRT_OK = 0
RRT_ERR_INVALID = -1
RRT_ERR_CUDA = -2
RRT_ERR_UNSUPPORTED = -3
RRT_ERR_EMPTY = -4
RRT_ERR_IO = -5
RRT_NO_HIT = 0xFFFFFFFF
RRT_BUILD_FAST = 0
RRT_BUILD_LITERAL = 1
RRT_BUILD_DEVICE_LBVH = 2


class RrtError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"rrt status {status}: {message}")
        self.status = status


_lib = None


def declared_symbols() -> list[str]:
    """Every function name include/rrt.h and include/rrt_test.h declare (used by the export test)."""
    text = HEADER.read_text() + TEST_HEADER.read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(rrt_[a-z0-9_]+)\s*\(", text)))


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise RrtError(RRT_ERR_INVALID,
                       f"{LIB_PATH} is missing: build it with `python -m rs_ray_toy_b200.build` "
                       "(there is no CPU fallback)")
    L = C.CDLL(str(LIB_PATH))
    vp, u32, i32, u64, dbl, sz = C.c_void_p, C.c_uint32, C.c_int, C.c_uint64, C.c_double, C.c_size_t
    pvp = C.POINTER(C.c_void_p)
    sig = {
        "rrt_create": (i32, [i32, pvp]),
        "rrt_destroy": (None, [vp]),
        "rrt_last_error": (C.c_char_p, []),
        "rrt_launch_count": (u64, [vp]),
        "rrt_host_alloc": (i32, [vp, sz, pvp]),
        "rrt_host_free": (i32, [vp, vp]),
        "rrt_scene_begin": (i32, [vp, pvp]),
        "rrt_scene_destroy": (None, [vp]),
        "rrt_scene_add_mesh": (i32, [vp, u32, vp, u32, vp, u32, vp, vp, u32, vp, vp, C.POINTER(u32)]),
        "rrt_scene_add_triangles": (i32, [vp, u32, u32, u32, vp, vp]),
        "rrt_scene_add_sphere": (i32, [vp, vp, vp, dbl, dbl, dbl, dbl, u32, u32, vp, vp]),
        "rrt_scene_commit": (i32, [vp, u32, u32]),
        "rrt_scene_num_prims": (i32, [vp, C.POINTER(u32)]),
        "rrt_world_bound": (i32, [vp, vp]),
        "rrt_scene_stats": (i32, [vp, vp]),
        "rrt_scene_build_info": (i32, [vp, vp]),
        "rrt_lbvh_host_probe": (i32, [u32, vp, u32, u32, C.POINTER(u32), vp, vp, vp]),
        "rrt_intersect_device": (i32, [vp, u64, vp, vp, vp]),
        "rrt_intersect_p_device": (i32, [vp, u64, vp, vp, vp]),
        "rrt_intersect": (i32, [vp, u64, vp, vp]),
        "rrt_intersect_p": (i32, [vp, u64, vp, vp]),
        "rrt_intersect_f32_device": (i32, [vp, u64, vp, vp, vp]),
        "rrt_intersect_p_f32_device": (i32, [vp, u64, vp, vp, vp]),
        "rrt_intersect_f32": (i32, [vp, u64, vp, vp]),
        "rrt_intersect_p_f32": (i32, [vp, u64, vp, vp]),
        "rrt_intersect_surface_device": (i32, [vp, u64, vp, vp, vp]),
        "rrt_intersect_surface": (i32, [vp, u64, vp, vp]),
        "rrt_rays_f32_host_probe": (i32, [u64, vp, vp, u64, vp, vp]),
        "rrt_scene_update_instances": (i32, [vp, u32, u32, vp, vp]),
        "rrt_scene_update_mesh": (i32, [vp, u32, u32, u32, vp, u32, u32, vp]),
        "rrt_scene_update_mesh_device": (i32, [vp, u32, u32, u32, vp, u32, u32, vp, vp]),
        "rrt_scene_export_tree": (i32, [vp, vp, u64, C.POINTER(u64)]),
        "rrt_scene_commit_from_tree": (i32, [vp, vp, u64]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def check(status: int):
    if status != RRT_OK:
        raise RrtError(status, lib().rrt_last_error().decode(errors="replace"))
