"""CPU checks of the surface records (rrt_surface, include/rrt.h): the numpy dtype and the Rust binding have the C
layout, and the library exports both surface entries.  The records' values are checked on the GPU (test_gpu_surface.py)."""
import re
import subprocess
from pathlib import Path

from rs_ray_toy_b200 import capi
from rs_ray_toy_b200.aggregate import HIT_DTYPE, SURFACE_DTYPE
from rs_ray_toy_b200.build import build_library

ROOT = Path(__file__).resolve().parent.parent
FIELDS = ["hit", "p", "wo", "n", "uv", "dpdu", "dpdv", "dndu", "dndv", "sh_n", "sh_dpdu", "sh_dpdv", "sh_dndu", "sh_dndv"]


def test_dtype_matches_the_c_layout(tmp_path):
    src = tmp_path / "surface.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "rrt.h"\nint main(void) {\n'
                   '  printf("sizeof %zu\\n", sizeof(rrt_surface));\n' +
                   "".join(f'  printf("{f} %zu %zu\\n", offsetof(rrt_surface, {f}), sizeof(((rrt_surface*)0)->{f}));\n'
                           for f in FIELDS) + "  return 0;\n}\n")
    exe = tmp_path / "surface"
    r = subprocess.run(["gcc", "-I", str(ROOT / "include"), "-o", str(exe), str(src)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    out = [line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True).stdout.splitlines()]
    assert out[0] == ["sizeof", "336"] and SURFACE_DTYPE.itemsize == 336
    assert list(SURFACE_DTYPE.names) == FIELDS
    for name, off, size in out[1:]:
        dt, o = SURFACE_DTYPE.fields[name][:2]
        assert (o, dt.itemsize) == (int(off), int(size)), name
    assert SURFACE_DTYPE.fields["hit"][0] == HIT_DTYPE


def test_rust_struct_lists_the_same_fields():
    rs = (ROOT / "rust" / "rrt-sys" / "src" / "lib.rs").read_text()
    body = re.search(r"pub struct rrt_surface \{(.*?)\}", rs, flags=re.S).group(1)
    fields = re.findall(r"pub (\w+): (\[f64; (\d)\]|rrt_hit)", body)
    assert [f[0] for f in fields] == FIELDS
    for name, ty, k in fields:
        if name == "hit":
            assert ty == "rrt_hit"
        else:
            assert int(k) == SURFACE_DTYPE.fields[name][0].shape[0], name
    assert re.search(r"pub fn rrt_intersect_surface\(scene: \*const rrt_scene, n: u64, rays: \*const rrt_ray, "
                     r"surfaces: \*mut rrt_surface\) -> c_int;", rs)
    assert re.search(r"pub fn rrt_intersect_surface_device\(scene: \*const rrt_scene, n: u64, d_rays: \*const rrt_ray, "
                     r"d_surfaces: \*mut rrt_surface, cuda_stream: \*mut c_void\) -> c_int;", rs)


def test_surface_entries_are_exported():
    build_library()
    L = capi.lib()
    for name in ("rrt_intersect_surface", "rrt_intersect_surface_device"):
        assert name in capi.declared_symbols() and hasattr(L, name)


def test_surface_oracle_agrees_with_the_oracle():
    """tests/surface_oracle.py assembles its scenes as oracle_lib does: the same hits, and the hit point, geometric and
    shading normals orc_intersect reports, bit for bit, on instanced meshes with normals and on clipped spheres."""
    import numpy as np

    import oracle_lib as O
    import surface_oracle as SO
    from rs_ray_toy_b200 import synth
    from rs_ray_toy_b200 import transform as T

    for tier in (O.TIER_F, O.TIER_L):
        a, b = O.OracleScene(tier), SO.SurfaceOracle(tier)
        for s in (a, b):
            g0 = s.add_geo_triangles(s.add_mesh(synth.CUBE_P, synth.CUBE_VI, synth.CUBE_N, synth.CUBE_NI))
            for k in range(20):
                m, inv = T.make_to_world((k % 5 * 3.0 - 6.0, k // 5 * 3.0 - 6.0, 0.0), (1.0, 0.5, 0.2), 17.0 * k)
                s.add_prims(g0, 12, s.add_xform(m, inv))
            if tier == O.TIER_F:
                m, inv = T.make_to_world((0.0, 0.0, 5.0), (0.0, 1.0, 0.0), 30.0)
                g = s.add_geo_sphere(s.add_sphere(None, None, 1.5, -0.8, 1.2, 250.0))
                s.add_prims(g, 1, s.add_xform(m, inv))
            s.build(4)
        rays = synth.camera_like_rays(20000, (0.5, -1.0, -30.0), 8.0, seed=9)
        ra, rb = a.intersect(rays, want_geom=True, nthreads=4), b.intersect_si(rays, nthreads=4)
        hit = ra["prim"] >= 0
        assert hit.sum() > 2000
        assert np.array_equal(ra["prim"], rb["prim"])
        assert np.array_equal(ra["t"][hit], rb["t"][hit]) and np.array_equal(ra["uv"][hit], rb["uv"][hit])
        geom = np.concatenate([rb["si"][:, 0:3], rb["si"][:, 6:9], rb["si"][:, 23:26]], axis=1)
        assert np.array_equal(ra["geom"][hit].view(np.uint64), geom[hit].view(np.uint64))
        assert not rb["si"][~hit].any()
