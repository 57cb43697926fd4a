"""CPU checks of the fp32 ray / hit records (rrt_ray_f32, rrt_hit_f32 in include/rrt.h): their C layout equals the
numpy dtypes and the Rust bindings, the four entry points are exported and bound, and the library's own conversions
(csrc/rays_f32.cuh, run on the host through rrt_rays_f32_host_probe) promote exactly and round like numpy."""
import re
import subprocess
from pathlib import Path

import numpy as np
import pytest

from rs_ray_toy_b200 import capi
from rs_ray_toy_b200.aggregate import (HIT_DTYPE, HIT_F32_DTYPE, RAY_F32_DTYPE, pack_rays_f32, promote_rays_f32,
                                       rays_f32_host_probe)
from rs_ray_toy_b200.build import build_library

ROOT = Path(capi.__file__).resolve().parent.parent
ENTRIES = ["rrt_intersect_f32", "rrt_intersect_p_f32", "rrt_intersect_f32_device", "rrt_intersect_p_f32_device"]


@pytest.fixture(scope="module")
def library():
    build_library()
    return capi.lib()


def test_c_layout_equals_the_numpy_dtypes(tmp_path):
    fields = {"rrt_ray_f32": (RAY_F32_DTYPE, ["o", "t_max", "d", "reserved"]),
              "rrt_hit_f32": (HIT_F32_DTYPE, ["prim_id", "t", "u", "v"])}
    src = tmp_path / "layout.c"
    body = "".join(f'  printf("{s} sizeof %zu\\n", sizeof({s}));\n' +
                   "".join(f'  printf("{s} {f} %zu\\n", offsetof({s}, {f}));\n' for f in names)
                   for s, (_, names) in fields.items())
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "rrt.h"\nint main(void) {\n' + body + "  return 0;\n}\n")
    exe = tmp_path / "layout"
    r = subprocess.run(["gcc", "-I", str(ROOT / "include"), "-o", str(exe), str(src)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = {}
    for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines():
        s, f, v = line.split()
        got[(s, f)] = int(v)
    assert got[("rrt_ray_f32", "sizeof")] == 32 == RAY_F32_DTYPE.itemsize
    assert got[("rrt_hit_f32", "sizeof")] == 16 == HIT_F32_DTYPE.itemsize
    for s, (dt, names) in fields.items():
        for f in names:
            assert got[(s, f)] == dt.fields[f][1], (s, f)


def test_entry_points_are_exported_and_bound_in_rust(library):
    rs = (ROOT / "rust" / "rrt-sys" / "src" / "lib.rs").read_text()
    bound = set(re.findall(r"pub fn (rrt_[a-z0-9_]+)\s*\(", rs))
    for name in ENTRIES:
        assert hasattr(library, name), name
        assert name in bound, name
        assert name in capi.declared_symbols(), name
    sizes = dict(re.findall(r"size_of::<(rrt_[a-z0-9_]+)>\(\) == (\d+)", rs))
    assert sizes["rrt_ray_f32"] == "32" and sizes["rrt_hit_f32"] == "16"


def test_promotion_is_exact():
    rng = np.random.default_rng(3)
    n = 4096
    bits = rng.integers(0, 2**32, (n, 7), dtype=np.uint64).astype(np.uint32)
    a = bits.view(np.float32)
    a[np.isnan(a)] = 1.5
    special = np.array([0.0, -0.0, np.inf, -np.inf, 1e-45, -1e-45, 1.1754942e-38, 1.17549435e-38,
                        3.4028235e38, -3.4028235e38, 1.0, np.float32(np.pi)], dtype=np.float32)
    a[: special.size, :] = special[:, None]
    r = pack_rays_f32(a)
    promoted, _ = rays_f32_host_probe(r, np.zeros(0, dtype=HIT_DTYPE))
    want = a.astype(np.float64)
    for got, w in ((promoted["o"], want[:, 0:3]), (promoted["d"], want[:, 3:6]), (promoted["t_max"], want[:, 6])):
        assert np.array_equal(got.view(np.uint64), np.ascontiguousarray(w).view(np.uint64))
    assert (promoted["time"] == 0.0).all()
    assert np.array_equal(promoted, promote_rays_f32(a))
    # and back: every promoted value rounds to the float it came from
    assert np.array_equal(promoted["o"].astype(np.float32).view(np.uint32), a[:, 0:3].view(np.uint32))


def _rounding_cases():
    rng = np.random.default_rng(11)
    f = rng.uniform(-1e6, 1e6, 2000).astype(np.float32)
    nxt = np.nextafter(f, np.float32(np.inf))
    ties = (f.astype(np.float64) + nxt.astype(np.float64)) / 2           # exactly half way: to even
    sub = (rng.integers(1, 1 << 23, 2000).astype(np.uint32)).view(np.float32)
    sub_nxt = np.nextafter(sub, np.float32(np.inf))
    sub_ties = (sub.astype(np.float64) + sub_nxt.astype(np.float64)) / 2  # ties among subnormals
    tiny = 2.0 ** -149
    edges = np.array([0.0, -0.0, np.inf, -np.inf, tiny, tiny / 2, tiny / 2 * (1 + 2**-40), -tiny / 2, tiny * 1.5,
                      tiny * 2.5, 2.0 ** -126 * (1 - 2**-25), float(np.finfo(np.float32).max),
                      float(np.finfo(np.float32).max) * (1 + 2**-25), float(np.finfo(np.float32).max) * (1 + 2**-24),
                      1e300, -1e300, 1e-300, 1.0 + 2**-24, 1.0 + 3 * 2**-24, 1.0 - 2**-25, np.pi, 0.1])
    plain = rng.standard_normal(2000) * 10.0 ** rng.integers(-40, 39, 2000)
    return np.concatenate([ties, sub_ties, sub.astype(np.float64) * (1 + 2**-30), edges, plain])


def test_hit_rounding_equals_numpy_astype_float32():
    v = _rounding_cases()
    n = v.size
    hits = np.zeros(n, dtype=HIT_DTYPE)
    hits["prim_id"] = np.arange(n, dtype=np.uint32)
    hits["reserved"] = 0xDEADBEEF
    hits["t"] = v
    hits["u"] = v[::-1]
    hits["v"] = np.roll(v, 7)
    _, compact = rays_f32_host_probe(np.zeros(0, dtype=RAY_F32_DTYPE), hits)
    assert np.array_equal(compact["prim_id"], hits["prim_id"])
    for f in ("t", "u", "v"):
        with np.errstate(over="ignore"):
            want = hits[f].astype(np.float32)
        assert np.array_equal(compact[f].view(np.uint32), want.view(np.uint32)), f


def test_miss_record_keeps_its_id_and_rounds_its_fields():
    hits = np.zeros(3, dtype=HIT_DTYPE)
    hits["prim_id"] = capi.RRT_NO_HIT
    hits["t"] = [np.inf, 1e300, 0.1]
    hits["u"] = [0.0, -0.0, 1e-320]
    hits["v"] = [np.nan, 0.5, -np.inf]
    _, c = rays_f32_host_probe(np.zeros(0, dtype=RAY_F32_DTYPE), hits)
    assert (c["prim_id"] == capi.RRT_NO_HIT).all()
    assert c["t"][0] == np.inf and c["t"][1] == np.inf and c["t"][2] == np.float32(0.1)
    assert c["u"].view(np.uint32).tolist() == [0, 0x80000000, 0]
    assert np.isnan(c["v"][0]) and c["v"][1] == 0.5 and c["v"][2] == -np.inf


def test_pack_rays_f32_refuses_what_it_would_have_to_round():
    with pytest.raises(TypeError):
        pack_rays_f32(np.zeros((4, 7)))
    with pytest.raises(ValueError):
        pack_rays_f32(np.zeros((4, 8), dtype=np.float32))
    a = np.arange(14, dtype=np.float32).reshape(2, 7)
    r = pack_rays_f32(a)
    assert r["o"].tolist() == [[0, 1, 2], [7, 8, 9]] and r["d"].tolist() == [[3, 4, 5], [10, 11, 12]]
    assert r["t_max"].tolist() == [6, 13] and (r["reserved"] == 0).all()
