"""Spatial splits in the host SAH builder (csrc/bvh_sah.cpp), without a GPU.  tests/cpp/sbvh_check.cpp builds the
object-split and the spatial-split tree over a triangle file, checks the spatial one (child boxes nested, subtree totals,
every triangle referenced, points sampled on every triangle inside a leaf that references it), walks rays through both
in f64 with the trace kernel's order and accept rule, and reports the closest hits and what the walks cost."""
import os
import re
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest

from rs_ray_toy_b200 import synth

ROOT = Path(__file__).resolve().parent.parent
CSRC = ROOT / "rs_ray_toy_b200" / "csrc"
# the traversal stack holds max_depth + 2 levels; at the Node32 kernel's 8 CTAs per SM, 227 KB of shared memory allow ~55
MAX_DEPTH = 53


def grass(n, seed=11):
    """Thin blades on the unit square, leaning along two crossing diagonals: each blade's box overlaps many others while
    the blade fills a sliver of it — the scene object splits cannot separate and spatial splits must."""
    rng = np.random.default_rng(seed)
    base = np.concatenate([rng.random((n, 2)), np.zeros((n, 1))], axis=1)
    side = np.concatenate([rng.choice([-1.0, 1.0], (n, 1)), np.ones((n, 2))], axis=1)
    lean = np.array([0.03, 0.02, 0.05]) * rng.uniform(0.7, 1.3, (n, 1)) * side
    width = np.concatenate([rng.uniform(-0.002, 0.002, (n, 2)), np.zeros((n, 1))], axis=1)
    p = np.stack([base, base + width, base + lean], axis=1).astype(np.float32).astype(np.float64)
    return p.reshape(-1, 3), np.arange(3 * n, dtype=np.uint32).reshape(n, 3)


@pytest.fixture(scope="module")
def checker(tmp_path_factory):
    gxx = shutil.which("g++") or "/opt/gcc/bin/g++"
    if not Path(gxx).exists():
        pytest.skip("no g++ on this box")
    exe = tmp_path_factory.mktemp("sbvh") / "sbvh_check"
    subprocess.run([gxx, "-O2", "-std=c++17", "-pthread", "-ffp-contract=off", "-I", str(CSRC), "-I", str(ROOT / "include"),
                    "-o", str(exe), str(ROOT / "tests" / "cpp" / "sbvh_check.cpp"), str(CSRC / "bvh_sah.cpp")], check=True)
    return exe


@pytest.fixture(scope="module")
def data(tmp_path_factory):
    d = tmp_path_factory.mktemp("sbvh_data")

    def make(name, p, idx, n_rays):
        p[idx].reshape(-1, 9).tofile(d / f"{name}_tris.bin")
        synth.bounce_rays(p, idx, n_rays, seed=synth.SEED_C3_RAYS).tofile(d / f"{name}_rays.bin")
        return d / f"{name}_tris.bin", d / f"{name}_rays.bin"

    out = {"c3": make("c3", *synth.soup_triangles(1 << 20), 1 << 16),
           "soup300k": make("soup300k", *synth.soup_triangles(300000), 2048),
           "grass": make("grass", *grass(40000), 1 << 15)}
    for n in (2, 3, 17, 500):
        out[f"soup{n}"] = make(f"soup{n}", *synth.soup_triangles(n, edge=0.3), 4096)
    return out


def run(checker, files, threads=None, **env):
    e = dict(os.environ, **{k: str(v) for k, v in env.items()})
    if threads is not None:
        e["T"] = str(threads)
    r = subprocess.run([str(checker), str(files[0]), str(files[1])], capture_output=True, text=True, timeout=600, env=e)
    out = r.stdout
    assert r.returncode == 0, out + r.stderr
    assert "structure VALID" in out and "coverage COMPLETE" in out and "closest hits IDENTICAL" in out, out
    refs, depth = map(int, re.search(r"^fingerprint \w+ refs (\d+) depth (\d+)", out, re.M).groups())
    n = int(re.search(r"^object  build .* (\d+) refs", out, re.M).group(1))
    cost = {k: (float(a), float(b)) for k, a, b in
            re.findall(r"^cost (\w+)\s*: ([\d.]+) interior visits, ([\d.]+) leaf tests", out, re.M)}
    return {"out": out, "n": n, "refs": refs, "depth": depth, "cost": cost,
            "fingerprint": re.search(r"^fingerprint .*$", out, re.M).group(0)}


def test_config3_tree_is_valid_gives_the_same_hits_and_costs_less(checker, data):
    """The config-3 soup (1 Mi triangles) and 2^16 of its bounce rays: a valid tree within the reference budget and the
    depth the stack allows, the object-split tree's closest hits bit for bit, and fewer node visits and leaf tests."""
    r = run(checker, data["c3"])
    assert r["n"] < r["refs"] <= 1.3 * r["n"], r["out"]
    assert r["depth"] <= MAX_DEPTH, r["out"]
    (vo, to), (vs, ts) = r["cost"]["object"], r["cost"]["spatial"]
    assert vs < vo and ts < to, r["out"]


def test_tree_does_not_depend_on_the_thread_count(checker, data):
    """300k triangles: the top nodes (>= 2^18 references) split their binning and partition passes over threads, and
    the free slots of the reference budget are shared out by count — the tree must be the one a single thread builds."""
    fps = [run(checker, data["soup300k"], threads=t)["fingerprint"] for t in (1, 3, 16)]
    assert fps[0] == fps[1] == fps[2], fps


def test_grass_is_split_and_stays_valid(checker, data):
    """Long diagonal slivers: spatial splits must happen, and the tree obeys everything the soup's does."""
    r = run(checker, data["grass"])
    assert r["refs"] > 1.05 * r["n"] and r["refs"] <= 1.3 * r["n"], r["out"]
    assert r["depth"] <= MAX_DEPTH, r["out"]
    (vo, to), (vs, ts) = r["cost"]["object"], r["cost"]["spatial"]
    assert vs + ts < vo + to, r["out"]
    fps = [run(checker, data["grass"], threads=t)["fingerprint"] for t in (1, 16)]
    assert fps[0] == fps[1], fps


@pytest.mark.parametrize("n", [2, 3, 17, 500])
def test_small_scenes(checker, data, n):
    """Large triangles (edges up to 0.3 in the unit cube) in tiny scenes: the budget rounds down to few or no free slots."""
    r = run(checker, data[f"soup{n}"])
    assert r["n"] <= r["refs"] <= max(r["n"], int(1.3 * r["n"])), r["out"]


@pytest.mark.parametrize("cap", ["1", "1.1", "2"])
def test_reference_cap_is_kept(checker, data, cap):
    """RRT_SBVH_CAP bounds the references; at 1 the spatial tree is the object-split tree."""
    r = run(checker, data["grass"], RRT_SBVH_CAP=cap)
    assert r["refs"] <= float(cap) * r["n"], r["out"]
    if cap == "1":
        assert r["refs"] == r["n"] and r["cost"]["object"] == r["cost"]["spatial"], r["out"]
