"""Trees with spatial splits on the GPU: a triangle referenced from several leaves must not change a closest or an any
hit (Tier F: closest t, exact ties to the lowest prim id), and a tree with such duplicates must survive export / import."""
import numpy as np
import pytest

import scenes
from rs_ray_toy_b200 import synth
from test_sbvh_host import grass

pytestmark = pytest.mark.gpu


def _closest_matches(hits, ref):
    c = scenes.compare_closest(hits, ref["prim"], ref["t"])
    assert c["mismatch_excl_ties"] == 0 and c["t_bad"] == 0, c
    return c


def test_grass_closest_and_any_hit_vs_oracle(ctx):
    """Long diagonal slivers, where the builder must split references: closest and any hits are the oracle's, and the
    records outnumber the primitives."""
    p, idx = grass(40000)
    rays = synth.bounce_rays(p, idx, 200000, seed=21)
    rng = np.random.default_rng(22)
    far = np.concatenate([rng.uniform(-0.5, 1.5, (50000, 3)), synth.random_unit_vectors(50000, rng), np.full((50000, 1), np.inf)], axis=1)
    rays = np.concatenate([rays, far])
    agg = scenes.gpu_soup(ctx, p, idx)
    st = agg.stats()
    assert st["n_prims"] == 40000 and 40000 < st["n_records"] <= 52000, st
    oracle = scenes.oracle_soup(p, idx)
    _closest_matches(agg.intersect(rays), oracle.intersect(rays))
    sh = synth.shadow_rays_from(rays, (0.5, 0.5, 2.0))
    occ_ref, _ = oracle.intersect_p(sh)
    assert (agg.intersect_p(sh) == occ_ref).all()


def test_config3_soup_keeps_node32_and_splits(ctx):
    """Config 3's soup is committed with spatial splits and still quantised to Node32, at a depth the stack holds."""
    p, idx = synth.soup_triangles(1 << 20)
    agg = scenes.gpu_soup(ctx, p, idx)
    st, info = agg.stats(), agg.build_info()
    assert info["node_bytes"] == 32, info
    assert st["n_prims"] == 1 << 20 and (1 << 20) < st["n_records"] <= 1.3 * (1 << 20), st
    assert st["max_depth"] <= 53, st
    assert (st["device_bytes"] - 48 * st["n_records"]) // st["n_nodes"] == 32, st
    rays = synth.bounce_rays(p, idx, 100000, seed=23)
    _closest_matches(agg.intersect(rays), scenes.oracle_soup(p, idx).intersect(rays))


def test_tree_with_duplicates_exports_and_imports(ctx):
    """rrt_scene_export_tree / rrt_scene_commit_from_tree carry the duplicated records: the imported aggregate has the
    same statistics and gives the same hits, bit for bit."""
    from rs_ray_toy_b200.aggregate import GpuAggregate

    p, idx = grass(20000, seed=5)
    rays = synth.bounce_rays(p, idx, 100000, seed=24)
    a = scenes.gpu_soup(ctx, p, idx)
    assert a.stats()["n_records"] > 20000
    blob = a.export_tree()
    b = GpuAggregate(ctx)
    b.add_triangles(b.add_mesh(p, idx), 0)
    b.commit_from_tree(blob)
    sa, sb = a.stats(), b.stats()
    for k in ("n_nodes", "n_leaves", "max_depth", "device_bytes", "n_records", "n_prims"):
        assert sa[k] == sb[k], (k, sa, sb)
    ha, hb = a.intersect(rays), b.intersect(rays)
    assert ha.tobytes() == hb.tobytes()
    assert (a.intersect_p(rays) == b.intersect_p(rays)).all()
