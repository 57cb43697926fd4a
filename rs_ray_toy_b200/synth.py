"""Synthetic workloads of BASELINE.json's configs (seeded, numpy only, no device code).

Scenes are returned as plain arrays in the reference's own terms — mesh vertices `p`
(f64), 0-based triangle vertex indices, instance transforms as (m, m_inv) 4x4 pairs —
so the same arrays feed both the CPU oracle (tests only) and the CUDA library.

Vertices are drawn in float32 and widened to float64: the reference computes in f64
(`src/geometry.rs:12-20`), and an fp32-exact vertex set lets the device keep 12-byte
vertices without changing a single input bit.  Rays stay full f64.
"""
from __future__ import annotations

import numpy as np

SEED_C2_INSTANCES = 2
SEED_C3_SOUP = 3
SEED_C3_RAYS = 4
SEED_C4_SPHERES = 5
SEED_C5_SOUP = 6


def _rng(seed: int) -> np.random.Generator:
    return np.random.Generator(np.random.PCG64(seed))


def soup_triangles(n_tris: int, edge: float = 0.01, seed: int = SEED_C3_SOUP):
    """Config 3/5 'random-soup' mesh: v0 ~ U([0,1]^3), v1,v2 = v0 + U([-edge,edge]^3).

    Returns (p[3n,3] f64, idx[n,3] u32): one private vertex triple per triangle, the
    layout `create_triangle_mesh` (`src/shape/triangle.rs:131-165`) would get from an
    .obj without shared vertices.
    """
    rng = _rng(seed)
    v0 = rng.random((n_tris, 3), dtype=np.float32)
    d1 = (rng.random((n_tris, 3), dtype=np.float32) * 2 - 1) * np.float32(edge)
    d2 = (rng.random((n_tris, 3), dtype=np.float32) * 2 - 1) * np.float32(edge)
    p = np.empty((n_tris, 3, 3), dtype=np.float32)
    p[:, 0] = v0
    p[:, 1] = v0 + d1
    p[:, 2] = v0 + d2
    idx = np.arange(3 * n_tris, dtype=np.uint32).reshape(n_tris, 3)
    return p.reshape(-1, 3).astype(np.float64), idx


def _concentric_disk(u: np.ndarray) -> np.ndarray:
    """`concentric_sample_disk`, `src/sampling.rs:277-298` (vectorised)."""
    uo = 2.0 * u - 1.0
    x, y = uo[:, 0], uo[:, 1]
    use_x = np.abs(x) > np.abs(y)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(use_x, x, y)
        theta = np.where(use_x, (np.pi / 4) * (y / x), (np.pi / 2) - (np.pi / 4) * (x / y))
    theta = np.where((x == 0) & (y == 0), 0.0, theta)
    r = np.where((x == 0) & (y == 0), 0.0, r)
    return np.stack([r * np.cos(theta), r * np.sin(theta)], axis=1)


def bounce_rays(p: np.ndarray, idx: np.ndarray, n_rays: int, seed: int = SEED_C3_RAYS, offset: float = 1e-4):
    """Config 3 'incoherent diffuse bounce' rays.

    Pick a triangle uniformly, a uniform barycentric point on it, lift the origin by
    `offset` along the unit normal and draw a cosine-weighted direction about that normal
    (`cosine_sample_hemisphere`, `src/sampling.rs:265-274`).  t_max = +inf.
    Returns rays[n,7] f64 = (o, d, t_max) with |d| = 1 to f64 rounding.
    """
    rng = _rng(seed)
    tri = rng.integers(0, idx.shape[0], size=n_rays)
    v = p[idx[tri]]  # [n,3,3]
    b = rng.random((n_rays, 2))
    su = np.sqrt(b[:, 0])
    b0 = 1.0 - su
    b1 = b[:, 1] * su
    pt = b0[:, None] * v[:, 0] + b1[:, None] * v[:, 1] + (1.0 - b0 - b1)[:, None] * v[:, 2]
    n = np.cross(v[:, 1] - v[:, 0], v[:, 2] - v[:, 0])
    ln = np.linalg.norm(n, axis=1, keepdims=True)
    ln[ln == 0] = 1.0
    n = n / ln
    flip = rng.random(n_rays) < 0.5
    n[flip] = -n[flip]
    d2 = _concentric_disk(rng.random((n_rays, 2)))
    z = np.sqrt(np.maximum(0.0, 1.0 - d2[:, 0] ** 2 - d2[:, 1] ** 2))
    # local frame about n (coordinate_system, src/geometry.rs:1146-1161)
    big_x = np.abs(n[:, 0]) > np.abs(n[:, 1])
    s = np.where(big_x[:, None],
                 np.stack([-n[:, 2], np.zeros(n_rays), n[:, 0]], axis=1),
                 np.stack([np.zeros(n_rays), n[:, 2], -n[:, 1]], axis=1))
    ls = np.linalg.norm(s, axis=1, keepdims=True)
    ls[ls == 0] = 1.0
    s = s / ls
    t = np.cross(n, s)
    d = d2[:, 0:1] * s + d2[:, 1:2] * t + z[:, None] * n
    d = d / np.linalg.norm(d, axis=1, keepdims=True)
    rays = np.empty((n_rays, 7), dtype=np.float64)
    rays[:, 0:3] = pt + offset * n
    rays[:, 3:6] = d
    rays[:, 6] = np.inf
    return rays


def shadow_rays_from(rays: np.ndarray, light_pos, seed: int = 11):
    """Any-hit workload: from each ray origin toward a point light, t_max just short of it."""
    o = rays[:, 0:3]
    seg = np.asarray(light_pos, dtype=np.float64)[None, :] - o
    dist = np.linalg.norm(seg, axis=1, keepdims=True)
    out = np.empty_like(rays)
    out[:, 0:3] = o
    out[:, 3:6] = seg / dist
    out[:, 6] = dist[:, 0] * (1.0 - 1e-4)
    return out


def random_unit_vectors(n: int, rng: np.random.Generator) -> np.ndarray:
    z = 1.0 - 2.0 * rng.random(n)
    r = np.sqrt(np.maximum(0.0, 1.0 - z * z))
    phi = 2.0 * np.pi * rng.random(n)
    return np.stack([r * np.cos(phi), r * np.sin(phi), z], axis=1)


def instance_params(n: int, extent: float, seed: int, rotate: bool = True):
    """Config 2/4 instance blocks: world_pos ~ U([-extent,extent]^3), random axis/angle, scale 1.

    Positions are float32-exact.  Returns dict(world_pos[n,3], axis[n,3], angle[n]).
    """
    rng = _rng(seed)
    pos = ((rng.random((n, 3), dtype=np.float32) * 2 - 1) * np.float32(extent)).astype(np.float64)
    if rotate:
        axis = random_unit_vectors(n, rng)
        angle = rng.random(n) * 360.0
    else:
        axis = np.zeros((n, 3))
        angle = np.zeros(n)
    return {"world_pos": pos, "axis": axis, "angle": angle}


def camera_like_rays(n: int, eye, extent: float, seed: int = 12):
    """Rays from one eye point through uniformly random points of the cube [-extent,extent]^3."""
    rng = _rng(seed)
    tgt = (rng.random((n, 3)) * 2 - 1) * extent
    eye = np.asarray(eye, dtype=np.float64)
    d = tgt - eye[None, :]
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    rays = np.empty((n, 7))
    rays[:, 0:3] = eye
    rays[:, 3:6] = d
    rays[:, 6] = np.inf
    return rays


CUBE_P = np.array(
    [[1, 1, -1], [1, -1, -1], [1, 1, 1], [1, -1, 1], [-1, 1, -1], [-1, -1, -1], [-1, 1, 1], [-1, -1, 1]],
    dtype=np.float64,
)
# samples/cube.obj faces (1-based in the file; 0-based here), `v//vn`
CUBE_VI = np.array(
    [[4, 2, 0], [2, 7, 3], [6, 5, 7], [1, 7, 5], [0, 3, 1], [4, 1, 5],
     [4, 6, 2], [2, 6, 7], [6, 4, 5], [1, 3, 7], [0, 2, 3], [4, 0, 1]],
    dtype=np.uint32,
)
CUBE_N = np.array([[0, 1, 0], [0, 0, 1], [-1, 0, 0], [0, -1, 0], [1, 0, 0], [0, 0, -1]], dtype=np.float64)
CUBE_NI = np.repeat(np.array([0, 1, 2, 3, 4, 5, 0, 1, 2, 3, 4, 5], dtype=np.uint32)[:, None], 3, axis=1)


# ---- scene.json writers (reference-compatible files for configs 1, 2 and 4) ------------------------
# Lens prescription used by the reference's sample scene (a 13-interface double-Gauss design in
# millimetres: curvature radius, thickness, index of refraction, aperture diameter per interface).
DGAUSS_LENS = [
    71.97476, 2.43276, 1.54, 47.432, 23.39436, 19.9914, 1, 35.992, 26.17428, 10.25244, 1.772, 24.728,
    -45.26588, 3.53848, 1.617, 19.624, 142.11604, 1.6368, 1, 18.304, 0, 4.55532, 0, 17.512,
    -19.17168, 4.86508, 1.617, 16.368, -22.57728, 0.23012, 1, 18.304, -333.553, 6.19212, 1.713, 21.296,
    -15.1822, 2.65364, 1.805, 22.88, -33.5324, 7.96136, 1, 24.552, -15.40572, 2.43276, 1.617, 26.84,
    -23.94656, 0, 1, 35.992,
]


def write_cube_obj(path):
    """An 8-vertex, 12-triangle cube with per-face normals in the .obj dialect objparser.rs reads
    (`v`, `vn`, `f v//vn`), matching CUBE_P / CUBE_VI / CUBE_N above."""
    lines = ["o Cube"]
    lines += ["v %.6f %.6f %.6f" % tuple(p) for p in CUBE_P]
    lines += ["vn %.4f %.4f %.4f" % tuple(n) for n in CUBE_N]
    for t in range(12):
        lines.append("f " + " ".join("%d//%d" % (CUBE_VI[t, k] + 1, CUBE_NI[t, k] + 1) for k in range(3)))
    with open(path, "w") as f:
        f.write("\n".join(lines) + "\n")


def _const_rgb_texture(name, rgb):
    """The reference-loadable way to give a material a constant colour: a BilerpTexture whose corners
    agree (renderprocess.rs:437-447 reads v10 and v11 from key "v01" as well)."""
    v = {"values": [float(rgb[0]), float(rgb[1]), float(rgb[2])]}
    return {"texture_name": name, "texture_type": "BilerpTexture", "v00": v, "v01": v}


def _const_float_texture(name, value):
    return {"texture_name": name, "texture_type": "BilerpTexture", "v00": float(value), "v01": float(value)}


def _camera(world_pos, look, up=(0.0, 1.0, 0.0), focus_distance=30.0, aperture_diameter=50.0):
    return {"lens_data": DGAUSS_LENS, "focus_distance": focus_distance, "aperture_diameter": aperture_diameter,
            "world_pos": list(world_pos), "look": list(look), "up": list(up)}


def scene_c1(directory, xres=640, yres=360, nsamp=17, integrator="Path", max_depth=5):
    """Config 1: the reference's sample scene (three instanced cubes, three point lights, the
    double-Gauss camera at (0,15,-25) looking at (35,0,0), 20 mm film) with the reproducible
    Halton sampler and the Path integrator.  Returns the scene.json path."""
    import json
    import os
    os.makedirs(directory, exist_ok=True)
    write_cube_obj(os.path.join(directory, "cube.obj"))
    cfg = {
        "float_texture": [], "rgb_texture": [],
        "materials": [{"material_type": "MetalMaterial", "material_name": "mat_metal"},
                      {"material_type": "PlasticMaterial", "material_name": "mat_plastic"},
                      {"material_type": "MatteMaterial", "material_name": "mat_matte"}],
        "objs": [{"filename": "cube.obj", "obj_name": "cube_01"}],
        "lights": [
            {"light_type": "point", "world_pos": [25.66, 8.69, 4.0], "spectrum": {"values": [800, 800, 800]}},
            {"light_type": "point", "world_pos": [25.66, 6.69, -4.0], "spectrum": {"values": [800, 0, 0]}},
            {"light_type": "point", "world_pos": [30, -3.69, -6.0], "spectrum": {"values": [0, 1000, 1000]}}],
        "infinite_lights": [],
        "Aggregate": {"max_prims_in_node": 4, "primitives": [{
            "primitive_type": "triangle", "material_name": "mat_matte", "obj_name": "cube_01",
            "instances": [
                {"world_pos": [35.2, 1.0, 2.8], "scale": [1, 1, 1], "rotation_axis": [1.0, 0.0, 0.0], "rotation_angle": 15},
                {"world_pos": [35.2, -0.3, -2.4], "scale": [1, 1, 1], "rotation_axis": [0.0, 0.0, 1.0], "rotation_angle": 35},
                {"world_pos": [35.2, -1.3, 0.4], "scale": [1, 1, 1], "rotation_axis": [0.0, 0.0, 1.0], "rotation_angle": 78}]}]},
        "Integrator": {"integrator_type": integrator, "max_depth": max_depth, "rr_threshold": 1.0},
        "Sampler": {"sampler_type": "HaltonSampler", "nsamp": nsamp},
        "Film": {"xres": xres, "yres": yres, "diagonal": 20, "Filter": {}},
        "Camera": _camera((0.0, 15, -25.0), (35, 0, 0)),
    }
    path = os.path.join(directory, "scene.json")
    with open(path, "w") as f:
        json.dump(cfg, f, indent=1)
    return path


def scene_c1_as_shipped(directory):
    """Config 1 exactly as the reference ships it (samples/scene.json): the same geometry, lights, film and camera as
    scene_c1, plus what scene_c1 leaves out — the unreferenced WindyTexture / ImageTexture("s_01.png") declarations,
    the `Debug` material, `Integrator {Debug, light_strategy all}` and `Sampler {StratifiedSampler}` (4 x 4, jittered,
    4 sampled dimensions by default).  tests/test_reference_image.py checks this dict against a stored copy of the
    reference's file (tests/golden/scene_c1_as_shipped.json).  s_01.png is NOT written: no material names that texture."""
    import json
    import os
    cfg = json.loads(open(scene_c1(directory)).read())
    cfg["float_texture"] = [{"texture_name": "windy_01", "texture_type": "WindyTexture", "world_pos": [1, 1, 1]}]
    cfg["rgb_texture"] = [{"texture_name": "s_01", "texture_type": "ImageTexture", "filename": "s_01.png"}]
    cfg["materials"].append({"material_type": "Debug", "material_name": "mat_debug"})
    cfg["Integrator"] = {"integrator_type": "Debug", "light_strategy": "all"}
    cfg["Sampler"] = {"sampler_type": "StratifiedSampler"}
    path = os.path.join(directory, "scene_as_shipped.json")
    with open(path, "w") as f:
        json.dump(cfg, f, indent=1)
    return path


def write_test_png(path, width, height, seed=0, alpha=False):
    """A synthetic 8-bit PNG (smooth gradients + a grid + noise, so that filtering matters) written with PIL — the
    harness's encoder; the product decodes with its own reader (csrc/png_read.cpp)."""
    from PIL import Image
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:height, 0:width]
    r = 127.5 * (1 + np.sin(x * 0.21 + seed)) * (y / max(1, height - 1))
    g = 255.0 * ((x // 7 + y // 5) % 2) * 0.6 + 40
    b = 255.0 * (x / max(1, width - 1)) ** 2
    img = np.stack([r, g, b], axis=-1) + rng.uniform(-12, 12, (height, width, 3))
    img = np.clip(img, 0, 255).astype(np.uint8)
    if alpha:
        img = np.concatenate([img, np.full((height, width, 1), 200, dtype=np.uint8)], axis=-1)
    Image.fromarray(img, "RGBA" if alpha else "RGB").save(path)
    return path


def scene_env_and_images(directory, xres=192, yres=108, nsamp=9, integrator="Path", max_depth=4):
    """Config 1's cubes with what SURVEY §8f rows 2-3 still lacked: an InfiniteAreaLight (environment map, listed both in
    `lights` — next-event estimation with a live BSDF-sampling half — and in `infinite_lights` — radiance of escaped
    camera rays) and ImageTextures (a 300 x 140 map that MIPMap::create resamples to 512 x 256, trilinear and EWA, with
    UV / planar mappings) driving kd and ks, next to a point light.  Mirror and plastic cubes reflect the map."""
    import json
    import os
    os.makedirs(directory, exist_ok=True)
    cfg = json.loads(open(scene_c1(directory, xres=xres, yres=yres, nsamp=nsamp, integrator=integrator, max_depth=max_depth)).read())
    # sizes: a MIPMap needs two levels or more for its EWA lookups (with one level the reference indexes past the end
    # of its pyramid and panics, Q32), and a level is kept only while both sides are >= 64 texels
    write_test_png(os.path.join(directory, "env.png"), 200, 90, seed=3, alpha=True)
    write_test_png(os.path.join(directory, "tex_a.png"), 300, 140, seed=1)
    write_test_png(os.path.join(directory, "tex_b.png"), 256, 128, seed=2)
    cfg["rgb_texture"] = [
        {"texture_name": "img_ewa", "texture_type": "ImageTexture", "filename": "tex_a.png",
         "mapping": {"mapping": "uv", "su": 3.0, "sv": 2.0, "du": 0.25, "dv": 0.5}},
        {"texture_name": "img_tri", "texture_type": "ImageTexture", "filename": "tex_b.png", "do_trilinear": True, "wrap": "clamp",
         "mapping": {"mapping": "planar", "v1": [0.0, 0.31, 0.0], "v2": [0.0, 0.0, 0.27], "udelta": 0.1, "vdelta": 0.2}},
        {"texture_name": "img_black", "texture_type": "ImageTexture", "filename": "tex_b.png", "wrap": "black", "max_aniso": 2.0}]
    cfg["materials"] = [{"material_type": "MatteMaterial", "material_name": "mat_matte", "kd": "img_ewa"},
                        {"material_type": "PlasticMaterial", "material_name": "mat_plastic", "kd": "img_tri", "ks": "img_black"},
                        {"material_type": "MirrorMaterial", "material_name": "mat_mirror"}]
    env = {"light_type": "infinite", "mapname": "env.png", "l": {"values": [2.0, 2.0, 2.0]},
           "rotation_axis": [0.0, 1.0, 0.0], "rotation_angle": 40.0}
    cfg["lights"] = [env, {"light_type": "point", "spectrum": {"values": [300, 300, 300]}}]
    cfg["infinite_lights"] = [env]
    prim = cfg["Aggregate"]["primitives"][0]
    inst = prim["instances"]
    prims = []
    for k, name in enumerate(("mat_matte", "mat_plastic", "mat_mirror")):
        q = dict(prim)
        q["material_name"] = name
        q["instances"] = [inst[k]]
        prims.append(q)
    cfg["Aggregate"]["primitives"] = prims
    path = os.path.join(directory, "scene_env.json")
    with open(path, "w") as f:
        json.dump(cfg, f, indent=1)
    return path


def scene_more_materials(directory, xres=192, yres=108, nsamp=9, integrator="Path", max_depth=5, env=False):
    """Config 1's cubes plus five spheres carrying the materials SURVEY §8f row 3 still lacked: TranslucentMaterial (four
    lobes, one with a textured kd and remapped roughness), DisneyMaterial in five settings (default-ish with sheen and
    clearcoat; metallic and anisotropic; thin with all eight lobes; specular transmission; texture-driven color,
    metallic and roughness) and the Debug material.  Point lights, plus an environment map when `env`."""
    import json
    import os
    os.makedirs(directory, exist_ok=True)
    cfg = json.loads(open(scene_c1(directory, xres=xres, yres=yres, nsamp=nsamp, integrator=integrator, max_depth=max_depth)).read())
    # a material parameter is a texture NAME (fetch_float_texture / fetch_rgb_texture, renderprocess.rs:614-661: an inline
    # number is ignored and the default used), so every value below is declared as a constant texture first
    ftex, ctex = [], []

    def f(v):  # one texture per distinct value: the device table holds 32 rows
        name = "f_" + str(v).replace(".", "_")
        if all(t["texture_name"] != name for t in ftex):
            ftex.append(_const_float_texture(name, v))
        return name

    def c(r, g, b):
        name = f"c_{len(ctex)}"
        ctex.append(_const_rgb_texture(name, (r, g, b)))
        return name

    cfg["materials"] = [
        {"material_type": "TranslucentMaterial", "material_name": "m_trans", "kd": c(0.3, 0.5, 0.4), "ks": c(0.3, 0.3, 0.3),
         "reflect": c(0.5, 0.5, 0.5), "transmit": c(0.6, 0.5, 0.7), "roughness": f(0.2)},
        {"material_type": "TranslucentMaterial", "material_name": "m_trans_tex", "kd": "c_checks", "roughness": f(0.3),
         "remap_roughness": True, "transmit": c(0.9, 0.9, 0.9)},
        {"material_type": "DisneyMaterial", "material_name": "m_disney", "color": c(0.6, 0.3, 0.2), "roughness": f(0.4), "sheen": f(0.6),
         "sheen_tint": f(0.3), "clearcoat": f(0.8), "clearcoat_gloss": f(0.7), "specular_tint": f(0.4)},
        {"material_type": "DisneyMaterial", "material_name": "m_disney_metal", "color": c(0.9, 0.7, 0.3), "metallic": f(0.85),
         "anisotropic": f(0.6), "roughness": f(0.35)},
        {"material_type": "DisneyMaterial", "material_name": "m_disney_thin", "color": c(0.3, 0.7, 0.5), "thin": True, "spec_trans": f(0.5),
         "flatness": f(0.4), "diff_trans": f(0.6), "sheen": f(0.5), "clearcoat": f(0.5), "roughness": f(0.45), "eta": f(1.3)},
        {"material_type": "DisneyMaterial", "material_name": "m_disney_glass", "color": c(0.8, 0.85, 0.9), "spec_trans": f(0.7),
         "roughness": f(0.25), "eta": f(1.45)},
        {"material_type": "DisneyMaterial", "material_name": "m_disney_tex", "color": "c_checks", "metallic": "f_checks",
         "roughness": "f_rough", "clearcoat": f(0.3)},
        {"material_type": "Debug", "material_name": "m_debug"},
        # a MixMaterial whose second name is unknown is skipped by the reference's loader (renderprocess.rs:681-693)
        {"material_type": "MixMaterial", "material_name": "m_mix", "mat1": "m_trans", "mat2": "nowhere"}]
    cfg["float_texture"] = ftex + [
        _const_float_texture("f_lo", 0.15), _const_float_texture("f_hi", 0.9),
        {"texture_name": "f_checks", "texture_type": "CheckerBoardTexture", "aamode": "none", "t1": "f_lo", "t2": "f_hi",
         "mapping": {"mapping": "uv", "su": 6.0, "sv": 6.0, "du": 0.0, "dv": 0.0}},
        {"texture_name": "f_rough", "texture_type": "BilerpTexture", "v00": 0.15, "v01": 0.7}]
    cfg["rgb_texture"] = ctex + [
        _const_rgb_texture("c_red", (0.7, 0.2, 0.1)), _const_rgb_texture("c_blue", (0.1, 0.3, 0.8)),
        {"texture_name": "c_checks", "texture_type": "CheckerBoardTexture", "aamode": "none", "t1": "c_red", "t2": "c_blue",
         "mapping": {"mapping": "uv", "su": 4.0, "sv": 4.0, "du": 0.0, "dv": 0.0}}]
    prim = cfg["Aggregate"]["primitives"][0]
    inst = prim["instances"]
    prims = []
    for k, name in enumerate(("m_trans", "m_disney", "m_disney_thin")):
        q = dict(prim)
        q["material_name"] = name
        q["instances"] = [inst[k]]
        prims.append(q)
    spheres = [("m_trans_tex", [33.0, 1.8, -1.2]), ("m_disney_metal", [33.4, -1.6, 1.9]), ("m_disney_glass", [37.0, 2.6, 0.2]),
               ("m_disney_tex", [36.0, 0.2, 5.2]), ("m_debug", [34.0, 2.9, 4.6]), ("m_mix", [31.0, 0.0, 0.0])]
    for name, pos in spheres:
        prims.append({"primitive_type": "sphere", "material_name": name, "radius": 0.85, "world_pos": pos})
    cfg["Aggregate"]["primitives"] = prims
    if env:
        write_test_png(os.path.join(directory, "env.png"), 200, 90, seed=3)
        e = {"light_type": "infinite", "mapname": "env.png", "l": {"values": [1.5, 1.5, 1.5]}}
        cfg["lights"] = [e] + cfg["lights"][:1]
        cfg["infinite_lights"] = [e]
    path = os.path.join(directory, "scene_materials.json")
    with open(path, "w") as f:
        json.dump(cfg, f, indent=1)
    return path


def scene_area_lights(directory, xres=192, yres=108, nsamp=9, integrator="Path", max_depth=5):
    """Config 1's cubes lit by two DiffuseAreaLights (SURVEY.md §8f row 2): a sphere emitter above the cubes and
    triangle 4 of cube.obj (the light shape is the raw mesh triangle, Q7), plus one point light.  The emitters
    are sampled for next-event estimation only — the loader attaches no area light to any primitive (Q22)."""
    import json
    import os
    os.makedirs(directory, exist_ok=True)
    write_cube_obj(os.path.join(directory, "cube.obj"))
    cfg = json.loads(open(scene_c1(directory, xres=xres, yres=yres, nsamp=nsamp, integrator=integrator, max_depth=max_depth)).read())
    cfg["materials"] = [{"material_type": "MatteMaterial", "material_name": "mat_matte"},
                        {"material_type": "PlasticMaterial", "material_name": "mat_plastic"}]
    cfg["lights"] = [
        {"light_type": "diffuse", "spectrum": {"values": [40, 36, 30]}, "n_samples": 1,
         "light_shape": {"shape_type": "sphere", "radius": 1.5, "world_pos": [33.0, 6.0, -1.0]}},
        {"light_type": "diffuse", "spectrum": {"values": [5, 30, 60]},
         "light_shape": {"shape_type": "triangle", "obj_name": "cube_01", "tri_num": 4}},
        {"light_type": "point", "spectrum": {"values": [300, 300, 300]}}]
    prim = cfg["Aggregate"]["primitives"][0]
    second = dict(prim)
    second["material_name"] = "mat_plastic"
    second["instances"] = [{"world_pos": [36.5, 2.2, -0.6], "scale": [1, 1, 1], "rotation_axis": [0.0, 1.0, 0.0], "rotation_angle": 20}]
    cfg["Aggregate"]["primitives"] = [prim, second]
    path = os.path.join(directory, "scene_area.json")
    with open(path, "w") as f:
        json.dump(cfg, f, indent=1)
    return path


def write_floor_obj(path, half=6.0, y=-2.4, cx=35.2, cz=0.0, uv_scale=8.0):
    """A two-triangle floor with texture coordinates (`v`, `vt`, `vn`, `f v/vt/vn`)."""
    xs, zs = (cx - half, cx + half), (cz - half, cz + half)
    lines = ["o Floor"]
    for (x, z) in ((xs[0], zs[0]), (xs[1], zs[0]), (xs[1], zs[1]), (xs[0], zs[1])):
        lines.append("v %.6f %.6f %.6f" % (x, y, z))
    for (u, v) in ((0, 0), (uv_scale, 0), (uv_scale, uv_scale), (0, uv_scale)):
        lines.append("vt %.4f %.4f" % (u, v))
    lines.append("vn 0 1 0")
    lines += ["f 1/1/1 3/3/1 2/2/1", "f 1/1/1 4/4/1 3/3/1"]
    with open(path, "w") as f:
        f.write("\n".join(lines) + "\n")


def scene_textured(directory, xres=192, yres=108, nsamp=9, integrator="Path", max_depth=5):
    """SURVEY.md §8f row 3 (procedural part): config 1's cubes on a floor, plus three spheres, with every in-scope texture
    type driving a material parameter or a bump map — Checkerboard 2D over mesh uvs (closed-form filter: the loader's default, fed by
    the camera ray's differentials) and over a planar mapping (point-sampled),
    Checkerboard 3D with a texture transform, Bilerp (float and rgb), Scale, Mix (whose amount is looked up under
    "t2", renderprocess.rs:319), UV, spherical and cylindrical mappings — on Matte / Plastic / Metal / Mirror."""
    import json
    import os
    os.makedirs(directory, exist_ok=True)
    cfg = json.loads(open(scene_c1(directory, xres=xres, yres=yres, nsamp=nsamp, integrator=integrator, max_depth=max_depth)).read())
    write_floor_obj(os.path.join(directory, "floor.obj"))

    def rgbv(r, g, b):
        return {"values": [r, g, b]}

    cfg["float_texture"] = [
        _const_float_texture("f_lo", 0.05),
        _const_float_texture("f_hi", 0.6),
        {"texture_name": "f_ramp", "texture_type": "BilerpTexture", "v00": 0.02},            # v01 absent: corners 0.02 1 0 1
        {"texture_name": "f_rough_check", "texture_type": "CheckerBoardTexture", "dimension": 3, "t1": "f_lo", "t2": "f_hi",
         "scale": [2.0, 2.0, 2.0]},
        {"texture_name": "f_sigma", "texture_type": "ScaleTexture", "t1": "f_ramp", "t2": "f_sixty"},  # f_sixty unknown: 1.0
        {"texture_name": "dark", "texture_type": "BilerpTexture", "v00": 0.3, "v01": 0.3},   # float amount for the rgb Mix below
        {"texture_name": "f_wrinkle", "texture_type": "WrinkledTexture", "octaves": 5, "omega": 0.6, "scale": [0.7, 0.7, 0.7]},
        # bump maps (Material::bump): a uv-mapped ramp scaled down to millimetres on the floor, the noise on a cube
        {"texture_name": "f_small", "texture_type": "BilerpTexture", "v00": 0.05, "v01": 0.05},
        {"texture_name": "f_bumps", "texture_type": "ScaleTexture", "t1": "f_ramp", "t2": "f_small"},
    ]
    cfg["rgb_texture"] = [
        _const_rgb_texture("white", (0.85, 0.85, 0.8)),
        _const_rgb_texture("dark", (0.1, 0.12, 0.3)),
        _const_rgb_texture("red", (0.7, 0.15, 0.1)),
        {"texture_name": "floor_check", "texture_type": "CheckerBoardTexture", "t1": "white", "t2": "dark"},   # closed-form filter
        {"texture_name": "planar_check", "texture_type": "CheckerBoardTexture", "aamode": "none", "t1": "red", "t2": "white",
         "mapping": {"mapping": "planar", "v1": [1.3, 0.0, 0.2], "v2": [0.0, 1.7, 0.0], "udelta": 0.25, "vdelta": -0.5}},
        {"texture_name": "solid_check", "texture_type": "CheckerBoardTexture", "dimension": 3, "t1": "white", "t2": "red",
         "world_pos": [0.3, 0.1, 0.2], "rotation_axis": [0.0, 1.0, 0.0], "rotation_angle": 30, "scale": [1.5, 1.5, 1.5]},
        {"texture_name": "uvcol", "texture_type": "UVTexture", "mapping": {"mapping": "uv", "su": 3.0, "sv": 2.0, "du": 0.0, "dv": 0.0}},
        {"texture_name": "grad", "texture_type": "BilerpTexture", "v00": rgbv(0.9, 0.2, 0.1), "v01": rgbv(0.1, 0.3, 0.9),
         "mapping": {"mapping": "spherical"}, "world_pos": [33.0, -1.0, 3.0]},
        {"texture_name": "cyl", "texture_type": "UVTexture", "mapping": {"mapping": "cylindrical"}, "world_pos": [37.0, 0.0, -3.0]},
        {"texture_name": "mixed", "texture_type": "MixTexture", "t1": "uvcol", "t2": "dark"},          # amount: float "dark" = 0.3
        {"texture_name": "tinted", "texture_type": "ScaleTexture", "t1": "floor_check", "t2": "grad"},
        # 50-unit checks over the floor (edges at x = 35 and z = 0), closed-form: interaction.rs:237-238 computes the y
        # neighbour's plane distance from the wrong dot product (Q29), so dpdy is tens of units long at a first hit —
        # an 8-checks-per-floor board filters to flat grey there, while this one gets wide but partial footprints
        # whose value depends on every component of the camera ray's differentials
        {"texture_name": "big_check", "texture_type": "CheckerBoardTexture", "t1": "white", "t2": "red",
         "mapping": {"mapping": "planar", "v1": [0.02, 0.0, 0.0], "v2": [0.0, 0.0, 0.02], "udelta": 0.3, "vdelta": 0.0}},
        {"texture_name": "floor_kd", "texture_type": "ScaleTexture", "t1": "floor_check", "t2": "big_check"},
        # Perlin-noise textures (fBm / turbulence; their octave count follows the screen-space footprint)
        {"texture_name": "waves", "texture_type": "WindyTexture", "world_pos": [0.5, 0.25, 0.0]},
        {"texture_name": "wrinkles", "texture_type": "WrinkledTexture", "octaves": 6, "omega": 0.5, "scale": [0.5, 0.5, 0.5]},
        {"texture_name": "marbled", "texture_type": "MixTexture", "t1": "white", "t2": "wrinkles"},  # amount: float "wrinkles"? unknown -> 0.5
        {"texture_name": "rippled", "texture_type": "ScaleTexture", "t1": "grad", "t2": "waves"},
    ]
    cfg["materials"] = [
        {"material_type": "MatteMaterial", "material_name": "m_floor", "kd": "floor_kd", "bump_map": "f_bumps"},
        {"material_type": "MatteMaterial", "material_name": "m_planar", "kd": "planar_check", "sigma": "f_sigma", "bump_map": "f_wrinkle"},
        {"material_type": "PlasticMaterial", "material_name": "m_solid", "kd": "solid_check", "ks": "white", "roughness": "f_rough_check"},
        {"material_type": "PlasticMaterial", "material_name": "m_mixed", "kd": "mixed", "ks": "rippled", "roughness": "f_lo"},
        {"material_type": "MatteMaterial", "material_name": "m_grad", "kd": "marbled", "sigma": "f_wrinkle"},
        {"material_type": "MetalMaterial", "material_name": "m_metal", "roughness": "f_rough_check", "k": "tinted", "bump_map": "f_wrinkle"},
        {"material_type": "MirrorMaterial", "material_name": "m_mirror", "kr": "cyl"},
    ]
    cfg["objs"].append({"filename": "floor.obj", "obj_name": "floor_01"})
    inst = cfg["Aggregate"]["primitives"][0]["instances"]
    cube = {"primitive_type": "triangle", "obj_name": "cube_01"}
    cfg["Aggregate"]["primitives"] = [
        {"primitive_type": "triangle", "obj_name": "floor_01", "material_name": "m_floor", "instances": [{"world_pos": [0, 0, 0]}]},
        dict(cube, material_name="m_planar", instances=[inst[0]]),
        dict(cube, material_name="m_solid", instances=[inst[1]]),
        dict(cube, material_name="m_mixed", instances=[inst[2]]),
        {"primitive_type": "sphere", "radius": 1.0, "material_name": "m_grad", "instances": [{"world_pos": [33.0, -1.0, 3.0]}]},
        {"primitive_type": "sphere", "radius": 0.9, "material_name": "m_metal", "instances": [{"world_pos": [33.5, -1.2, -4.0]}]},
        {"primitive_type": "sphere", "radius": 1.1, "material_name": "m_mirror", "instances": [{"world_pos": [37.5, -0.8, -3.0]}]},
    ]
    cfg["lights"] = [
        {"light_type": "distant", "l": {"values": [2.5, 2.4, 2.2]}, "from": [-0.4, 1.0, -0.6], "to": [0, 0, 0]},
        {"light_type": "point", "spectrum": {"values": [900, 900, 900]}}]
    path = os.path.join(directory, "scene_textured.json")
    with open(path, "w") as f:
        json.dump(cfg, f, indent=1)
    return path


def scene_clipped_spheres(directory, xres=192, yres=108, nsamp=9, integrator="Path", max_depth=5):
    """SURVEY.md §8a6 in the renderer: config 1's floor-less cubes swapped for spheres that are clipped in z and phi
    (bowls and wedges whose inside is seen through the opening: hits at the far root), stretched by their own object
    transform and by their instances, with uv-driven textures so that the hit point's (u, v) shows."""
    import json
    import os
    os.makedirs(directory, exist_ok=True)
    cfg = json.loads(open(scene_c1(directory, xres=xres, yres=yres, nsamp=nsamp, integrator=integrator, max_depth=max_depth)).read())
    cfg["rgb_texture"] = [
        _const_rgb_texture("white", (0.85, 0.85, 0.8)),
        _const_rgb_texture("blue", (0.1, 0.2, 0.6)),
        {"texture_name": "check", "texture_type": "CheckerBoardTexture", "aamode": "none", "t1": "white", "t2": "blue",
         "mapping": {"mapping": "uv", "su": 8.0, "sv": 4.0, "du": 0.0, "dv": 0.0}},
        {"texture_name": "uvcol", "texture_type": "UVTexture"},
    ]
    cfg["float_texture"] = []
    cfg["materials"] = [
        {"material_type": "MatteMaterial", "material_name": "m_check", "kd": "check"},
        {"material_type": "PlasticMaterial", "material_name": "m_uv", "kd": "uvcol", "roughness": 0.2},
        {"material_type": "MetalMaterial", "material_name": "m_metal"},
    ]
    cfg["Aggregate"]["primitives"] = [
        # a bowl (lower part of a sphere), opening towards the camera side, stretched by its instance
        {"primitive_type": "sphere", "radius": 1.6, "z_min": -1.6, "z_max": 0.3, "material_name": "m_check",
         "instances": [{"world_pos": [35.0, 0.5, 2.6], "rotation_axis": [1.0, 0.2, 0.0], "rotation_angle": 70, "scale": [1.0, 1.0, 1.3]}]},
        # a wedge: three quarters of a sphere in phi, the object transform of the sphere itself non-uniform
        {"primitive_type": "sphere", "radius": 1.2, "phi_max": 250.0, "material_name": "m_uv",
         "instances": [{"world_pos": [35.4, -0.2, -0.6], "rotation_axis": [0.0, 1.0, 0.0], "rotation_angle": 200, "scale": [1.0, 0.7, 1.0]},
                       {"world_pos": [33.0, 2.4, -3.2], "rotation_axis": [0.3, 1.0, 0.2], "rotation_angle": 40, "scale": [0.8, 0.8, 0.8]}]},
        # a band (both poles cut away and a slice in phi)
        {"primitive_type": "sphere", "radius": 1.0, "z_min": -0.5, "z_max": 0.5, "phi_max": 300.0, "material_name": "m_metal",
         "instances": [{"world_pos": [36.5, -0.8, -3.4], "rotation_axis": [1.0, 0.0, 0.0], "rotation_angle": 90}]},
        # a full sphere stretched by an object transform of its own, not instanced (Q5a: its (u, v) come from the world point)
        {"primitive_type": "sphere", "radius": 0.8, "material_name": "m_uv",
         "world_pos": [34.2, 1.6, 0.9], "rotation_axis": [0.0, 0.0, 1.0], "rotation_angle": 25, "scale": [1.4, 0.8, 1.0]},
        # and one ordinary full sphere
        {"primitive_type": "sphere", "radius": 0.8, "material_name": "m_check", "instances": [{"world_pos": [33.5, -1.2, 1.0]}]},
    ]
    cfg["objs"] = []
    cfg["lights"] = [
        {"light_type": "distant", "l": {"values": [2.5, 2.4, 2.2]}, "from": [-0.4, 1.0, -0.6], "to": [0, 0, 0]},
        {"light_type": "point", "spectrum": {"values": [900, 900, 900]}}]
    path = os.path.join(directory, "scene_clipped.json")
    with open(path, "w") as f:
        json.dump(cfg, f, indent=1)
    return path


def scene_c2(directory, n_instances=10000, xres=1920, yres=1080, nsamp=2, extent=50.0, seed=SEED_C2_INSTANCES):
    """Config 2: the cube instanced `n_instances` times (random position / axis / angle, unit scale),
    Matte, one point light (which sits at the origin whatever its world_pos, Q17), DirectLighting
    with max_depth 1, Halton nsamp 2 (= 1 rendered sample), camera at (0,0,-4*extent)."""
    import json
    import os
    os.makedirs(directory, exist_ok=True)
    write_cube_obj(os.path.join(directory, "cube.obj"))
    prm = instance_params(n_instances, extent, seed)
    # the point light sits at the origin (Q17): keep it out of the cubes (half-diagonal 1.74) by
    # moving any instance centre closer than 3 units radially out to 3
    pos = prm["world_pos"]
    r = np.linalg.norm(pos, axis=1)
    near = r < 3.0
    pos[near] = (pos[near] / np.maximum(r[near], 1e-9)[:, None] * 3.0).astype(np.float32).astype(np.float64)
    inst = [{"world_pos": prm["world_pos"][i].tolist(), "rotation_axis": prm["axis"][i].tolist(),
             "rotation_angle": float(prm["angle"][i]), "scale": [1, 1, 1]} for i in range(n_instances)]
    cfg = {
        "materials": [{"material_type": "MatteMaterial", "material_name": "mat_matte"}],
        "objs": [{"filename": "cube.obj", "obj_name": "cube_01"}],
        "lights": [{"light_type": "point", "spectrum": {"values": [20000, 20000, 20000]}}],
        "infinite_lights": [],
        "Aggregate": {"max_prims_in_node": 4, "primitives": [
            {"primitive_type": "triangle", "material_name": "mat_matte", "obj_name": "cube_01", "instances": inst}]},
        "Integrator": {"integrator_type": "DirectLighting", "max_depth": 1, "light_strategy": "one"},
        "Sampler": {"sampler_type": "HaltonSampler", "nsamp": nsamp},
        "Film": {"xres": xres, "yres": yres, "diagonal": 35, "Filter": {}},
        "Camera": _camera((0.0, 0.0, -4.0 * extent), (0.0, 0.0, 0.0), focus_distance=4.0 * extent),
    }
    path = os.path.join(directory, "scene.json")
    with open(path, "w") as f:
        json.dump(cfg, f)
    return path


def scene_c4(directory, n_spheres=100000, xres=1920, yres=1080, nsamp=65, extent=50.0, seed=SEED_C4_SPHERES,
             max_depth=5, extra_materials=False):
    """Config 4: `n_spheres` unit-instanced spheres of radius 0.5 as 16 sphere entries (8 Plastic
    presets, roughness 0.05-0.5; 8 Metal presets, copper, roughness 0.01-0.3) x instances[], one
    distant and one point light, Path integrator.  `extra_materials` swaps presets for Mirror, smooth
    Glass, two rough Glasses and an Oren-Nayar Matte (test coverage of the other lobes)."""
    import json
    import os
    os.makedirs(directory, exist_ok=True)
    prm = instance_params(n_spheres, extent, seed, rotate=False)
    ftex, rtex, mats = [], [], []
    for k in range(8):
        rough = 0.05 + (0.5 - 0.05) * k / 7.0
        kd = [0.15 + 0.08 * k, 0.6 - 0.05 * k, 0.25 + 0.03 * k]
        ftex.append(_const_float_texture(f"rough_p{k}", rough))
        rtex.append(_const_rgb_texture(f"kd_p{k}", kd))
        mats.append({"material_type": "PlasticMaterial", "material_name": f"plastic_{k}", "kd": f"kd_p{k}",
                     "roughness": f"rough_p{k}"})
    for k in range(8):
        rough = 0.01 + (0.3 - 0.01) * k / 7.0
        ftex.append(_const_float_texture(f"rough_m{k}", rough))
        mats.append({"material_type": "MetalMaterial", "material_name": f"metal_{k}", "roughness": f"rough_m{k}"})
    if extra_materials:
        mats[7] = {"material_type": "MirrorMaterial", "material_name": "plastic_7"}
        mats[15] = {"material_type": "GlassMaterial", "material_name": "metal_7"}
        mats[3] = {"material_type": "MatteMaterial", "material_name": "plastic_3", "sigma": "rough_m7"}
        # rough glass (MicrofacetReflection + MicrofacetTransmission), anisotropic; and one with remapped roughness
        mats[14] = {"material_type": "GlassMaterial", "material_name": "metal_6", "u_roughness": "rough_m6", "v_roughness": "rough_m3"}
        mats[13] = {"material_type": "GlassMaterial", "material_name": "metal_5", "u_roughness": "rough_p4", "v_roughness": "rough_p4",
                    "remap_roughness": True, "eta": "rough_eta"}
        ftex.append(_const_float_texture("rough_eta", 1.33))
    names = [m["material_name"] for m in mats]
    prims = []
    per = (n_spheres + 15) // 16
    for k in range(16):
        sl = slice(k * per, min(n_spheres, (k + 1) * per))
        inst = [{"world_pos": p.tolist()} for p in prm["world_pos"][sl]]
        if inst:
            prims.append({"primitive_type": "sphere", "radius": 0.5, "material_name": names[k], "instances": inst})
    cfg = {
        "float_texture": ftex, "rgb_texture": rtex, "materials": mats, "objs": [],
        "lights": [{"light_type": "distant", "l": {"values": [3.0, 3.0, 3.0]}, "from": [0.3, 1.0, -0.5], "to": [0, 0, 0]},
                   {"light_type": "point", "spectrum": {"values": [30000, 30000, 30000]}}],
        "infinite_lights": [],
        "Aggregate": {"max_prims_in_node": 4, "primitives": prims},
        "Integrator": {"integrator_type": "Path", "max_depth": max_depth, "rr_threshold": 1.0},
        "Sampler": {"sampler_type": "HaltonSampler", "nsamp": nsamp},
        "Film": {"xres": xres, "yres": yres, "diagonal": 35, "Filter": {"filter_type": "BoxFilter", "radius": [0.5, 0.5]}},
        "Camera": _camera((0.0, 0.0, -4.0 * extent), (0.0, 0.0, 0.0), focus_distance=4.0 * extent),
    }
    path = os.path.join(directory, "scene.json")
    with open(path, "w") as f:
        json.dump(cfg, f)
    return path


def default_render_desc(xres, yres, nsamp, cam_pos, cam_look, cam_up=(0.0, 1.0, 0.0), focus_distance=30.0,
                        aperture_diameter=50.0, diagonal_mm=35.0, integrator="Path", max_depth=5, seed=1):
    """An rrt_render_desc with the loader's defaults (renderprocess.rs:1306-1499) for scenes that are
    assembled through the aggregate API instead of a scene.json (configs 3 and 5: millions of
    triangles do not belong in a text file)."""
    from .render import RenderDesc
    d = RenderDesc()
    d.xres, d.yres = xres, yres
    d.diagonal_mm, d.scale, d.max_sample_luminance = diagonal_mm, 1.0, float("inf")
    d.filter_kind = 0
    d.filter_radius[:] = [0.5, 0.5]
    d.filter_alpha = 2.0
    d.cam_pos[:] = list(cam_pos)
    d.cam_look[:] = list(cam_look)
    d.cam_up[:] = list(cam_up)
    d.shutter_open, d.shutter_close = 0.0, 1.0
    d.aperture_diameter, d.focus_distance = aperture_diameter, focus_distance
    d.simple_weighting = 1
    d.nsamp, d.sample_at_center, d.seed = nsamp, 0, seed
    d.integrator_kind = 0 if integrator == "Path" else 1
    d.max_depth, d.rr_threshold = max_depth, 1.0
    return d


def c5_texture_rows():
    """The optional textures of scene_c5_api(textured=True) as plain tuples (kind, values, mapping, map8, t1, t2,
    world_to_texture) — shared with the oracle-side twin in tests/scenes.py: a 3D checkerboard of 1/8-unit cells for
    the Matte kd and a planar-mapped float ramp for the Plastic roughness."""
    w2t = np.diag([8.0, 8.0, 8.0, 1.0])
    return [
        (0, [(0.75, 0.7, 0.6)], 0, (1, 1, 0, 0, 0, 0, 0, 0), -1, -1, np.eye(4)),
        (0, [(0.15, 0.2, 0.5)], 0, (1, 1, 0, 0, 0, 0, 0, 0), -1, -1, np.eye(4)),
        (5, [], 0, (1, 1, 0, 0, 0, 0, 0, 0), 0, 1, w2t),
        (1, [0.05, 0.4, 0.1, 0.6], 1, (1, 0, 0, 0, 1, 0, 0.0, 0.0), -1, -1, np.eye(4)),
    ]


def scene_c5_api(ctx, n_tris=1 << 22, edge=0.006, xres=3840, yres=2160, nsamp=257, seed=SEED_C5_SOUP, max_depth=5,
                 textured=False, commit=None):
    """Config 5: a `n_tris` random-soup mesh (half Matte, half Plastic), one point light at the origin
    (Q17) and one distant light, camera outside the unit cube looking at its centre.  Returns
    (aggregate, Render).  `textured` drives the Matte kd and the Plastic roughness by c5_texture_rows()
    (rrt_scene_set_textures / rrt_scene_set_material_textures)."""
    from .aggregate import GpuAggregate
    from .render import Render, distant_light, matte, plastic, point_light
    p, idx = soup_triangles(n_tris, edge, seed)
    half = n_tris // 2
    agg = GpuAggregate(ctx)
    m0 = agg.add_mesh(p[: 3 * half], idx[:half])
    m1 = agg.add_mesh(p[3 * half:], idx[half:] - 3 * half)
    agg.add_triangles(m0, 0)
    agg.add_triangles(m1, 1)
    if commit is None:
        agg.commit(4)
    else:
        commit(agg)   # e.g. parallel.commit_replicated: one rank builds the tree, the others receive it
    desc = default_render_desc(xres, yres, nsamp, cam_pos=(0.5, 0.5, -2.5), cam_look=(0.5, 0.5, 0.5), focus_distance=3.0,
                               max_depth=max_depth, seed=1)
    textures = slots = None
    if textured:
        from . import render as R
        textures = [R.texture(k, v, mapping=mp, map8=m8, t1=t1, t2=t2, world_to_texture=w) for (k, v, mp, m8, t1, t2, w) in c5_texture_rows()]
        slots = np.full((2, R.MATERIAL_SLOTS), -1, dtype=np.int32)
        slots[0, R.SLOT_KD] = 2
        slots[1, R.SLOT_ROUGHNESS] = 3
    r = Render.create(agg, [matte((0.6, 0.55, 0.5)), plastic((0.3, 0.4, 0.6), (0.3, 0.3, 0.3), 0.15)],
                      [point_light((4.0, 4.0, 4.0)), distant_light((2.0, 2.0, 2.0), frm=(0.3, 1.0, -0.6), to=(0, 0, 0))],
                      desc, DGAUSS_LENS, textures=textures, material_slots=slots)
    return agg, r
