"""The reference's own rendered image (samples/scene.png) against the oracle, and config 1 exactly as shipped
(`Integrator: Debug`, `Sampler: StratifiedSampler`) through the oracle's literal tier.

FINDING (stated in DESIGN.md §2 "Oracle pin status"): samples/scene.png was NOT rendered from the samples/scene.json
that ships next to it, so it cannot pin the oracle.  Evidence, all checked below against the committed fixture
tests/golden/reference_scene_png.npz (made by tests/golden/make_reference_image_fixture.py from the PNG):
  1. Geometry.  The PNG shows a cube whose visible face is a square rotated IN the image plane — that is the instance
     rotated 15 deg about the x axis seen along x — and two cubes of very different apparent size.  scene.json looks
     from (0,15,-25) towards (35,0,0), i.e. along (0.77,-0.33,0.55): no face of the three unit-scale cubes at x = 35.2
     projects to a square there.  Mask IoU between the PNG and the literal-tier render of scene.json is 0.27 (a render
     of the same scene under a different jitter seed scores > 0.97).
  2. Colour.  75 % of the PNG's coloured pixels have blue < red (mean R:G:B = 15.6 : 15.9 : 9.5).  In scene.json every
     point light sits at the origin (Q17, renderprocess.rs:996) with summed intensity (1600, 1800, 1800) on a grey
     Matte (kd 0.5) under `0.1 + direct`: blue == green >= red on EVERY pixel, whatever the geometry.
So the PNG predates the JSON (different camera, instance placement and lights); nothing else under /root/reference is
an output of the reference.  The oracle stays pinned by the reference's five KATs + line-by-line restatement."""
import ctypes as C
import json
from pathlib import Path

import numpy as np
import pytest

import oracle_lib as O
import oracle_scene as S
from rs_ray_toy_b200 import synth

GOLD = Path(__file__).resolve().parent / "golden" / "reference_scene_png.npz"
# A stored copy of the reference's samples/scene.json (the reference tree is not part of this repository): what
# scene_c1_as_shipped wrote when this test still compared it with the reference's own file.
REF_JSON = Path(__file__).resolve().parent / "golden" / "scene_c1_as_shipped.json"


def quantise(img):
    """write_image (renderprocess.rs:1501-1530): sRGB gamma (misc.rs:46-52), clamp(255 g + 0.5) as u8."""
    g = np.where(img <= 0.0031308, 12.92 * img, 1.055 * np.power(np.maximum(img, 0), 1.0 / 2.4) - 0.055)
    r = np.clip(255.0 * g + 0.5, 0.0, 255.0)
    return np.where(np.isnan(r), 0.0, r).astype(np.uint8)


@pytest.fixture(scope="module")
def shipped(tmp_path_factory):
    path = synth.scene_c1_as_shipped(str(tmp_path_factory.mktemp("c1_shipped")))
    sc = S.load(path, tier=O.TIER_L)
    return path, sc, sc.render(seed=1, want_dump=True)


def test_synth_as_shipped_is_the_reference_file(tmp_path):
    ours = json.loads(Path(synth.scene_c1_as_shipped(str(tmp_path))).read_text())
    assert ours == json.loads(REF_JSON.read_text())


def test_as_shipped_scene_renders_in_the_literal_tier(shipped):
    """samples/scene.json unmodified: Debug integrator (intersect_debug.rs:56-89), StratifiedSampler 4x4 = 16, of which
    15 are rendered (Q10); unreferenced textures (one of them an ImageTexture) and the Debug material are ignored."""
    path, sc, out = shipped
    st = out["stats"]
    assert st["camera_rays"] + st["zero_weight"] == 640 * 360 * 15
    assert st["extension_rays"] == st["camera_rays"] and st["bounces"] == 0 and st["asserts"] == 0
    rgb = out["rgb"]
    # every light at the origin (Q17), grey Matte: G == B to rounding (XYZ round trip), R <= G, and a hit is never darker than 0.1's share
    # (the XYZ -> RGB matrix is the 4-digit inverse of RGB -> XYZ, spectrum.rs:2075-2090: equal to 6e-7 relative)
    assert np.allclose(rgb[..., 1], rgb[..., 2], rtol=2e-6, atol=0) and (rgb[..., 0] <= rgb[..., 1] * (1 + 2e-6)).all()
    # pixels that received at least one hit are exactly the coloured ones (0.1 per hit survives the 8-bit quantisation)
    d = out["dump"]
    hit = np.zeros((360, 640), dtype=bool)
    h = d[d[:, 3] >= 0]
    hit[h[:, 1].astype(int), h[:, 0].astype(int)] = True
    img = quantise(rgb)
    coloured = img.astype(int).sum(-1) > 0
    assert np.array_equal(coloured, hit)
    # the same seed gives the same film; another seed moves the jitter but not the picture
    again = sc.render(seed=1)["rgb"]
    assert np.array_equal(again, rgb)
    other = quantise(sc.render(seed=2)["rgb"]).astype(int).sum(-1) > 0
    iou = (coloured & other).sum() / (coloured | other).sum()
    assert iou > 0.97
    # Debug without lights is the hit mask times 0.1: same coloured pixels
    cfg = json.loads(Path(path).read_text())
    nolight = S.load(path, {"lights": []}, tier=O.TIER_L).render(seed=1)["rgb"]
    assert np.array_equal(quantise(nolight).astype(int).sum(-1) > 0, coloured)
    assert (nolight <= rgb + 1e-15).all() and cfg["Integrator"]["integrator_type"] == "Debug"


def test_reference_png_was_not_rendered_from_the_shipped_json(shipped):
    """The finding in the module docstring, as numbers."""
    _, _, out = shipped
    g = np.load(GOLD)
    ref_mask = np.unpackbits(g["mask"])[: 360 * 640].reshape(360, 640).astype(bool)
    assert int(g["coloured"]) == ref_mask.sum() == 53182
    img = quantise(out["rgb"]).astype(int)
    ours = img.sum(-1) > 0
    iou = (ours & ref_mask).sum() / (ours | ref_mask).sum()
    assert iou < 0.35                      # 0.27: not the same view of the same cubes
    assert float(g["frac_blue_below_red"]) > 0.7 and not (img[ours][:, 2] < img[ours][:, 0]).any()
    # the PNG's yellow: blue is 60 % of red on average; scene.json's lights can only give blue >= red
    m = g["mean_rgb_coloured"]
    assert m[2] / m[0] < 0.7 and img[ours][:, 2].mean() >= img[ours][:, 0].mean()


def test_stratified_sampler_tables():
    """stratified.rs:34-118 + sampling.rs:181-193: per dimension one jittered value per stratum, shuffled; 2D strata are
    the xs x ys grid in row-major order before the shuffle; draws past the tables are U[-1, 1) (Q12)."""
    L = O.lib()
    L.orc_kat_stratified.argtypes = [C.c_uint64, C.c_int64, C.c_int64, C.c_int64, C.c_uint32, C.c_uint32, C.c_uint32,
                                     C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    xs, ys, nd = 4, 4, 4
    n = xs * ys
    seen = []
    for (px, py, jitter) in [(0, 0, 1), (17, 5, 1), (639, 359, 1), (3, 3, 0)]:
        a, b, ov = np.zeros((nd, n)), np.zeros((nd, n, 2)), np.zeros((n, 4))
        L.orc_kat_stratified(7, 640, px, py, xs, ys, nd, jitter, a.ctypes.data, b.ctypes.data, ov.ctypes.data)
        for d in range(nd):
            assert sorted(np.floor(a[d] * n).astype(int)) == list(range(n))
            cells = np.floor(b[d, :, 1] * ys).astype(int) * xs + np.floor(b[d, :, 0] * xs).astype(int)
            assert sorted(cells) == list(range(n))
        assert ((a >= 0) & (a < 1)).all() and ((b >= 0) & (b < 1)).all()
        if not jitter:
            assert np.allclose(np.sort(a[0]), (np.arange(n) + 0.5) / n, rtol=0, atol=0)
        assert ((ov[1:] >= -1) & (ov[1:] < 1)).all() and (ov[1:] < 0).any() and len(np.unique(ov[1:])) == (n - 1) * 4
        seen.append(a.copy())
    assert not np.array_equal(seen[0], seen[1])   # tables differ from pixel to pixel
    # shuffled: over many pixels the stratum held by sample slot 0 (the one Q10 drops) is uniform
    first = []
    for px in range(200):
        a, b, ov = np.zeros((nd, n)), np.zeros((nd, n, 2)), np.zeros((n, 4))
        L.orc_kat_stratified(7, 640, px, 11, xs, ys, nd, 1, a.ctypes.data, b.ctypes.data, ov.ctypes.data)
        first.append(int(b[0, 0, 1] * ys) * xs + int(b[0, 0, 0] * xs))
    assert len(set(first)) == n and max(np.bincount(first)) < 30
