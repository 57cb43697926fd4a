"""The image path on the host: the library's PNG reader, MIPMap::create + lookups (csrc/image_host.cpp, csrc/mipmap_core.h —
the code the shade kernels run) and the InfiniteAreaLight functions, against the oracle's separate restatement of
mipmap.rs / memory.rs / lights/infinite.rs (oracle/rt_mipmap.hpp).  Bit for bit: both sides use libm on the host."""
import ctypes as C

import numpy as np
import pytest

import oracle_lib as O
import oracle_scene as S
from rs_ray_toy_b200 import capi, synth


def _libs():
    Lo, Ld = O.lib(), capi.lib()
    Lo.orc_scene_new.restype = C.c_void_p
    Lo.orc_add_image.restype = C.c_int32
    Lo.orc_add_image.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_int32, C.c_double, C.c_uint32]
    Lo.orc_mipmap_probe.restype = C.c_int32
    Lo.orc_mipmap_probe.argtypes = [C.c_void_p, C.c_int32, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]
    Lo.orc_envlight_probe.restype = C.c_int32
    Lo.orc_envlight_probe.argtypes = [C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]
    Ld.rrt_png_host_probe.restype = C.c_int
    Ld.rrt_png_host_probe.argtypes = [C.c_char_p, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.c_void_p, C.c_uint64]
    Ld.rrt_mipmap_host_probe.restype = C.c_int
    Ld.rrt_mipmap_host_probe.argtypes = [C.c_uint32, C.c_uint32, C.c_void_p, C.c_int, C.c_double, C.c_uint32, C.c_uint64, C.c_void_p,
                                         C.c_void_p, C.c_void_p]
    Ld.rrt_envlight_host_probe.restype = C.c_int
    Ld.rrt_envlight_host_probe.argtypes = [C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_uint64, C.c_void_p, C.c_void_p]
    return Lo, Ld


def read_png(path):
    _, Ld = _libs()
    w, h = C.c_uint32(), C.c_uint32()
    capi.check(Ld.rrt_png_host_probe(str(path).encode(), C.byref(w), C.byref(h), None, 0))
    out = np.zeros((h.value, w.value, 3), dtype=np.uint8)
    capi.check(Ld.rrt_png_host_probe(str(path).encode(), C.byref(w), C.byref(h), out.ctypes.data, out.size))
    return out


def test_png_reader_matches_pil(tmp_path):
    from PIL import Image
    rng = np.random.default_rng(3)
    for k, (w, h, mode) in enumerate([(37, 21, "RGB"), (64, 64, "RGBA"), (5, 9, "L"), (33, 7, "LA"), (130, 3, "RGB")]):
        ch = {"RGB": 3, "RGBA": 4, "L": 1, "LA": 2}[mode]
        a = rng.integers(0, 256, (h, w, ch), dtype=np.uint8)
        # smooth rows too, so that every scanline filter type is chosen by the encoder
        a[::2] = (np.linspace(0, 255, w)[None, :, None] * np.ones((1, 1, ch))).astype(np.uint8)
        path = tmp_path / f"t{k}.png"
        Image.fromarray(a.squeeze() if ch == 1 else a, mode).save(path, optimize=bool(k % 2))
        assert np.array_equal(read_png(path), S.decode_rgb8(path))
    pal = Image.fromarray(rng.integers(0, 256, (20, 31, 3), dtype=np.uint8), "RGB").quantize(13)
    pal.save(tmp_path / "p.png")
    assert np.array_equal(read_png(tmp_path / "p.png"), S.decode_rgb8(tmp_path / "p.png"))
    with pytest.raises(capi.RrtError):
        read_png(tmp_path / "missing.png")
    (tmp_path / "bad.png").write_bytes(b"not a png at all")
    with pytest.raises(capi.RrtError):
        read_png(tmp_path / "bad.png")


@pytest.mark.parametrize("w,h,tri,wrap", [(300, 140, 0, 0), (256, 128, 1, 2), (256, 128, 0, 1), (718, 300, 0, 0), (130, 129, 1, 0), (64, 16, 1, 2)])
def test_mipmap_equals_the_oracles(tmp_path, w, h, tri, wrap):
    """MIPMap::create (Lanczos resampling to powers of two, the BlockedArray's folding index, the pyramid that stops at
    64 texels) and lookup_d / lookup_w: trilinear, EWA (its st[0] row offset included), the three wrap modes."""
    Lo, Ld = _libs()
    img = S.decode_rgb8(synth.write_test_png(str(tmp_path / "a.png"), w, h, seed=w + h))
    rng = np.random.default_rng(w * 7 + h)
    n = 4000
    q = np.zeros((n, 6))
    q[:, 0:2] = rng.uniform(-0.6, 1.6, (n, 2))
    scale = 10.0 ** rng.uniform(-4.5, -0.5, (n, 1))
    q[:, 2:6] = rng.normal(size=(n, 4)) * scale
    q[::7, 4:6] = 0.0          # no y differential: triangle(0)
    q[::11, 2:6] = 0.0         # a later bounce: no differentials at all
    q[5::13, 2:4] *= 300.0     # strongly anisotropic footprints
    sc = Lo.orc_scene_new(0)
    k = Lo.orc_add_image(sc, w, h, img.ctypes.data, tri, 8.0, wrap)
    assert k == 0
    ref, got = np.zeros((n, 6)), np.zeros((n, 6))
    ri, gi = np.zeros(32, dtype=np.uint64), np.zeros(32, dtype=np.uint64)
    assert Lo.orc_mipmap_probe(sc, 0, n, q.ctypes.data, ref.ctypes.data, ri.ctypes.data) == 0
    capi.check(Ld.rrt_mipmap_host_probe(w, h, img.ctypes.data, tri, 8.0, wrap, n, q.ctypes.data, got.ctypes.data, gi.ctypes.data))
    assert np.array_equal(ri, gi) and ri[0] >= 1
    assert np.array_equal(ref, got, equal_nan=True)
    # (an EWA footprint whose ellipse test — made with the st[0] row offset, Q32 — admits no texel divides 0 by 0: the
    # reference returns NaN there, and si_render turns such a sample black)
    assert np.nanmax(got[:, :3]) > 0.05
    if wrap != 1:   # ImageWrap::Black reads cell (0, 0) for every in-range texel (Q32): a two-colour texture
        assert len(np.unique(got[:, 3])) > 100


def test_a_new_oracle_scene_holds_no_images_of_a_freed_one():
    """The oracle keys a scene's images by its address, which a scene made after a free may reuse."""
    Lo, _ = _libs()
    img = np.zeros((140, 300, 3), dtype=np.uint8)
    for _ in range(3):
        sc = Lo.orc_scene_new(0)
        assert [Lo.orc_add_image(sc, 300, 140, img.ctypes.data, 0, 8.0, 0) for _ in range(3)] == [0, 1, 2]
        Lo.orc_scene_free(sc)


def test_tiny_images_are_refused():
    """An 8 x 8 level indexes outside its BlockedArray: the reference panics at load (memory.rs:76-85)."""
    _, Ld = _libs()
    img = np.zeros((8, 8, 3), dtype=np.uint8)
    info, out = np.zeros(32, dtype=np.uint64), np.zeros(6)
    assert Ld.rrt_mipmap_host_probe(8, 8, img.ctypes.data, 1, 8.0, 0, 0, None, None, info.ctypes.data) == capi.RRT_ERR_UNSUPPORTED


def test_infinite_light_equals_the_oracles(tmp_path):
    """InfiniteAreaLight::new's sin-weighted luminance distribution at twice the map's resolution, sample_li, le and
    pdf_li with its quirks (Q34), under a rotated light_to_world."""
    Lo, Ld = _libs()
    img = S.decode_rgb8(synth.write_test_png(str(tmp_path / "e.png"), 200, 90, seed=4, alpha=True))
    m, inv = O.make_to_world((0, 0, 0), (0.2, 1.0, -0.3), 40.0, (1, 1, 1))
    wb = np.array([-3.0, -2.0, -1.0, 5.0, 6.0, 9.0])
    centre = (wb[:3] + wb[3:]) / 2
    radius = float(np.sqrt(((centre - wb[3:]) ** 2).sum()))
    rng = np.random.default_rng(8)
    n = 3000
    q = np.zeros((n, 8))
    q[:, 0:3] = rng.uniform(-2, 2, (n, 3))
    q[:, 3:5] = rng.uniform(0, 1, (n, 2))
    q[:5, 3:5] = [[0, 0], [0.999999, 0.999999], [0.5, 0.0], [-0.3, 0.4], [0.2, -0.7]]   # corners; negative = overflow draws (Q12)
    d = rng.normal(size=(n, 3))
    q[:, 5:8] = d / np.linalg.norm(d, axis=1, keepdims=True)
    q[5, 5:8] = (0, 0, 1)
    q[6, 5:8] = (0, 0, -1)
    ref, got = np.zeros((n, 12)), np.zeros((n, 12))
    mm, ii = np.ascontiguousarray(m.reshape(16)), np.ascontiguousarray(inv.reshape(16))
    assert Lo.orc_envlight_probe(200, 90, img.ctypes.data, mm.ctypes.data, ii.ctypes.data, wb.ctypes.data, n, q.ctypes.data, ref.ctypes.data) == 0
    capi.check(Ld.rrt_envlight_host_probe(200, 90, img.ctypes.data, mm.ctypes.data, ii.ctypes.data, radius, n, q.ctypes.data, got.ctypes.data))
    assert np.array_equal(ref, got, equal_nan=True)
    assert (got[:, 6] > 0).mean() > 0.9 and got[:, 8:11].max() > 0.1
