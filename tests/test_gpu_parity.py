"""Parity of the CUDA path (through the C ABI) with the oracle and the reference's golden vectors.  GPU only.
Bar: bit-exact z, colour and normals (integer/bit compare of the float32 buffers)."""
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, TriModel, bits_equal, case_model, random_scene

pytestmark = pytest.mark.gpu
CHECKS = json.load(open(os.path.join(GOLDEN, "checksums.json")))
def seeded(key):
    """What the reference computed on the seeded inputs below (tests/golden/make_golden_seeded.py)."""
    with open(os.path.join(GOLDEN, "seeded_checksums.json")) as fh:
        return json.load(fh)[key]


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def Filler():
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller
    return AdvancedPixelBufferFiller


@pytest.fixture(scope="module")
def O():
    from oracle import oracle
    return oracle


def buffers(f):
    return f.get_z_buffer().copy(), f.get_color_buffer().copy(), f.get_normals_buffer().copy()


def assert_same(got, want, what=""):
    for name, g, w in zip(("z", "color", "normals"), got, want):
        if not bits_equal(g, w):
            bad = np.argwhere(g.view(np.uint32) != w.view(np.uint32))
            raise AssertionError(f"{what}: {name} differs at {len(bad)} words, first {bad[:5].tolist()}: "
                                 f"got {g[tuple(bad[0])]!r} want {w[tuple(bad[0])]!r}")


@pytest.mark.parametrize("path", ["tiled", "atomic"])
@pytest.mark.parametrize("seed", range(30))
def test_random_scenes_bit_exact(seed, path, Filler, O):
    rng = np.random.default_rng(1000 + seed)
    h, w, fov = int(rng.integers(8, 200)), int(rng.integers(8, 200)), float(rng.uniform(20, 120))
    m = random_scene(seed)
    g, o = Filler(h, w, fov=fov), O.OracleFiller(h, w, fov=fov)
    for _ in range(2 if seed % 3 == 0 else 1):
        g.render_arrays(m._vertices_by_triangles, m._colors_by_triangles, m._normals_by_triangles, path=path)
        o.render_model(m)
    assert_same(buffers(g), buffers(o), f"seed {seed} {h}x{w} {path}")


@pytest.mark.parametrize("seed", range(6))
def test_dense_scenes_bit_exact(seed, Filler, O):
    """Many triangles per tile (several staging passes of the tile rasterizer) and large triangles (many tiles)."""
    m = random_scene(100 + seed, T=6000, span=0.6)
    h, w = (257, 391) if seed % 2 else (512, 512)
    g, o = Filler(h, w, fov=70.0), O.OracleFiller(h, w, fov=70.0)
    g.render_model(m)
    o.render_model(m)
    assert_same(buffers(g), buffers(o), f"dense seed {seed}")


@pytest.mark.parametrize("case", ["trex_1024x1024_fov45", "trex_512x512_fov90", "trex_333x777_fov60",
                                  "trex_2048x2048_fov45", "bunny_1024x1024_fov45", "bunny_500x300_fov30",
                                  "bunny_2048x2048_fov45", "bunny_4096x4096_fov45", "basketball_2048x2048_fov45",
                                  "basketball_1000x1500_fov70"])
def test_reference_golden_checksums(case, Filler, trex, bunny, basketball):
    info = CHECKS["cases"][case]
    m = {"trex": trex, "bunny": bunny, "basketball": basketball}[info["model"]]
    f = Filler(info["h"], info["w"], fov=info["fov"], n_threads=8)
    f.render_model(m)
    z, c, n = f.get_z_buffer(), f.get_color_buffer(), f.get_normals_buffer()
    assert int((z < 1e5).sum()) == info["covered"]
    assert (sha(z), sha(c), sha(n)) == (info["z"], info["color"], info["normals"])


def test_trex_128_full_arrays(Filler, trex):
    g = np.load(os.path.join(GOLDEN, "trex_128.npz"))
    f = Filler(128, 128, fov=45.0)
    f.render_model(trex)
    assert_same(buffers(f), (g["z"], g["color"], g["normals"]), "trex 128")


def test_compositing_two_models_matches_reference(Filler, trex, bunny):
    info = CHECKS["cases"]["trex_then_bunny_640x480_fov50"]
    f = Filler(640, 480, fov=50.0)
    f.render_model(trex)
    f.render_model(bunny)
    assert (sha(f.get_z_buffer()), sha(f.get_color_buffer()), sha(f.get_normals_buffer())) == \
        (info["z"], info["color"], info["normals"])


def _tri(vs, nz=-1.0, col=100.0):
    v = np.asarray(vs, dtype=np.float32).reshape(-1, 3, 3)
    n = np.zeros_like(v)
    n[..., 2] = nz
    c = np.full_like(v, col)
    return v, c, n


KATS = {
    # two triangles sharing the diagonal of a square: inclusive edges, both rasterize the shared pixels
    "shared_edge": _tri([[[-0.5, -0.5, 1], [0.5, -0.5, 1], [0.5, 0.5, 1]], [[-0.5, -0.5, 1], [0.5, 0.5, 1], [-0.5, 0.5, 1]]]),
    # identical geometry twice: exact depth tie -> the higher triangle index must win
    "exact_tie": _tri([[[-0.5, -0.5, 1], [0.5, -0.5, 1], [0.0, 0.5, 1]]] * 2),
    "off_screen": _tri([[[5, 5, 1], [6, 5, 1], [5, 6, 1]]]),
    "zero_area": _tri([[[-0.5, -0.5, 1], [0.0, 0.0, 1], [0.5, 0.5, 1]]]),
    "behind_camera": _tri([[[-0.5, -0.5, -1], [0.5, -0.5, -1], [0.0, 0.5, -1]]]),
    "straddles_camera_plane": _tri([[[-0.5, -0.5, -0.3], [0.5, -0.5, 0.7], [0.0, 0.5, 1.0]]]),
    "back_facing": _tri([[[-0.5, -0.5, 1], [0.5, -0.5, 1], [0.0, 0.5, 1]]], nz=1.0),
    "zero_normal_sum_is_culled": _tri([[[-0.5, -0.5, 1], [0.5, -0.5, 1], [0.0, 0.5, 1]]], nz=0.0),
    "huge": _tri([[[-300, -300, 1], [300, -300, 1], [0.0, 300, 1]]]),
    "out_of_int_range": _tri([[[-3e9, -0.5, 1.0], [3e9, 0.5, 1.0], [0.0, 4e9, 1.0]],
                              [[-0.4, -0.4, 1.5], [0.4, -0.4, 1.5], [0.0, 0.4, 1.5]]]),
    "inf_vertex": _tri([[[-0.5, -0.5, 1], [np.inf, -0.5, 1], [0.0, 0.5, 1]], [[-0.4, -0.4, 1.5], [0.4, -0.4, 1.5], [0.0, 0.4, 1.5]]]),
    "nan_vertex": _tri([[[-0.5, np.nan, 1], [0.5, -0.5, 1], [0.0, 0.5, 1]], [[-0.4, -0.4, 1.5], [0.4, -0.4, 1.5], [0.0, 0.4, 1.5]]]),
    "negative_zero_depth_tie": _tri([[[-0.5, -0.5, 1], [0.5, -0.5, 1], [0.0, 0.5, 1]]]),
}
KATS["exact_tie"][1][1] = 200.0   # second copy has another colour so the winner is visible
KATS["exact_tie"][1][0] = 50.0


@pytest.mark.parametrize("path", ["tiled", "atomic"])
@pytest.mark.parametrize("name", sorted(KATS))
@pytest.mark.parametrize("size", [(64, 64), (50, 70)])
def test_known_answer_cases(name, size, path, Filler, O):
    v, c, n = KATS[name]
    h, w = size
    # vertices on pixel centres: fov 90, square image -> x_screen = (x/z + 1) * w/2 lands on integers for these inputs
    g, o = Filler(h, w, fov=90.0), O.OracleFiller(h, w, fov=90.0)
    g.render_arrays(v, c, n, path=path)
    o.render_arrays(v, c, n)
    assert_same(buffers(g), buffers(o), name)
    if name == "exact_tie":
        z, col, _ = buffers(g)
        assert (z < 1e5).any() and (col[z < 1e5] > 150.0).all()   # the later copy (colour 200) wins
    if name in ("off_screen", "back_facing", "zero_normal_sum_is_culled"):
        assert (g.get_z_buffer() == np.float32(1e6)).all()


def test_empty_model_and_single_triangle(Filler, O):
    f = Filler(33, 17, fov=60.0)
    e = np.zeros((0, 3, 3), np.float32)
    f.render_arrays(e, e, e)
    assert (f.get_z_buffer() == np.float32(1e6)).all() and not f.get_color_buffer().any()
    v, c, n = KATS["shared_edge"]
    o = O.OracleFiller(33, 17, fov=60.0)
    f.render_arrays(v[:1], c[:1], n[:1])
    o.render_arrays(v[:1], c[:1], n[:1])
    assert_same(buffers(f), buffers(o), "single")


def test_clear_is_fused_and_equals_fresh_filler(Filler, O, trex):
    f = Filler(200, 300, fov=45.0)
    m = random_scene(3)
    f.render_model(m)
    f.clear()
    f.render_model(trex)
    o = O.OracleFiller(200, 300, fov=45.0)
    o.render_model(trex)
    assert_same(buffers(f), buffers(o), "clear+render")
    f.clear()
    assert (f.get_z_buffer() == np.float32(1e6)).all() and not f.get_normals_buffer().any()


def test_pair_list_overflow_is_detected_and_retried(Filler, O):
    # a few hundred full-screen triangles at 512x512: far more (triangle,tile) pairs than the default workspace holds
    T = 600
    v = np.tile(np.array([[[-30, -30, 1.0], [30, -30, 1.0], [0.0, 30, 1.0]]], np.float32), (T, 1, 1))
    v[:, :, 2] += np.linspace(0, 0.5, T, dtype=np.float32)[:, None]
    n = -np.ones((T, 3, 3), np.float32)
    c = np.random.default_rng(0).random((T, 3, 3)).astype(np.float32) * 255
    f, o = Filler(512, 512, fov=90.0), O.OracleFiller(512, 512, fov=90.0)
    f.render_arrays(v, c, n)
    o.render_arrays(v, c, n)
    assert_same(buffers(f), buffers(o), "overflow retry")


def test_api_contract_matches_reference(Filler, trex):
    f = Filler(64, 48, fov=45.0, z_near=0.1, z_far=1000.0, n_threads=8)
    assert f.get_size() == (64, 48)
    z = f.get_z_buffer()
    assert z.dtype == np.float32 and z.shape == (64, 48) and (z == np.float32(1e6)).all()
    assert f.get_color_buffer().shape == (64, 48, 3) and f.get_normals_buffer().shape == (64, 48, 3)
    # live views: same memory on every call, writable, and later renders show through the array already held
    c1 = f.get_color_buffer()
    assert c1 is f.get_color_buffer() and c1.flags.writeable
    v0 = trex._vertices_by_triangles.copy()
    f.render_model(trex)
    assert np.array_equal(v0, trex._vertices_by_triangles)          # the model is never mutated
    assert c1.any() and (z < 1e5).any()
    with pytest.raises(ValueError, match="expected 'float' but got 'double'"):
        f.render_model(TriModel(v0.astype(np.float64), trex._colors_by_triangles, trex._normals_by_triangles))
    with pytest.raises(AttributeError):
        f.render_model(TriModel(v0, None, trex._normals_by_triangles))
    # a vertex with camera z == 0 (stated divergence, DESIGN 2: the reference build prints an unraisable ZeroDivisionError
    # and rasterizes half-projected garbage): that vertex gets IEEE inf / NaN here, host and device inputs alike, and the
    # frame is the one the C oracle (same IEEE arithmetic, no division check) draws
    bad = v0.copy()
    bad[7, 1, 2] = 0.0
    from oracle import oracle as O
    g, o = Filler(1024, 1024, fov=45.0), O.OracleFiller(1024, 1024, fov=45.0)
    g.render_model(TriModel(bad, trex._colors_by_triangles, trex._normals_by_triangles))
    o.render_arrays(bad, trex._colors_by_triangles, trex._normals_by_triangles)
    assert_same(buffers(g), buffers(o), "vertex at z == 0")


def test_host_writes_through_live_views_persist(Filler, O, trex):
    """Renderer.render's pattern (crender/cy/renderer.py:47-49): illumination mutates the colour view in place, the
    next get_color_buffer() shows it, and a later render composites over the mutated buffers."""
    f, o = Filler(96, 96, fov=45.0), O.OracleFiller(96, 96, fov=45.0)
    f.render_model(trex)
    o.render_model(trex)
    for x in (f, o):
        x.get_color_buffer()[...] *= np.float32(0.5)
        x.get_z_buffer()[:10] = np.float32(-5.0)     # nothing can be drawn in front of these rows any more
    assert bits_equal(f.get_color_buffer(), o.get_color_buffer())
    m = random_scene(11)
    f.render_model(m)
    o.render_model(m)
    assert_same(buffers(f), buffers(o), "after host writes")


def test_device_resident_inputs(Filler, O, trex):
    import torch
    f, o = Filler(256, 256, fov=45.0), O.OracleFiller(256, 256, fov=45.0)
    dv, dc, dn = (torch.from_numpy(a).cuda() for a in
                  (trex._vertices_by_triangles, trex._colors_by_triangles, trex._normals_by_triangles))
    f.render_arrays(dv, dc, dn)
    o.render_model(trex)
    assert_same(buffers(f), buffers(o), "device inputs")
    assert f.launch_count >= 4


def test_band_sharded_fillers_concatenate_to_full_frame(Filler, O, trex):
    h, w = 300, 260
    o = O.OracleFiller(h, w, fov=45.0)
    o.render_model(trex)
    parts = []
    for r0, r1 in [(0, 70), (70, 75), (75, 201), (201, 300)]:
        f = Filler(h, w, fov=45.0, band=(r0, r1))
        f.render_model(trex)
        parts.append(buffers(f))
    got = tuple(np.concatenate([p[i] for p in parts], axis=0) for i in range(3))
    assert_same(got, buffers(o), "bands")


@pytest.mark.parametrize("prepass", [1, 0])
def test_band_prepass_switch_changes_nothing(Filler, O, bunny, prepass):
    """CRB_OPT_BAND_PREPASS: with the chunk pre-pass (k_band_chunks + list-walking k_setup / k_fill) or without it, every band
    equals the oracle's rows -- including empty bands, a ragged last chunk, device-resident inputs and repeated frames."""
    import torch
    from cython3dmodelrenderer_b200 import _lib
    h, w = 640, 512
    o = O.OracleFiller(h, w, fov=45.0)
    o.render_model(bunny)
    want = buffers(o)
    dv, dc, dn = (torch.from_numpy(a).cuda() for a in
                  (bunny._vertices_by_triangles, bunny._colors_by_triangles, bunny._normals_by_triangles))
    for r0, r1 in [(0, 32), (32, 288), (288, 320), (320, 608), (608, 640)]:
        f = Filler(h, w, fov=45.0, band=(r0, r1))
        _lib.check(f._L.crb_set_option(f._handle, _lib.CRB_OPT_BAND_PREPASS, prepass))
        for rep in range(2):
            f.clear()
            f.render_arrays(dv, dc, dn)
            assert_same(buffers(f), tuple(a[r0:r1] for a in want), f"band {r0}:{r1} prepass={prepass} frame {rep}")
    # composite of two models into one band (no clear in between)
    f = Filler(h, w, fov=45.0, band=(128, 416))
    _lib.check(f._L.crb_set_option(f._handle, _lib.CRB_OPT_BAND_PREPASS, prepass))
    m2 = random_scene(3, T=5000)
    f.render_arrays(dv, dc, dn)
    f.render_model(m2)
    o.render_model(m2)
    assert_same(buffers(f), tuple(a[128:416] for a in buffers(o)), "band composite")


@pytest.mark.parametrize("seed", [0, 5, 7, 11])
def test_band_prepass_is_conservative_on_odd_vertices(Filler, O, seed):
    """The chunk pre-pass decides with an approximate reciprocal and a widened band; it must never drop a chunk that k_setup
    would draw from.  Random scenes (some behind the camera, some snapped to the pixel grid) salted with vertices that are
    huge, tiny in z, infinite or NaN, cut into thin bands with boundaries the triangles straddle."""
    import torch
    h, w = 256, 192
    m = random_scene(seed, T=6000, span=1.5)
    v = m._vertices_by_triangles
    rng = np.random.default_rng(100 + seed)
    idx = rng.choice(v.shape[0], 60, replace=False)
    odd = np.array([1e30, -1e30, 3e9, -3e9, 1e-30, -1e-30, np.inf, -np.inf, np.nan, 1e-42], dtype=np.float32)
    for j, t in enumerate(idx):
        v[t, j % 3, (j // 3) % 3] = odd[j % len(odd)]
    v[v[..., 2] == 0] += np.float32(0.01)
    o = O.OracleFiller(h, w, fov=60.0)
    o.render_model(m)
    want = buffers(o)
    dv, dc, dn = (torch.from_numpy(a).cuda() for a in (v, m._colors_by_triangles, m._normals_by_triangles))
    for r0, r1 in [(0, 32), (32, 64), (64, 160), (160, 224), (224, 256)]:
        f = Filler(h, w, fov=60.0, band=(r0, r1))
        f.render_arrays(dv, dc, dn)
        assert_same(buffers(f), tuple(a[r0:r1] for a in want), f"seed {seed} band {r0}:{r1}")


def test_guro_on_device_and_u8_output(Filler, O, trex):
    f, o = Filler(200, 200, fov=45.0), O.OracleFiller(200, 200, fov=45.0)
    f.render_model(trex)
    o.render_model(trex)
    light = -np.asarray([0, 0, 1], dtype="float32")
    light = light / np.linalg.norm(light)
    f.illuminate_guro(light)
    O.guro(o.get_color_buffer(), o.get_normals_buffer(), [0, 0, 1])
    assert bits_equal(f.get_color_buffer(), o.get_color_buffer())
    u8 = f.color_u8_flipped().cpu().numpy()
    assert np.array_equal(u8, o.get_color_buffer()[::-1].astype("uint8"))   # run.py:26


def test_batched_views_match_oracle_on_transformed_arrays(Filler, O, trex):
    """C5 parity (SURVEY 8d): per view, the oracle is fed the camera-space arrays the view transform produces."""
    import torch
    from cython3dmodelrenderer_b200 import views as VW
    h, w = 160, 192
    f = Filler(h, w, fov=45.0)
    dv, dc, dn = (torch.from_numpy(a).cuda() for a in
                  (trex._vertices_by_triangles, trex._colors_by_triangles, trex._normals_by_triangles))
    V = 11
    views = VW.orbit_views(V)
    out = f.render_views(dv, dc, dn, views, chunk=4, color_u8_out=True)   # 3 chunks: 4 + 4 + 3
    for k in range(V):
        vk, nk = VW.transform_arrays_host(views[k], trex._vertices_by_triangles, trex._normals_by_triangles)
        gv, gn = f.transform_view(dv, dn, views[k])
        assert bits_equal(gv.cpu().numpy(), vk) and bits_equal(gn.cpu().numpy(), nk)
        o = O.OracleFiller(h, w, fov=45.0)
        o.render_arrays(vk, trex._colors_by_triangles, nk)
        got = (out["z"][k].cpu().numpy(), out["color"][k].cpu().numpy(), out["normals"][k].cpu().numpy())
        assert_same(got, buffers(o), f"view {k}")
        assert np.array_equal(out["color_u8"][k].cpu().numpy(), o.get_color_buffer()[::-1].astype("uint8"))
    assert len({sha(out["z"][k].cpu().numpy()) for k in range(V)}) == V   # the views really differ


def test_batched_views_fused_guro_and_colour_only(Filler, O, trex):
    import torch
    from cython3dmodelrenderer_b200 import views as VW
    h, w = 128, 128
    f = Filler(h, w, fov=45.0)
    dv, dc, dn = (torch.from_numpy(a).cuda() for a in
                  (trex._vertices_by_triangles, trex._colors_by_triangles, trex._normals_by_triangles))
    views = VW.orbit_views(16, first=3, count=3)
    out = f.render_views(dv, dc, dn, views, want=("color",), guro_light=[0, 0, 1])
    assert set(out) == {"color"}
    for k in range(3):
        vk, nk = VW.transform_arrays_host(views[k], trex._vertices_by_triangles, trex._normals_by_triangles)
        o = O.OracleFiller(h, w, fov=45.0)
        o.render_arrays(vk, trex._colors_by_triangles, nk)
        O.guro(o.get_color_buffer(), o.get_normals_buffer(), [0, 0, 1])
        assert bits_equal(out["color"][k].cpu().numpy(), o.get_color_buffer())


def test_fast_division_is_ieee():
    """div_rn_by (reciprocal + two FMA residual steps) must return exactly what the division instruction returns."""
    import ctypes
    from cython3dmodelrenderer_b200 import _lib
    L = _lib.load_library()
    bad, first = ctypes.c_uint64(), (ctypes.c_uint32 * 2)()
    total = 0
    for seed in range(4):
        _lib.check(L.crb_selftest_fdiv(0, 1 << 30, seed * 7919 + 1, ctypes.byref(bad), first))
        total += bad.value
        assert bad.value == 0, f"{bad.value} mismatches, e.g. a={first[0]:#x} d={first[1]:#x}"
    assert total == 0


def test_scaled_sphere_matches_oracle(Filler, O):
    """Config C4 at 1/16 scale (627 200 triangles, 2048^2): full-frame bit compare against the oracle (SURVEY 8d)."""
    from cython3dmodelrenderer_b200 import synthetic
    m = synthetic.uv_sphere(800, 393)
    assert m._vertices_by_triangles.shape[0] == 627200
    f, o = Filler(2048, 2048, fov=45.0), O.OracleFiller(2048, 2048, fov=45.0)
    f.render_model(m)
    o.render_model(m)
    assert int((o.get_z_buffer() < 1e5).sum()) == 2399973      # SURVEY 8d probe of the reference build
    assert_same(buffers(f), buffers(o), "sphere 1/16")


def test_pageable_host_arrays_through_the_staging_ring(Filler, O, trex, monkeypatch):
    """CRB_HOST_PAGEABLE (large NumPy inputs are staged by the library's worker threads through its pinned ring): forced on
    for a small model, two renders composited, arrays mutated right after the call returns (they have been read by then)."""
    monkeypatch.setattr(Filler, "PAGEABLE_MIN_BYTES", 0)
    f, o = Filler(320, 256, fov=45.0), O.OracleFiller(320, 256, fov=45.0)
    v, c, n = (a.copy() for a in (trex._vertices_by_triangles, trex._colors_by_triangles, trex._normals_by_triangles))
    f.render_arrays(v, c, n)
    o.render_arrays(v, c, n)
    v[:] = 0.5; c[:] = 1.0; n[:] = -1.0                 # the frame above must not see this
    m2 = random_scene(11, T=2000)
    f.render_model(m2)
    o.render_model(m2)
    assert_same(buffers(f), buffers(o), "pageable host arrays")


def test_recurring_host_arrays_are_read_in_place(Filler, O, trex):
    """The reference idiom renders the same Model with a new filler per frame: from the third frame on its arrays are page-locked
    in place and read by the GPU directly (crb_host_register, CRB_SYNC_UPLOAD).  Results must not depend on which path ran, and a
    change the caller makes right after render_model returns must show in the next frame, not in this one."""
    from cython3dmodelrenderer_b200 import pixel_buffer_filler as P
    v, c, n = (a.copy() for a in (trex._vertices_by_triangles, trex._colors_by_triangles, trex._normals_by_triangles))
    m = TriModel(v, c, n)
    o = O.OracleFiller(200, 256, fov=45.0)
    o.render_model(m)
    want = buffers(o)
    for frame in range(4):
        f = Filler(200, 256, fov=45.0)
        f.render_model(m)
        if frame == 3:
            assert P._HostArrays.registered.get(v.ctypes.data) == v.nbytes        # frames 2.. read the arrays in place
            keep = c.copy()
            c[:] = 0.0                                                             # after the call returned: not in this frame
            assert_same(buffers(f), want, "frame 3, colours zeroed after render_model")
            c[:] = keep
        else:
            assert_same(buffers(f), want, f"frame {frame}")
    c[:] = c * np.float32(0.5)                                                     # an in-place change is seen by the next frame
    o2 = O.OracleFiller(200, 256, fov=45.0)
    o2.render_model(m)
    f = Filler(200, 256, fov=45.0)
    f.render_model(m)
    assert_same(buffers(f), buffers(o2), "after an in-place change")
    ptr = v.ctypes.data
    del m, v, f
    import gc
    gc.collect()
    assert ptr not in P._HostArrays.registered                                     # released with the array


def test_full_size_sphere_properties(Filler):
    """Config C4 at full size (10 003 200 triangles, 8192^2): too big for a CPU compare in seconds, so size-independent
    properties: band-sharded == unsharded (exact), tiled path == atomic path (exact), re-rendering is idempotent, the
    silhouette is the scaled silhouette of the oracle-checked 1/16 case."""
    import torch
    from cython3dmodelrenderer_b200 import synthetic
    m = synthetic.uv_sphere(3200, 1564)
    T = m._vertices_by_triangles.shape[0]
    assert T == 10003200
    dv, dc, dn = (torch.from_numpy(a).cuda() for a in (m._vertices_by_triangles, m._colors_by_triangles, m._normals_by_triangles))
    f = Filler(8192, 8192, fov=45.0)
    f.render_arrays(dv, dc, dn)
    z, c, n = (t.clone() for t in f.device_buffers())
    cov = z < 1e5
    ys, xs = torch.nonzero(cov, as_tuple=True)
    assert abs(int(cov.sum()) - 16 * 2399973) < 16 * 2399973 * 0.002
    assert (int(xs.min()), int(xs.max()), int(ys.min()), int(ys.max())) == (600, 7592, 600, 7592)
    f.render_arrays(dv, dc, dn)                     # same triangles again: equal depths overwrite with equal values
    z2, c2, n2 = f.device_buffers()
    assert torch.equal(z2.view(torch.int32), z.view(torch.int32)) and torch.equal(c2.view(torch.int32), c.view(torch.int32))
    del f, z2, c2, n2
    g = Filler(8192, 8192, fov=45.0)
    g.render_arrays(dv, dc, dn, path="atomic")
    za, ca, na = g.device_buffers()
    assert torch.equal(za.view(torch.int32), z.view(torch.int32)) and torch.equal(ca.view(torch.int32), c.view(torch.int32)) \
        and torch.equal(na.view(torch.int32), n.view(torch.int32))
    del g, za, ca, na
    for r0, r1 in [(0, 4096), (4096, 8192)]:
        b = Filler(8192, 8192, fov=45.0, band=(r0, r1))
        b.render_arrays(dv, dc, dn)
        zb, cb, nb = b.device_buffers()
        assert torch.equal(zb.view(torch.int32), z[r0:r1].view(torch.int32))
        assert torch.equal(cb.view(torch.int32), c[r0:r1].view(torch.int32))
        assert torch.equal(nb.view(torch.int32), n[r0:r1].view(torch.int32))
        del b


def _sha_dev(t):
    """sha256 of a CUDA tensor's bytes (downloaded in one piece)."""
    return hashlib.sha256(t.contiguous().cpu().numpy().tobytes()).hexdigest()


def test_full_size_sphere_equals_reference_golden(Filler):
    """Config C4 at FULL size (10 003 200 triangles, 8192^2) against the golden the reference build itself rendered
    (tests/golden/make_golden.py, n_threads=1; the C oracle reproduces it in tests/test_oracle_pinning.py): all three
    buffers of the single-GPU frame, and of the frame concatenated from four cost-balanced row bands (what the ranks
    of a band-sharded run hold, SURVEY 8e), bit for bit."""
    import torch
    from cython3dmodelrenderer_b200 import sharding
    info = CHECKS["cases"]["sphere10m_8192x8192_fov45"]
    m, _ = case_model(info)
    assert sha(m._vertices_by_triangles) == info["v_in"] and sha(m._colors_by_triangles) == info["c_in"] \
        and sha(m._normals_by_triangles) == info["n_in"], "the synthetic sphere is not the one the golden was made from"
    dv, dc, dn = (torch.from_numpy(a).cuda() for a in (m._vertices_by_triangles, m._colors_by_triangles, m._normals_by_triangles))
    f = Filler(8192, 8192, fov=45.0)
    f.render_arrays(dv, dc, dn)
    z, c, n = f.device_buffers()
    assert int((z < 1e5).sum()) == info["covered"] == 38399961
    assert (_sha_dev(z), _sha_dev(c), _sha_dev(n)) == (info["z"], info["color"], info["normals"])
    del f, z, c, n
    bands = sharding.balanced_bands(sharding.tile_row_costs(dv, dn, 8192, 8192, 45.0), 4, 8192)
    assert bands[0][0] == 0 and bands[-1][1] == 8192 and all(a[1] == b[0] for a, b in zip(bands, bands[1:]))
    parts = []
    for r0, r1 in bands:
        b = Filler(8192, 8192, fov=45.0, band=(r0, r1))
        b.render_arrays(dv, dc, dn)
        parts.append(tuple(t.cpu() for t in b.device_buffers()))
        del b
    for k, name in enumerate(("z", "color", "normals")):
        whole = torch.cat([p[k] for p in parts], dim=0)
        assert hashlib.sha256(whole.numpy().tobytes()).hexdigest() == info[name], f"band-concatenated {name}"


def test_orbit_views_at_1024_equal_reference_goldens(Filler, trex):
    """Config C5 at its real size: evenly spread views of the 1024^2 T-Rex orbit, rendered the way bench.py renders
    them (one render_views call, 128 views per launch, GPU view transform), against goldens the reference build rendered
    from the camera-space arrays of the same views (tests/golden/make_golden.py)."""
    import torch
    from cython3dmodelrenderer_b200 import views as VW
    dv, dc, dn = (torch.from_numpy(a).cuda() for a in
                  (trex._vertices_by_triangles, trex._colors_by_triangles, trex._normals_by_triangles))
    f = Filler(1024, 1024, fov=45.0)
    out = f.render_views(dv, dc, dn, VW.orbit_views(128), chunk=128)
    checked = 0
    for key, info in sorted(CHECKS["cases"].items()):
        if info.get("orbit") != 128:
            continue
        k = info["view"]
        assert int((out["z"][k] < 1e5).sum()) == info["covered"], key
        assert (_sha_dev(out["z"][k]), _sha_dev(out["color"][k]), _sha_dev(out["normals"][k])) == \
            (info["z"], info["color"], info["normals"]), key
        checked += 1
    assert checked == 4
    del out
    # two views of the 1024-view orbit (config C5's own view count), as a rank of an 8-GPU run would render them
    ks = sorted(info["view"] for info in CHECKS["cases"].values() if info.get("orbit") == 1024)
    views = np.stack([VW.orbit_views(1024, first=k, count=1)[0] for k in ks])
    out = f.render_views(dv, dc, dn, views, chunk=2)
    for i, k in enumerate(ks):
        info = CHECKS["cases"][f"trex_orbit1024_view{k}_1024x1024_fov45"]
        assert (_sha_dev(out["z"][i]), _sha_dev(out["color"][i]), _sha_dev(out["normals"][i])) == \
            (info["z"], info["color"], info["normals"]), k


@pytest.mark.parametrize("mode", ["tma", "tma_vec_rows", "tma_direct_rows", "plain", "tiny_grid", "tma_tiny_grid"])
@pytest.mark.parametrize("size", [(96, 128), (100, 76), (50, 36), (257, 388), (64, 30)])
def test_fused_clear_store_paths(mode, size, Filler, O):
    """clear()+render takes the store path the layout allows: TMA boxes (rows that are 16-byte multiples), clipped by
    the hardware on partial tiles, or plain stores (W % 4 != 0, CRB_OPT_TMA off); a grid smaller than the number of busy
    tiles makes k_raster walk several tiles per CTA (CRB_OPT_RASTER_CTAS).  All of them must give the oracle's bits."""
    from cython3dmodelrenderer_b200 import _lib
    h, w = size
    for seed in (3, 5, 8):
        m = random_scene(seed, T=300)
        g, o = Filler(h, w, fov=60.0), O.OracleFiller(h, w, fov=60.0)
        g.set_option(_lib.CRB_OPT_TMA, 0 if mode in ("plain", "tiny_grid") else 1)
        g.set_option(_lib.CRB_OPT_TMA_ROWS, {"tma_vec_rows": 0, "tma_direct_rows": 2}.get(mode, 1))
        if "tiny_grid" in mode:
            g.set_option(_lib.CRB_OPT_RASTER_CTAS, 3)
        g.render_model(random_scene(seed + 50, T=40))      # stale contents the fused clear must wipe
        g.clear()
        for _ in range(2):                                 # second frame: grid sized from the first frame's statistics
            g.clear()
            g.render_model(m)
        o.render_model(m)
        assert_same(buffers(g), buffers(o), f"{mode} {h}x{w} seed {seed}")


def test_batched_views_partial_outputs_tma(Filler, O, trex):
    """render_views with only some of the three arrays requested (maps exist only for those)."""
    import torch
    from cython3dmodelrenderer_b200 import views as VW
    h, w = 96, 160
    dv, dc, dn = (torch.from_numpy(a).cuda() for a in
                  (trex._vertices_by_triangles, trex._colors_by_triangles, trex._normals_by_triangles))
    views = VW.orbit_views(8, first=1, count=3)
    f = Filler(h, w, fov=45.0)
    full = f.render_views(dv, dc, dn, views)
    for want in (("z",), ("color",), ("normals", "z")):
        part = f.render_views(dv, dc, dn, views, want=want)
        assert set(part) == set(want)
        for name in want:
            assert torch.equal(part[name].view(torch.int32), full[name].view(torch.int32)), (want, name)
    vk, nk = VW.transform_arrays_host(views[2], trex._vertices_by_triangles, trex._normals_by_triangles)
    o = O.OracleFiller(h, w, fov=45.0)
    o.render_arrays(vk, trex._colors_by_triangles, nk)
    assert_same(tuple(full[k][2].cpu().numpy() for k in ("z", "color", "normals")), buffers(o), "view 2")


@pytest.mark.parametrize("sparse", [True, False])
def test_host_frame_pipeline_matches_oracle(sparse, O, trex):
    """Pipelined host-buffer frames (crb_render_host + CRB_NO_SYNC over several fillers) give per frame the oracle's
    fresh-filler result, in submission order, for NumPy and pinned-tensor inputs alike."""
    import torch
    from cython3dmodelrenderer_b200 import HostFramePipeline, views as VW
    h, w = 192, 256
    pipe = HostFramePipeline(h, w, fov=45.0, depth=3, sparse=sparse)
    views = VW.orbit_views(7)
    frames = [VW.transform_arrays_host(views[k], trex._vertices_by_triangles, trex._normals_by_triangles) for k in range(7)]
    want = []
    for vk, nk in frames:
        o = O.OracleFiller(h, w, fov=45.0)
        o.render_arrays(vk, trex._colors_by_triangles, nk)
        want.append(buffers(o))
    pending = []
    got = [None] * 7
    for k, (vk, nk) in enumerate(frames):
        if k % 2:
            args = [torch.from_numpy(a).pin_memory() for a in (vk, trex._colors_by_triangles, nk)]
        else:
            args = [vk, trex._colors_by_triangles, nk]
        pending.append((k, pipe.submit(*args), args))
        if len(pending) == 3:
            kk, slot, _ = pending.pop(0)
            r = pipe.result(slot)
            got[kk] = (r["z"].copy(), r["color"].copy(), r["normals"].copy())
    for kk, slot, _ in pending:
        r = pipe.result(slot)
        got[kk] = (r["z"].copy(), r["color"].copy(), r["normals"].copy())
    for k in range(7):
        assert_same(got[k], want[k], f"pipelined frame {k}")


@pytest.mark.parametrize("lit", [False, True])
def test_host_image_pipeline_matches_run_py(lit, O, trex):
    """HostImagePipeline (N3): pinned [3,T,3,3] block in, run.py:26's `image[::-1].astype('uint8')` out (with
    GuroIllumination, renderer.py:48, when a light is given) -- equal to the oracle's frame converted the reference's way,
    for a sequence of different views through three slots."""
    import torch
    from cython3dmodelrenderer_b200 import HostImagePipeline, views as VW
    h, w = 160, 224
    pipe = HostImagePipeline(h, w, fov=45.0, depth=3, light=[0, 0, 1] if lit else None)
    views = VW.orbit_views(7)
    frames, want = [], []
    for k in range(7):
        vk, nk = VW.transform_arrays_host(views[k], trex._vertices_by_triangles, trex._normals_by_triangles)
        frames.append(torch.from_numpy(np.stack([vk, trex._colors_by_triangles, nk])).pin_memory())
        o = O.OracleFiller(h, w, fov=45.0)
        o.render_arrays(vk, trex._colors_by_triangles, nk)
        if lit:
            O.guro(o.get_color_buffer(), o.get_normals_buffer(), [0, 0, 1])
        want.append(o.get_color_buffer()[::-1].astype("uint8"))
    pending, got = [], [None] * 7
    for k in range(7):
        pending.append((k, pipe.submit(frames[k])))
        if len(pending) == 3:
            kk, slot = pending.pop(0)
            got[kk] = pipe.result(slot).copy()
    for kk, slot in pending:
        got[kk] = pipe.result(slot).copy()
    for k in range(7):
        assert np.array_equal(got[k], want[k]), f"image {k}"
    # a frame whose (triangle,tile) pairs do not fit the default list: detected from the status words that come back with
    # the image, the list is grown and the frame drawn again
    T = 600
    v = np.tile(np.array([[[-30, -30, 1.0], [30, -30, 1.0], [0.0, 30, 1.0]]], np.float32), (T, 1, 1))
    v[:, :, 2] += np.linspace(0, 0.5, T, dtype=np.float32)[:, None]
    n = -np.ones((T, 3, 3), np.float32)
    c = np.random.default_rng(0).random((T, 3, 3)).astype(np.float32) * 255
    big = HostImagePipeline(512, 512, fov=90.0, depth=2, light=[0, 0, 1] if lit else None)
    o = O.OracleFiller(512, 512, fov=90.0)
    o.render_arrays(v, c, n)
    if lit:
        O.guro(o.get_color_buffer(), o.get_normals_buffer(), [0, 0, 1])
    block = torch.from_numpy(np.stack([v, c, n])).pin_memory()
    for rep in range(3):
        img = big.result(big.submit(block))
        assert np.array_equal(img, o.get_color_buffer()[::-1].astype("uint8")), f"overflowing frame, pass {rep}"


@pytest.mark.parametrize("size", [(96, 128), (100, 76), (50, 37), (257, 388)])
def test_sparse_readback_equals_full_download(size, O):
    """CRB_DL_SPARSE: a sequence of unrelated fresh frames through ONE slot (so every frame's host arrays start from the
    previous frame's content) -- small scenes that leave most tiles empty, an empty scene, a dense one -- must leave the
    host arrays bit-identical to the oracle's fresh-filler result each time, while copying fewer tiles than a dense
    download would."""
    from cython3dmodelrenderer_b200 import HostFramePipeline
    h, w = size
    pipe = HostFramePipeline(h, w, fov=60.0, depth=1, sparse=True)
    tiles = ((h + 31) // 32) * ((w + 31) // 32)
    scenes = [random_scene(11, T=6, span=0.3), random_scene(12, T=300), random_scene(13, T=0), random_scene(14, T=3, span=0.2),
              random_scene(15, T=2000, span=0.8), random_scene(16, T=5, span=0.5)]
    copied = []
    for k, m in enumerate(scenes):
        slot = pipe.submit(m._vertices_by_triangles, m._colors_by_triangles, m._normals_by_triangles)
        r = pipe.result(slot)
        o = O.OracleFiller(h, w, fov=60.0)
        o.render_model(m)
        assert_same((r["z"], r["color"], r["normals"]), buffers(o), f"sparse frame {k} {h}x{w}")
        assert not r["z"].flags.writeable
        copied.append(pipe.readback_tiles())
    assert all(c <= tiles for c in copied)
    assert copied[2] <= tiles and copied[3] < tiles or tiles <= 4      # tiny scenes after an empty one copy few tiles


def test_chunk_pipeline_and_tma_switches_do_not_change_results(Filler, trex):
    """crb_set_option: the two-stream launch pipeline (two workspace sets) and the TMA stores are tuning switches."""
    import torch
    from cython3dmodelrenderer_b200 import _lib, views as VW
    h, w = 128, 160
    dv, dc, dn = (torch.from_numpy(a).cuda() for a in
                  (trex._vertices_by_triangles, trex._colors_by_triangles, trex._normals_by_triangles))
    views = VW.orbit_views(9)
    ref = None
    for pipe, tma in ((1, 1), (0, 1), (1, 0), (0, 0)):
        f = Filler(h, w, fov=45.0)
        _lib.check(f._L.crb_set_option(f._handle, _lib.CRB_OPT_CHUNK_PIPELINE, pipe))
        _lib.check(f._L.crb_set_option(f._handle, _lib.CRB_OPT_TMA, tma))
        for _ in range(2):      # twice: the second batch reuses both workspace sets
            out = f.render_views(dv, dc, dn, views, chunk=2)
        got = {k: out[k].cpu().numpy().view(np.uint32) for k in ("z", "color", "normals")}
        if ref is None:
            ref = got
        else:
            for k in ref:
                assert np.array_equal(ref[k], got[k]), (pipe, tma, k)


def test_integration_stub_flow_without_torch(O, trex):
    """INTEGRATION.md section 2: a maintainer's ctypes binding -- crb_create, crb_alloc_owned (library-owned device
    memory), crb_render_host with plain (pageable) NumPy arrays in and out, compositing two calls -- no torch anywhere."""
    import ctypes
    from cython3dmodelrenderer_b200 import _lib
    L = _lib.load_library()
    h, w = 200, 240
    f = ctypes.c_void_p()
    _lib.check(L.crb_create(h, w, 45.0, 0.1, 1000.0, 0, ctypes.byref(f)))
    try:
        v, c, n = (np.ascontiguousarray(a) for a in (trex._vertices_by_triangles, trex._colors_by_triangles, trex._normals_by_triangles))
        _lib.check(L.crb_alloc_owned(f, v.shape[0], 1, 0))
        z = np.empty((h, w), np.float32); col = np.empty((h, w, 3), np.float32); nrm = np.empty((h, w, 3), np.float32)
        o = O.OracleFiller(h, w, fov=45.0)
        for rep in range(2):                     # the second call composites into the first (equal depths overwrite)
            half = slice(0, v.shape[0] // 2) if rep == 0 else slice(None)
            _lib.check(L.crb_render_host(f, v[half].ctypes.data, c[half].ctypes.data, n[half].ctypes.data, v[half].shape[0], 0,
                                         _lib.CRB_BUF_ALL, z.ctypes.data, col.ctypes.data, nrm.ctypes.data, None))
            o.render_arrays(v[half], c[half], n[half])
            assert_same((z, col, nrm), buffers(o), f"stub call {rep}")
        need, cap = ctypes.c_int64(), ctypes.c_int64()
        _lib.check(L.crb_status(f, ctypes.byref(need), ctypes.byref(cap), None))
        assert 0 < need.value <= cap.value
    finally:
        L.crb_destroy(f)


@pytest.mark.parametrize("split", ["1", "0"])
def test_single_view_heavy_tile_split(split, Filler, O):
    """Single-view launches cut tiles with many triangles into four 8-row bands rasterized by different CTAs
    (CRB_OPT_SPLIT_HEAVY); fresh and compositing renders, partial tiles at the image edge."""
    from cython3dmodelrenderer_b200 import _lib
    for (h, w), seed in (((96, 128), 21), ((75, 100), 22), ((40, 33), 23)):
        m = random_scene(200 + seed, T=5000, span=0.5)          # hundreds of triangles per tile
        g, o = Filler(h, w, fov=70.0), O.OracleFiller(h, w, fov=70.0)
        g.set_option(_lib.CRB_OPT_SPLIT_HEAVY, int(split))
        g.clear()
        g.render_model(m)                                       # fused clear, TMA where the layout allows
        o.render_model(m)
        assert_same(buffers(g), buffers(o), f"split={split} fresh {h}x{w}")
        m2 = random_scene(300 + seed, T=3000, span=0.7)
        g.render_model(m2)                                      # composites into the first frame
        o.render_model(m2)
        assert_same(buffers(g), buffers(o), f"split={split} composite {h}x{w}")


def test_deferred_join_batches_match_joined_batches(Filler, trex):
    """CRB_DEFER_JOIN: back-to-back batches whose front end overlaps the previous batch's rasterizer (alternating
    workspace sets across calls) give the same slabs as joined calls; other entry points join by themselves."""
    import torch
    from cython3dmodelrenderer_b200 import views as VW
    h, w = 128, 160
    dv, dc, dn = (torch.from_numpy(a).cuda() for a in
                  (trex._vertices_by_triangles, trex._colors_by_triangles, trex._normals_by_triangles))
    batches = [VW.orbit_views(12, first=3 * k, count=3) for k in range(4)]
    f = Filler(h, w, fov=45.0)
    want = [{k: t.clone() for k, t in f.render_views(dv, dc, dn, b, chunk=3).items()} for b in batches]
    g = Filler(h, w, fov=45.0)
    outs = []
    for b in batches:
        outs.append(g.render_views(dv, dc, dn, b, chunk=3, check_status=False, defer_join=True))
    g.join()
    for k, (o, wnt) in enumerate(zip(outs, want)):
        for name in ("z", "color", "normals"):
            assert torch.equal(o[name].view(torch.int32), wnt[name].view(torch.int32)), (k, name)
    # an entry point that is not render_views joins on its own: the composited frame sees the finished batch state
    o2 = g.render_views(dv, dc, dn, batches[0], chunk=3, check_status=False, defer_join=True)
    g.clear(); g.render_arrays(dv, dc, dn)        # crb_render + crb_status join first
    z, c, n = g.device_buffers()
    assert int((z < 1e5).sum()) > 100 and torch.equal(o2["z"].view(torch.int32), want[0]["z"].view(torch.int32))


def flow_sums(image, filler):
    """Checksums of what run.py takes from one Renderer.render: the lit colour buffer, the uint8 image cv2.imwrite would
    write (run.py:26), and the filler's normals and depth."""
    z = filler.get_z_buffer()
    return {"covered": int((z < 1e5).sum()), "image": sha(image), "u8": sha(image[::-1].astype("uint8")),
            "normals": sha(filler.get_normals_buffer()), "z": sha(z)}


def _reference_flow_classes():
    """The reference's own Renderer / illumination / filler / iterator classes where oracle/_ref is present, else None."""
    from oracle import build_ref
    if not build_ref.built():
        return None
    import sys
    from conftest import ROOT
    ref = os.path.join(ROOT, "oracle", "_ref")
    if ref not in sys.path:
        sys.path.insert(0, ref)
    from crender.cy import Renderer
    from crender.cy.illumination import GuroIllumination, NoIllumination
    from crender.cy.pixel_buffer_filler import AdvancedPixelBufferFiller
    from crender.cy.triangle_iterator import SimpleIterator
    return Renderer, GuroIllumination, NoIllumination, AdvancedPixelBufferFiller, SimpleIterator


def test_reference_renderer_flow_with_the_drop_in_filler(Filler, trex, capfd):
    """The run.py flow (run.py:20-26) driving this filler, against the reference flow's buffers (tests/golden/
    make_golden_seeded.py): with this package's Renderer and GuroIllumination, and -- where oracle/_ref is present -- with
    the reference's OWN Renderer and GuroIllumination classes (crender/cy/renderer.py:42-49: render_model, in-place
    illumination on the live views, get_color_buffer), next to the same flow on the reference's own Cython filler."""
    import cython3dmodelrenderer_b200 as P
    h = w = 256
    light = np.array([0, 0, 1], dtype="float32")
    flows = [(Filler, P.Renderer, P.GuroIllumination, None)]
    ref = _reference_flow_classes()
    if ref is not None:
        RefRenderer, RefGuro, _, RefFiller, SimpleIterator = ref
        flows += [(RefFiller, RefRenderer, RefGuro, SimpleIterator), (Filler, RefRenderer, RefGuro, SimpleIterator)]
    for fcls, rcls, ill, it in flows:
        filler = fcls(h, w, fov=45, n_threads=1)
        image = rcls(filler, ill(light), it, h, w).render(trex)
        capfd.readouterr()
        got = flow_sums(image, filler)
        assert got["covered"] > 5000
        assert got == seeded("renderer_flow_trex_256x256_guro"), f"{fcls.__module__}.{rcls.__name__}: differs from the reference flow"


def test_drop_in_renderer_and_illumination_match_the_reference_flow(Filler, trex, bunny, capfd):
    """run.py:20-26 over two render() calls on the same filler (the second composites onto the lit frame and lights the whole
    buffer again, renderer.py:47-49), against the reference flow's buffers (tests/golden/make_golden_seeded.py): this package's
    Renderer + GuroIllumination + filler, and -- where oracle/_ref is present -- the reference's own classes on its own
    Cython filler and the reference's Renderer driving this package's filler AND GuroIllumination (draw_illumination
    recognises the filler's live views and lights the device buffers): bit-identical images, normals and depth."""
    import cython3dmodelrenderer_b200 as P
    h, w = 320, 256
    light = [0.3, -0.2, 1.0]
    ref = _reference_flow_classes()
    for kind, our_ill in (("guro", lambda: P.GuroIllumination(light)), ("none", P.NoIllumination)):
        flows = [(Filler, P.Renderer, our_ill, None)]
        if ref is not None:
            RefRenderer, RefGuro, RefNone, RefFiller, SimpleIterator = ref
            ref_ill = (lambda: RefGuro(light)) if kind == "guro" else RefNone
            flows += [(RefFiller, RefRenderer, ref_ill, SimpleIterator), (Filler, RefRenderer, our_ill, SimpleIterator)]
        for fcls, rcls, ill, it in flows:
            filler = fcls(h, w, fov=45, n_threads=1)
            renderer = rcls(filler, ill(), it, h, w)
            for k, m in enumerate((trex, bunny)):
                image = renderer.render(m)
                if fcls is Filler:
                    assert image is filler.get_color_buffer()      # the live view, the same object every time
                capfd.readouterr()
                got = flow_sums(image, filler)
                assert got["covered"] > 5000
                assert got == seeded("renderer_flow_trex_bunny_320x256")[kind][k], \
                    f"{kind}, render {k}, {fcls.__module__}.{rcls.__name__}: differs from the reference flow"
    # arrays that are not the live views of a filler of this package: no NumPy path here
    with pytest.raises(TypeError):
        P.GuroIllumination(light).draw_illumination(np.zeros((h, w, 3), np.float32), np.zeros((h, w, 3), np.float32))
    f = Filler(h, w, fov=45)
    f.render_model(trex)
    with pytest.raises(TypeError):      # (a copy is not the view)
        P.GuroIllumination(light).draw_illumination(f.get_color_buffer().copy(), f.get_normals_buffer())


@pytest.mark.parametrize("case", sorted(k for k in CHECKS["cases"] if k.endswith("_guro")))
def test_reference_golden_lit_colour(case, Filler, trex, bunny, basketball):
    """The reference's Renderer.render + GuroIllumination result (golden checksum of the lit colour buffer), three ways:
    NumPy illumination on the live host views, crb_guro on the device buffers, and CRB_GURO fused into shading."""
    import torch
    from cython3dmodelrenderer_b200 import views as VW
    info = CHECKS["cases"][case]
    m = {"trex": trex, "bunny": bunny, "basketball": basketball}[info["model"]]
    light = -np.asarray(info["light"], dtype="float32")
    light = light / np.linalg.norm(light)
    f = Filler(info["h"], info["w"], fov=info["fov"])
    f.render_model(m)
    assert int((f.get_z_buffer() < 1e5).sum()) == info["covered"]
    f.illuminate_guro(light)
    assert sha(f.get_color_buffer()) == info["color_lit"]
    dv, dc, dn = (torch.from_numpy(a).cuda() for a in (m._vertices_by_triangles, m._colors_by_triangles, m._normals_by_triangles))
    out = f.render_views(dv, dc, dn, VW.view_matrix()[None, :], want=("color",), guro_light=info["light"])
    assert sha(out["color"][0].cpu().numpy()) == info["color_lit"]
    # ... and a fourth: this package's Renderer + GuroIllumination (renderer.py / illumination.py: the run.py flow with the
    # illumination on the device buffers, only the lit colour crossing PCIe)
    from cython3dmodelrenderer_b200 import GuroIllumination, Renderer
    f2 = Filler(info["h"], info["w"], fov=info["fov"])
    image = Renderer(f2, GuroIllumination(info["light"]), None, info["h"], info["w"]).render(m)
    assert image is f2.get_color_buffer() and sha(image) == info["color_lit"]


def test_repeated_renders_are_bit_identical(Filler, trex):
    """Determinism under load (a stand-in for racecheck): the same dense frame and the same batch of views rendered many
    times, with the fused clear, must give the same bits every time."""
    import torch
    from cython3dmodelrenderer_b200 import views as VW
    m = random_scene(77, T=20000, span=0.6)
    dv, dc, dn = (torch.from_numpy(a).cuda() for a in (m._vertices_by_triangles, m._colors_by_triangles, m._normals_by_triangles))
    f = Filler(512, 512, fov=70.0)
    ref = None
    for it in range(25):
        f.clear()
        f.render_arrays(dv, dc, dn, check_status=(it == 0))
        z, c, n = f.device_buffers()
        cur = (z.clone(), c.clone(), n.clone())
        if ref is None:
            ref = cur
        else:
            for a, b in zip(ref, cur):
                assert torch.equal(a.view(torch.int32), b.view(torch.int32)), f"iteration {it}"
    tv, tc, tn = (torch.from_numpy(a).cuda() for a in (trex._vertices_by_triangles, trex._colors_by_triangles, trex._normals_by_triangles))
    g = Filler(256, 256, fov=45.0)
    views = VW.orbit_views(24)
    first = {k: t.clone() for k, t in g.render_views(tv, tc, tn, views, chunk=8).items()}
    for it in range(10):
        out = g.render_views(tv, tc, tn, views, chunk=8, check_status=False, defer_join=(it % 2 == 0))
        g.join()
        for k in first:
            assert torch.equal(first[k].view(torch.int32), out[k].view(torch.int32)), (it, k)


@pytest.mark.parametrize("size", [(1, 1), (1, 37), (33, 1), (2, 3), (31, 32), (32, 33)])
def test_degenerate_image_sizes(size, Filler, O):
    h, w = size
    for seed in (1, 2):
        m = random_scene(400 + seed, T=50)
        g, o = Filler(h, w, fov=60.0), O.OracleFiller(h, w, fov=60.0)
        g.clear()
        g.render_model(m)
        o.render_model(m)
        assert_same(buffers(g), buffers(o), f"{h}x{w} seed {seed}")


@pytest.mark.parametrize("wide_kernel", [1, 0])
def test_screen_filling_triangles_and_one_crowded_tile(wide_kernel, Filler, O):
    """Two extremes of the binning: triangles that cover every tile of a 1536x1024 frame (thousands of tiles per triangle;
    scattered by k_fill_wide, or -- option off, and in the second frame of the first case's filler if that frame had none -- by
    k_fill itself), and 30 000 small triangles inside a single tile (one list far longer than a staging batch, heavy-tile bands)."""
    rng = np.random.default_rng(5)
    big = np.array([[[-30, -30, 2.0], [30, -30, 2.0], [0, 40, 2.0]],
                    [[-25, 25, 1.5], [0, -35, 1.5], [25, 25, 1.5]],
                    [[-1.0, -1.0, 1.0], [1.0, -1.0, 3.0], [0.0, 1.2, 0.5]]], dtype=np.float32)
    nb = -np.abs(rng.standard_normal((3, 3, 3))).astype(np.float32)
    cb = (rng.random((3, 3, 3)) * 255).astype(np.float32)
    T = 30000
    ctr = np.array([0.2, -0.1, 1.0], dtype=np.float32) + rng.uniform(-0.008, 0.008, (T, 1, 3)).astype(np.float32) * np.float32([1, 1, 20])
    small = (ctr + rng.uniform(-0.004, 0.004, (T, 3, 3)).astype(np.float32) * np.float32([1, 1, 0])).astype(np.float32)
    ns = -np.abs(rng.standard_normal((T, 3, 3))).astype(np.float32)
    cs = (rng.random((T, 3, 3)) * 255).astype(np.float32)
    m = TriModel(np.concatenate([big, small]), np.concatenate([cb, cs]), np.concatenate([nb, ns]))
    h, w = 1024, 1536
    from cython3dmodelrenderer_b200 import _lib
    g, o = Filler(h, w, fov=45.0), O.OracleFiller(h, w, fov=45.0)
    g.set_option(_lib.CRB_OPT_WIDE_KERNEL, wide_kernel)
    g.clear()
    g.render_model(m)
    o.render_model(m)
    assert int((o.get_z_buffer() < 1e5).sum()) > h * w // 2
    assert_same(buffers(g), buffers(o), "big + crowded")
    # a frame without wide triangles, then the wide ones again: the launch decision follows the previous frame's report, the
    # result must not
    ms = TriModel(small, cs, ns)
    for model in (ms, m):
        g.clear()
        g.render_model(model)
        o = O.OracleFiller(h, w, fov=45.0)
        o.render_model(model)
        assert_same(buffers(g), buffers(o), "after a frame without wide triangles")


def test_render_host_overflow_is_never_silent(O, trex):
    """Synchronous crb_render_host: with a library-owned workspace an undersized pair list is grown and the frame drawn
    again; with a caller-owned workspace the call returns CRB_ERR_OVERFLOW and leaves the buffers untouched."""
    import ctypes
    import torch
    from cython3dmodelrenderer_b200 import _lib
    L = _lib.load_library()
    h, w = 160, 200
    v, c, n = (np.ascontiguousarray(a) for a in (trex._vertices_by_triangles, trex._colors_by_triangles, trex._normals_by_triangles))
    T = v.shape[0]
    o = O.OracleFiller(h, w, fov=45.0)
    o.render_arrays(v, c, n)
    z = np.empty((h, w), np.float32); col = np.empty((h, w, 3), np.float32); nrm = np.empty((h, w, 3), np.float32)
    f = ctypes.c_void_p()
    _lib.check(L.crb_create(h, w, 45.0, 0.1, 1000.0, 0, ctypes.byref(f)))
    try:
        _lib.check(L.crb_alloc_owned(f, T, 1, 64))                    # room for 64 pairs: far too small
        _lib.check(L.crb_render_host(f, v.ctypes.data, c.ctypes.data, n.ctypes.data, T, _lib.CRB_CLEAR_FIRST, _lib.CRB_BUF_ALL,
                                     z.ctypes.data, col.ctypes.data, nrm.ctypes.data, None))
        assert_same((z, col, nrm), buffers(o), "library-owned workspace grown")
    finally:
        L.crb_destroy(f)
    g = ctypes.c_void_p()
    _lib.check(L.crb_create(h, w, 45.0, 0.1, 1000.0, 0, ctypes.byref(g)))
    try:
        bz = torch.full((h, w), 7.0, device="cuda"); bc = torch.full((h, w, 3), 7.0, device="cuda"); bn = torch.full((h, w, 3), 7.0, device="cuda")
        _lib.check(L.crb_bind_buffers(g, bz.data_ptr(), bc.data_ptr(), bn.data_ptr()))
        nbytes = L.crb_workspace_bytes(g, T, 1, 64)
        ws = torch.empty(nbytes + 256, dtype=torch.uint8, device="cuda")
        _lib.check(L.crb_bind_workspace(g, (ws.data_ptr() + 255) // 256 * 256, nbytes, T, 1, 64, None))
        rc = L.crb_render_host(g, v.ctypes.data, c.ctypes.data, n.ctypes.data, T, _lib.CRB_CLEAR_FIRST, 0, None, None, None, None)
        assert rc == _lib.CRB_ERR_OVERFLOW
        assert b"pairs" in L.crb_last_error()
        torch.cuda.synchronize()
        assert float(bz.min()) == 7.0 and float(bc.max()) == 7.0       # frame not drawn, not even cleared
    finally:
        L.crb_destroy(g)


@pytest.mark.parametrize("shape", [1, 2, 3], ids=["large", "small", "wide"])
def test_both_rasterizer_shapes_bit_exact(shape, Filler, O, trex):
    """The tile rasterizer exists in three CTA shapes (CRB_OPT_RASTER_SHAPE: 128 threads / 96 staged triangles, 128 threads / 24
    staged triangles, 256 threads / 128 staged triangles), picked per launch from the posted statistics; forced here, each must
    give the oracle's bits on every kind of frame: fresh and compositing, light and crowded tiles (several staging passes),
    heavy tiles cut into row bands, known-answer cases, partial tiles, batched views with every output kind."""
    from cython3dmodelrenderer_b200 import _lib, views as VW
    import torch

    def filler(h, w, fov):
        g = Filler(h, w, fov=fov)
        g.set_option(_lib.CRB_OPT_RASTER_SHAPE, shape)
        return g
    for seed in range(8):
        rng = np.random.default_rng(4000 + seed)
        h, w, fov = int(rng.integers(8, 200)), int(rng.integers(8, 200)), float(rng.uniform(20, 120))
        m = random_scene(seed)
        g, o = filler(h, w, fov), O.OracleFiller(h, w, fov=fov)
        for _ in range(2 if seed % 3 == 0 else 1):
            g.render_model(m)
            o.render_model(m)
        assert_same(buffers(g), buffers(o), f"shape {shape} seed {seed} {h}x{w}")
    for (h, w), seed in (((257, 391), 100), ((96, 128), 221)):      # dense: hundreds of triangles per tile, split heavy tiles
        m = random_scene(seed, T=5000, span=0.55)
        g, o = filler(h, w, 70.0), O.OracleFiller(h, w, fov=70.0)
        g.clear(); g.render_model(m); o.render_model(m)
        assert_same(buffers(g), buffers(o), f"shape {shape} dense {h}x{w}")
        m2 = random_scene(300 + seed, T=2000, span=0.7)
        g.render_model(m2); o.render_model(m2)
        assert_same(buffers(g), buffers(o), f"shape {shape} dense composite {h}x{w}")
    for name in sorted(KATS):
        v, c, n = KATS[name]
        g, o = filler(50, 70, 90.0), O.OracleFiller(50, 70, fov=90.0)
        g.render_arrays(v, c, n); o.render_arrays(v, c, n)
        assert_same(buffers(g), buffers(o), f"shape {shape} {name}")
    info = CHECKS["cases"]["trex_1024x1024_fov45"]
    g = filler(1024, 1024, 45.0)
    g.render_model(trex)
    assert (sha(g.get_z_buffer()), sha(g.get_color_buffer()), sha(g.get_normals_buffer())) == (info["z"], info["color"], info["normals"])
    # batched views: float32 slabs, the flipped uint8 image, fused Guro -- against the other shape's bits and the oracle's first view
    dv, dc, dn = (torch.from_numpy(a).cuda() for a in (trex._vertices_by_triangles, trex._colors_by_triangles, trex._normals_by_triangles))
    vw = VW.orbit_views(12, first=0, count=5)
    outs = {}
    for sh in (1, 2, 3):
        g = Filler(160, 192, fov=45.0)
        g.set_option(_lib.CRB_OPT_RASTER_SHAPE, sh)
        r = g.render_views(dv, dc, dn, vw, color_u8_out=True, chunk=2)
        lit = g.render_views(dv, dc, dn, vw, want=("color",), guro_light=[0.3, -0.2, 1.0], color_u8_out=True, chunk=5)
        torch.cuda.synchronize()
        outs[sh] = [r[k].cpu().numpy() for k in ("z", "color", "normals", "color_u8")] + [lit["color"].cpu().numpy(), lit["color_u8"].cpu().numpy()]
    for other in (1, 2, 3):
        for a, b in zip(outs[shape], outs[other]):
            assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
    vk, nk = VW.transform_arrays_host(vw[0], trex._vertices_by_triangles, trex._normals_by_triangles)
    o = O.OracleFiller(160, 192, fov=45.0)
    o.render_arrays(vk, trex._colors_by_triangles, nk)
    assert_same(tuple(outs[shape][k][0] for k in range(3)), buffers(o), f"shape {shape} view 0")
