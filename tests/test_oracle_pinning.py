"""The CPU oracle (oracle/crender_oracle.c) against the reference: committed golden vectors that the reference's
own Cython build produced (tests/golden/make_golden.py), hand-derived known answers, and -- wherever oracle/_ref
is present -- the reference build itself on seeded random scenes.  CPU only."""
import hashlib
import json
import os
import sys

import numpy as np
import pytest

from conftest import GOLDEN, ROOT, TriModel, bits_equal, case_model, load_indexed, random_scene
from oracle import build_ref
from oracle import oracle as O

CHECKS = json.load(open(os.path.join(GOLDEN, "checksums.json")))
def seeded(key):
    """What the reference computed on the seeded inputs below (tests/golden/make_golden_seeded.py)."""
    with open(os.path.join(GOLDEN, "seeded_checksums.json")) as fh:
        return json.load(fh)[key]


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def buffer_sums(f):
    z = f.get_z_buffer()
    return {"covered": int((z < 1e5).sum()), "z": sha(z), "color": sha(f.get_color_buffer()),
            "normals": sha(f.get_normals_buffer())}


def random_scene_case(seed):
    """(h, w, fov, model, passes) of a seeded random scene; passes = 2 composites a second render into the same buffers."""
    rng = np.random.default_rng(1000 + seed)
    h, w, fov = int(rng.integers(8, 200)), int(rng.integers(8, 200)), float(rng.uniform(20, 120))
    return h, w, fov, random_scene(seed), 2 if seed % 3 == 0 else 1


def out_of_range_model():
    """Coordinates far outside int range after projection: exercises the (int)ceil() behaviour of the compiled reference."""
    v = np.array([[[-3e9, -0.5, 1.0], [3e9, 0.5, 1.0], [0.0, 4e9, 1.0]],
                  [[-0.5, -0.5, 1.0], [0.5, -0.5, 1.0], [0.0, 3e12, 2.0]],
                  [[-0.4, -0.4, 1.5], [0.4, -0.4, 1.5], [0.0, 0.4, 1.5]]], dtype=np.float32)
    n = -np.ones((3, 3, 3), np.float32)
    c = np.full((3, 3, 3), 100, np.float32)
    return TriModel(v, c, n)


def test_fixture_inputs_match_reference_checksums(trex, bunny, basketball):
    for name, m in (("trex", trex), ("bunny", bunny), ("basketball", basketball)):
        want = CHECKS["inputs"][name]
        assert sha(m._vertices_by_triangles) == want["v"]
        assert sha(m._colors_by_triangles) == want["c"]
        assert sha(m._normals_by_triangles) == want["n"]
    # SURVEY 8c check values (sha256[:16]) for the README flow
    assert CHECKS["inputs"]["trex"]["v"].startswith("a127569779db0498")
    assert CHECKS["cases"]["trex_1024x1024_fov45"]["z"].startswith("ce156226ddd3283a")
    assert CHECKS["cases"]["trex_1024x1024_fov45"]["covered"] == 252539


def test_projection_known_answer():
    # SURVEY 8a row a1: 1024^2, fov 45
    P = O.projection_matrix(1024, 1024, 45.0)
    assert float(P[0, 0]).hex() == "0x1.3504f40000000p+1" and P[0, 0] == P[1, 1]
    assert float(P[2, 2]).hex() == "0x1.00068e0000000p+0"
    assert float(P[3, 2]).hex() == "-0x1.99a4160000000p-4"
    assert P[2, 3] == 1.0 and np.count_nonzero(P) == 5
    P = O.projection_matrix(333, 777, 60.0)
    assert P[0, 0] == np.float32(P[1, 1] / np.float32(333 / 777))
    with pytest.raises(ZeroDivisionError):
        O.projection_matrix(8, 8, 45.0, z_near=1.0, z_far=1.0)
    with pytest.raises(ZeroDivisionError):
        O.projection_matrix(8, 0, 45.0)


def test_pixel_rect_known_answers():
    tri = np.array([[1.2, 2.0, 0], [5.0, 7.5, 0], [3.3, 4.4, 0]], dtype=np.float32)
    assert O.pixel_rect(tri, 10, 10) == (2, 5, 2, 8)          # ceil of min / max, half-open
    assert O.pixel_rect(tri - 20, 10, 10) == (0, 0, 0, 0)      # off-screen left/below -> empty
    assert O.pixel_rect(tri + 20, 10, 10) == (10, 10, 10, 10)  # off-screen right/above -> empty
    big = np.array([[-5e9, -1.0, 0], [5e9, 3.0, 0], [1.0, 1e20, 0]], dtype=np.float32)
    # out-of-int-range ceil -> INT_MIN (x86 cvttsd2si) -> clipped to 0: x_right = 0, y_bot = 0
    assert O.pixel_rect(big, 10, 10) == (0, 0, 0, 0)
    nan = np.array([[np.nan, 1.0, 0], [2.0, np.nan, 0], [4.0, 5.0, 0]], dtype=np.float32)
    assert O.pixel_rect(nan, 10, 10) == (2, 4, 1, 5)           # NaNs never win a comparison


def test_barycentric_known_answers():
    tri = np.array([[0, 0, 0], [4, 0, 0], [0, 4, 0]], dtype=np.float32)
    assert np.array_equal(O.barycentric(tri, 0, 0), [1, 0, 0])
    assert np.array_equal(O.barycentric(tri, 4, 0), [0, 1, 0])
    assert np.array_equal(O.barycentric(tri, 1, 1), [0.5, 0.25, 0.25])
    assert O.barycentric(tri, 3, 3)[0] < 0
    deg = np.array([[0, 0, 0], [1, 1, 0], [2, 2, 0]], dtype=np.float32)   # zero area: x/0 -> inf/NaN, no exception
    assert not np.isfinite(O.barycentric(deg, 5, 1)).any()


@pytest.mark.parametrize("case", sorted(k for k in CHECKS["cases"] if not k.startswith("trex_then") and not k.endswith("_guro")))
def test_oracle_reproduces_reference_checksums(case):
    """Every golden case the reference build rendered: the fixtures at 11 sizes, six views of the 1024^2 T-Rex orbit
    (config C5, camera-space arrays of the view transform) and the full-size 10 003 200-triangle sphere at 8192^2
    (config C4; there the oracle runs its row-band threads, bit-equal to n_threads=1 by construction)."""
    info = CHECKS["cases"][case]
    if info["h"] * info["w"] > 2048 * 2048 and os.environ.get("CRB_FULL_GOLDEN", "1") != "1":
        pytest.skip("large case")
    m, nt = case_model(info)
    if "v_in" in info:
        assert sha(m._vertices_by_triangles) == info["v_in"] and sha(m._normals_by_triangles) == info["n_in"]
    f = O.OracleFiller(info["h"], info["w"], fov=info["fov"], n_threads=nt)
    f.render_arrays(m._vertices_by_triangles, m._colors_by_triangles, m._normals_by_triangles)
    assert int((f.get_z_buffer() < 1e5).sum()) == info["covered"]
    assert sha(f.get_z_buffer()) == info["z"]
    assert sha(f.get_color_buffer()) == info["color"]
    assert sha(f.get_normals_buffer()) == info["normals"]


@pytest.mark.parametrize("case", sorted(k for k in CHECKS["cases"] if k.endswith("_guro")))
def test_oracle_reproduces_reference_lit_colour(case, trex, bunny, basketball):
    """Renderer.render with the reference's GuroIllumination (renderer.py:47-49): checksum of the lit colour buffer."""
    info = CHECKS["cases"][case]
    m = {"trex": trex, "bunny": bunny, "basketball": basketball}[info["model"]]
    f = O.OracleFiller(info["h"], info["w"], fov=info["fov"])
    f.render_model(m)
    assert int((f.get_z_buffer() < 1e5).sum()) == info["covered"]
    c = O.guro(f.get_color_buffer().copy(), f.get_normals_buffer(), info["light"])
    assert sha(c) == info["color_lit"]


def test_oracle_compositing_checksum(trex, bunny):
    info = CHECKS["cases"]["trex_then_bunny_640x480_fov50"]
    f = O.OracleFiller(640, 480, fov=50.0)
    f.render_model(trex)
    f.render_model(bunny)
    assert (sha(f.get_z_buffer()), sha(f.get_color_buffer()), sha(f.get_normals_buffer())) == \
        (info["z"], info["color"], info["normals"])


def test_oracle_full_arrays_trex_128(trex):
    g = np.load(os.path.join(GOLDEN, "trex_128.npz"))
    f = O.OracleFiller(128, 128, fov=45.0)
    f.render_model(trex)
    assert bits_equal(f.get_z_buffer(), g["z"]) and bits_equal(f.get_color_buffer(), g["color"]) \
        and bits_equal(f.get_normals_buffer(), g["normals"])


def test_oracle_band_threads_equal_sequential(trex):
    a = O.OracleFiller(300, 200, fov=45.0, n_threads=1)
    b = O.OracleFiller(300, 200, fov=45.0, n_threads=4)
    a.render_model(trex)
    b.render_model(trex)
    assert bits_equal(a.get_z_buffer(), b.get_z_buffer()) and bits_equal(a.get_color_buffer(), b.get_color_buffer()) \
        and bits_equal(a.get_normals_buffer(), b.get_normals_buffer())


def test_oracle_errors():
    f = O.OracleFiller(8, 8)
    m = TriModel(np.zeros((1, 3, 3)), np.zeros((1, 3, 3), np.float32), np.zeros((1, 3, 3), np.float32))
    with pytest.raises(ValueError, match="dtype mismatch"):
        f.render_model(m)
    with pytest.raises(AttributeError):
        f.render_model(TriModel(np.zeros((1, 3, 3), np.float32), None, np.zeros((1, 3, 3), np.float32)))


def test_guro_oracle_matches_numpy_formula():
    # crender/cy/illumination/guro_illumination.py:20-27 evaluated with NumPy itself
    rng = np.random.default_rng(3)
    n = rng.standard_normal((37, 53, 3)).astype(np.float32)
    n[::5, ::3] = 0
    c = (rng.random((37, 53, 3)) * 255).astype(np.float32)
    light = -np.asarray([0.2, -0.4, 1.0], dtype="float32")
    light = light / np.linalg.norm(light)
    want = c.copy()
    sp = np.sum(n * light, axis=-1, keepdims=True)
    want *= np.clip(sp / (np.linalg.norm(n, axis=-1, keepdims=True) + 1e-6), 0, 1)
    got = O.guro(c.copy(), n, [0.2, -0.4, 1.0])
    assert bits_equal(got, want)


# ---- against the reference's own compiled code: its results on seeded inputs (tests/golden/make_golden_seeded.py), and the
# build itself wherever oracle/_ref is present (CRB_REFERENCE_SRC at build time, or oracle/build_ref.py) ----
def _ref_filler_cls():
    ref = os.path.join(ROOT, "oracle", "_ref")
    if ref not in sys.path:
        sys.path.insert(0, ref)
    from crender.cy.pixel_buffer_filler import AdvancedPixelBufferFiller
    return AdvancedPixelBufferFiller


@pytest.mark.parametrize("seed", range(24))
def test_oracle_equals_reference_build_on_random_scenes(seed, capfd):
    h, w, fov, m, passes = random_scene_case(seed)
    o = O.OracleFiller(h, w, fov=fov)
    for _ in range(passes):
        o.render_model(m)
    assert buffer_sums(o) == seeded("random_scenes")[str(seed)]
    if not build_ref.built():
        return
    r = _ref_filler_cls()(h, w, fov=fov, n_threads=1)
    for _ in range(passes):
        r.render_model(m)
    capfd.readouterr()   # the reference printf()s per thread
    assert bits_equal(r.get_z_buffer(), o.get_z_buffer())
    assert bits_equal(r.get_color_buffer(), o.get_color_buffer())
    assert bits_equal(r.get_normals_buffer(), o.get_normals_buffer())


def test_oracle_equals_reference_build_out_of_range_coordinates(capfd):
    m = out_of_range_model()
    o = O.OracleFiller(64, 64, fov=90.0)
    o.render_model(m)
    assert (o.get_z_buffer() < 1e5).sum() > 0
    want = seeded("out_of_range")
    assert (sha(o.get_z_buffer()), sha(o.get_color_buffer())) == (want["z"], want["color"])
    if not build_ref.built():
        return
    r = _ref_filler_cls()(64, 64, fov=90.0, n_threads=1)
    r.render_model(m)
    capfd.readouterr()
    assert bits_equal(r.get_z_buffer(), o.get_z_buffer()) and bits_equal(r.get_color_buffer(), o.get_color_buffer())
