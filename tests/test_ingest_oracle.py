"""Model ingest (SURVEY 8f N4), CPU side: the ingest oracle (oracle/ingest_oracle.c + oracle/ingest.py) and the
library's host-only .obj reader (crb_obj_parse) against golden vectors made by the reference's own `Model`
(tests/golden/make_golden_ingest.py) and -- where oracle/_ref is present -- against that class itself."""
import json
import os
import sys
import warnings

import numpy as np
import pytest
from hypothesis import given, settings, strategies as st

from conftest import GOLDEN, ROOT, bits_equal, same_f32
from cython3dmodelrenderer_b200 import model as M
from oracle import ingest as I

OBJ = os.path.join(GOLDEN, "obj")
REF_OBJ = os.path.join(ROOT, "oracle", "_ref", "objects")
FIXTURES = ["quirks", "torus", "fan", "cube_pm"]


def golden(name):
    d = np.load(os.path.join(GOLDEN, f"ingest_{name}.npz"))
    return d, json.loads(str(d["hashes"]))


def same_parse(p, o):
    """Library reader output (arrays) == Python restatement output (lists)."""
    def arr(x, dt, cols):
        return np.array(x, dtype=dt).reshape(len(x), cols if len(x) == 0 else -1)
    assert bits_equal(p["vertices"], arr(o["vertices"], np.float32, 3))
    assert bits_equal(p["normals"], arr(o["normals"], np.float32, 3))
    widths = {len(r) for r in o["texture_coords"]}
    assert len(widths) <= 1
    assert bits_equal(p["texture_coords"], arr(o["texture_coords"], np.float32, p["texture_coords"].shape[1]))
    assert np.array_equal(p["tri_v"], arr(o["tri_v"], np.int32, 3))
    for k in ("tri_vt", "tri_vn"):
        assert (p[k] is None) == (o[k] is None), k
        if p[k] is not None:
            assert np.array_equal(p[k], arr(o[k], np.int32, 3)), k
    assert p["mtllibs"] == [m.rstrip("\n") for m in o["mtllibs"]]


@pytest.mark.parametrize("name", FIXTURES)
def test_reader_equals_python_restatement_and_reference_golden(name):
    raw = open(os.path.join(OBJ, name + ".obj"), "rb").read()
    p = M.parse_obj_text(raw)
    same_parse(p, I.parse_obj(raw.decode()))
    g, _ = golden(name)
    assert bits_equal(p["vertices"], g["read_vertices"])
    assert np.array_equal(p["tri_v"], g["read_triangles_vertices"])
    if "read_texture_coords" in g:
        assert bits_equal(p["texture_coords"], g["read_texture_coords"])
        assert np.array_equal(p["tri_vt"], g["read_triangles_texture_coords"])


def test_reader_quirks_in_detail():
    p = M.parse_obj_text(open(os.path.join(OBJ, "quirks.obj"), "rb").read())
    assert p["vertices"].shape == (13, 3) and p["tri_v"].shape == (13, 3)
    assert p["tri_vt"] is None and p["tri_vn"] is None      # a face without vt / vn ends those lists for good
    assert p["bad_lines"] >= 8 and p["first_bad_line"] > 0
    assert p["mtllibs"] == ["quirks.mtl", "/nonexistent/abs.mtl"]
    v = p["vertices"]
    assert np.isinf(v).any() and np.isnan(v).any()           # 'inf', '-Infinity', 'nan', 1e400 -> inf
    assert (p["tri_v"] < 0).any() and (p["tri_v"] == 0).any()


def test_reader_refuses_what_python_reads_differently():
    with pytest.raises(ValueError, match="not supported"):
        M.parse_obj_text(b"v 1_000 2 3\n")
    with pytest.raises(ValueError, match="not supported"):
        M.parse_obj_text("v １ 2 3\n".encode())           # full-width digit: a digit to float()
    with pytest.raises(OverflowError):
        M.parse_obj_text(b"v 0 0 0\nf 1 2 99999999999\n")
    with pytest.raises(ValueError, match="inhomogeneous"):
        M.parse_obj_text(b"vt 0.1 0.2\nvt 0.1 0.2 0.3\n")
    assert M.parse_obj_text(b"")["vertices"].shape == (0, 3)
    assert M.parse_obj_text(b"# only a comment")["tri_v"].shape == (0, 3)


_num = st.one_of(
    st.floats(allow_nan=False, allow_infinity=False, width=32).map(repr),
    st.integers(-50, 50).map(str),
    st.sampled_from(["1e5", "-.5", "+3.", "1E-3", "nan", "inf", "-Infinity", "1e999", "1e-999", "x", "1.2.3", "--1",
                     "0x1p3", "1e", "", "5/", "1,2", "٣"[:0] + "7"]))
_corner = st.one_of(
    st.integers(-6, 9).map(str),
    st.tuples(st.integers(-6, 9), st.integers(-6, 9)).map(lambda t: f"{t[0]}/{t[1]}"),
    st.tuples(st.integers(-6, 9), st.integers(-6, 9)).map(lambda t: f"{t[0]}//{t[1]}"),
    st.tuples(st.integers(-6, 9), st.integers(-6, 9), st.integers(-6, 9)).map(lambda t: "%d/%d/%d" % t),
    st.sampled_from(["1/x/1", "a", "1/", "/1", "1/2/3/4", "+2/+2/+2", "1.5", "//", "3/ /3"]))
_sep = st.sampled_from([" ", " ", " ", "  ", "\t", " \t "])
_line = st.one_of(
    st.tuples(st.sampled_from(["v", "vn", "vt", "v", "V", "vp"]), st.lists(st.tuples(_sep, _num), min_size=0, max_size=5))
      .map(lambda t: t[0] + " " + "".join(s + n for s, n in t[1])),
    st.tuples(st.just("f"), st.lists(st.tuples(_sep, _corner), min_size=0, max_size=6))
      .map(lambda t: t[0] + " " + "".join(s + n for s, n in t[1])),
    st.sampled_from(["", "#c", "# v 1 2 3", "g a", "mtllib a.mtl", "mtllib", "mtllib ", "v", "f", " v 1 2 3", "v\t1 2 3",
                     "usemtl x", "\x0cv 1 2 3", "v 1 2 3 \x0b", "v 1\x1c2\x1d3"]))
_eol = st.sampled_from(["\n", "\n", "\n", "\r\n", "\r"])


@settings(max_examples=300, deadline=None)
@given(st.lists(st.tuples(_line, _eol), min_size=0, max_size=25), st.booleans())
def test_reader_equals_python_restatement_on_generated_text(lines, final_newline):
    text = "".join(l + e for l, e in lines)
    if not final_newline:
        text = text.rstrip("\r\n")
    o = I.parse_obj(text)
    widths = {len(r) for r in o["texture_coords"]}
    too_big = [i for t in (o["tri_v"], o["tri_vt"] or [], o["tri_vn"] or []) for r in t for i in r if abs(i) >= 2**31]
    if len(widths) > 1:
        with pytest.raises(ValueError):
            M.parse_obj_text(text.encode())
        return
    assert not too_big
    same_parse(M.parse_obj_text(text.encode()), o)


# ---------------------------------------------------------------------------------------------- oracle arithmetic
@pytest.mark.parametrize("name", FIXTURES + ["torus_inv", "torus_ext"])
def test_oracle_normals_colours_gathers_equal_reference_golden(name):
    g, hashes = golden(name)
    import hashlib
    sha = lambda a: hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:16]   # noqa: E731
    inv = name == "torus_inv"
    for stage in ("read", "rot"):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            n = I.vertex_normals(g[f"{stage}_vertices"], g[f"{stage}_triangles_vertices"], invert=inv and stage == "read")
        assert same_f32(n, g[f"{stage}_normals"]), f"{name}/{stage}: vertex normals differ from the reference's"
        if not np.isnan(n).any():
            assert sha(I.gather(n, g[f"{stage}_triangles_normals"])) == hashes[f"{stage}_normals_by_triangles"]
        assert sha(I.gather(g[f"{stage}_vertices"], g[f"{stage}_triangles_vertices"])) == hashes[f"{stage}_vertices_by_triangles"]
    if "read_colors" in g:
        import cv2
        tex = cv2.imread(os.path.join(OBJ, "checker.png"))
        c = I.vertex_colors(g["read_texture_coords"], tex)
        assert bits_equal(c, g["read_colors"])
        assert sha(I.gather(c, g["read_triangles_texture_coords"])) == hashes["read_colors_by_triangles"]


def test_oracle_face_normal_known_answers():
    t = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], np.float32)
    n = I.face_normal(t)
    assert n.tolist() == [0.0, 0.0, 1.0] and np.signbit(n[:2]).all()   # -(+0.0) stays -0.0 through n / 1
    z = I.face_normal(np.zeros((3, 3), np.float32))
    assert np.signbit(z).all() and (z == 0).all()                       # zero norm: returned unnormalised
    # np.dot's double accumulator: a float accumulator gives 0x1.a7ecdap-3 for this pair (probe in the header)
    a = np.array([float.fromhex(h) for h in ("0x1.017ed8p-3", "-0x1.0e8cfep-3", "0x1.47e57ap-1")], np.float32)
    b = np.array([float.fromhex(h) for h in ("-0x1.86ce04p-1", "-0x1.a50d86p-5", "-0x1.e5899ep-2")], np.float32)
    assert float(a.dot(b)).hex() == "-0x1.9244ae0000000p-2"


def seeded(key):
    """What the reference computed on the seeded inputs below (tests/golden/make_golden_seeded.py)."""
    with open(os.path.join(GOLDEN, "seeded_checksums.json")) as fh:
        return json.load(fh)[key]


def _ref_model_cls():
    ref = os.path.join(ROOT, "oracle", "_ref")
    if ref not in sys.path:
        sys.path.insert(0, ref)
    warnings.filterwarnings("ignore", category=SyntaxWarning)
    from crender.cy.data_structures import Model
    return Model


def random_mesh(seed):
    """(vertices, triangles, texture coords, texture-coord triangles, texture, invert) of a seeded random mesh."""
    rng = np.random.default_rng(seed)
    V, T = int(rng.integers(4, 60)), int(rng.integers(1, 150))
    v = rng.standard_normal((V, 3)).astype(np.float32)
    if seed % 2:
        v = np.round(v * 2) / 2          # coplanar / repeated normals, degenerate triangles
    tri = rng.integers(-V, V, (T, 3)).astype(np.int32)
    vt = rng.uniform(-0.2, 1.2, (V + 3, 2)).astype(np.float32)
    tvt = rng.integers(0, V + 3, (T, 3)).astype(np.int32)
    tex = rng.integers(0, 256, (9, 13, 3), dtype=np.uint8)
    return v, tri, vt, tvt, tex, bool(seed % 3 == 0)


def sha_nan(a):
    """sha256 of float32 data with every NaN written as 0x7FC00000 (NaN bits mean nothing to NumPy code, see same_f32)."""
    import hashlib
    a = np.array(a, dtype=np.float32)
    a.view(np.uint32)[np.isnan(a)] = 0x7FC00000
    return hashlib.sha256(a.tobytes()).hexdigest()


def mesh_sums(normals, colors, normals_by_triangles, colors_by_triangles):
    return {"normals": sha_nan(normals), "colors": sha_nan(colors), "normals_by_triangles": sha_nan(normals_by_triangles),
            "colors_by_triangles": sha_nan(colors_by_triangles)}


@pytest.mark.parametrize("seed", range(6))
def test_oracle_equals_reference_model_on_random_meshes(seed):
    """The ingest oracle against the reference Model's results on seeded meshes (tests/golden/make_golden_seeded.py), and
    against that class itself where oracle/_ref is present."""
    v, tri, vt, tvt, tex, invert = random_mesh(seed)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        n = I.vertex_normals(v, tri, invert=invert)
    c = I.vertex_colors(vt, tex)
    assert mesh_sums(n, c, I.gather(n, tri), I.gather(c, tvt)) == seeded("random_meshes")[str(seed)]
    if not os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "crender")):
        return
    Ref = _ref_model_cls()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m = Ref(v.tolist(), tri.tolist(), vt.tolist(), tvt.tolist(), tex, invert_calculated_normals=invert)
    assert same_f32(n, m._normals)
    assert bits_equal(c, m._colors)
    assert same_f32(I.gather(n, tri), m._normals_by_triangles)
    assert bits_equal(I.gather(m._colors, tvt), m._colors_by_triangles)


@pytest.mark.ref
def test_reader_equals_reference_read_model_on_its_own_assets():
    """The reference's assets (not committed): checksums of what its Model read from them."""
    if not os.path.isdir(REF_OBJ):
        pytest.skip("oracle/_ref/objects not present")
    import hashlib
    sums = json.load(open(os.path.join(GOLDEN, "ingest_checksums.json")))
    sha = lambda a: hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:16]   # noqa: E731
    for name in ("T-Rex", "basketball", "bunny", "cube", "Cube2"):
        p = M.parse_obj_text(open(os.path.join(REF_OBJ, name + ".obj"), "rb").read())
        s = sums[name]
        assert sha(p["vertices"]) == s["read_vertices"]["sha256_16"], name
        assert sha(p["tri_v"]) == s["read_triangles_vertices"]["sha256_16"], name
        if "read_texture_coords" in s:
            assert sha(p["texture_coords"]) == s["read_texture_coords"]["sha256_16"], name
            assert sha(p["tri_vt"]) == s["read_triangles_texture_coords"]["sha256_16"], name
        n = I.vertex_normals(p["vertices"], p["tri_v"])
        assert sha(n) == s["read_normals"]["sha256_16"], name
