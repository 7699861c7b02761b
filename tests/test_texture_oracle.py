"""The oracle of per-pixel texturing (oracle/texture_oracle.py, an extension of this project; DESIGN 2), on the CPU.

The textured oracle composes two pinned pieces: oracle_render with the texture coordinates in the colour slots (the draw
loop, pinned against the reference build by test_oracle_pinning.py) and ingest_vertex_colors, the texel rule of
model.py:147-150 (pinned by test_ingest_oracle.py), applied to the interpolated (u, v) of every pixel the render drew.
These tests check that the composition is what DESIGN 2 defines: visibility, depth and normals are the per-vertex
oracle's, a constant texture colours exactly the pixels the per-vertex oracle draws, a pixel on a vertex gets that
vertex's texel, and every covered pixel -- out-of-range coordinates included -- takes the texel a NumPy float32
restatement of the interpolation and the rule names.
"""
import platform

import numpy as np
import pytest

from conftest import bits_equal, random_scene

F32 = np.float32
SPECIAL = np.array([np.nan, np.inf, -np.inf, 1e10, -1e10, -3.0, 0.0, 1.0, 0.5, 0.999, 1.0001, -0.0, 3e9], dtype=F32)


def O():
    from oracle import oracle
    return oracle


def TO():
    from oracle import texture_oracle
    return texture_oracle


def random_uvs(seed, T, special=True):
    """[T,3,3] texture coordinates (u, v, junk): mostly in [-0.2, 1.2], with `special` a tenth from SPECIAL."""
    rng = np.random.default_rng(1000 + seed)
    uv = rng.uniform(-0.2, 1.2, (T, 3, 3)).astype(F32)
    uv[..., 2] = rng.standard_normal((T, 3)).astype(F32) * F32(1e6)      # ignored by the rule
    if special:
        pick = rng.random((T, 3, 2)) < 0.1
        uv[..., :2][pick] = rng.choice(SPECIAL, int(pick.sum()))
    return uv


def random_texture(seed, h, w):
    return np.random.default_rng(2000 + seed).integers(0, 256, (h, w, 3), dtype=np.uint8)


def textured(h, w, v, uv, n, texture, fov=90.0, base=None):
    o = TO().TexturedOracleFiller(h, w, fov=fov)
    if base is not None:
        o.render_arrays(*base)
    o.render_arrays(v, uv, n, texture=texture)
    return o


def texel_rule(u, v, texture):
    """model.py:147-150 restated in NumPy float32: astype('int32') (x86-64: INT32_MIN for NaN / out of range), then clip."""
    th, tw = texture.shape[:2]
    with np.errstate(invalid="ignore", over="ignore"):
        row = np.clip(((F32(1) - np.asarray(v, F32)) * F32(th)).astype(np.int32), 0, th - 1)
        col = np.clip((np.asarray(u, F32) * F32(tw)).astype(np.int32), 0, tw - 1)
    return texture[row, col].astype(F32)


@pytest.mark.parametrize("seed", range(24))
def test_constant_texture_colours_the_pixels_the_vertex_oracle_draws(seed):
    """z and normals bit for bit; colour = the texel wherever the per-vertex oracle drew (its colour is NaN there when
    every corner colour is NaN), 0 elsewhere."""
    m = random_scene(seed)
    v, n = m._vertices_by_triangles, m._normals_by_triangles
    T = v.shape[0]
    texel = np.array([7, 130, 255], np.uint8)
    tex = np.broadcast_to(texel, (5, 3, 3)).copy()
    ref = O().OracleFiller(64, 80, fov=75.0)
    ref.render_arrays(v, np.full((T, 3, 3), np.nan, F32), n)
    got = textured(64, 80, v, random_uvs(seed, T), n, tex, fov=75.0)
    assert bits_equal(got.get_z_buffer(), ref.get_z_buffer())
    assert bits_equal(got.get_normals_buffer(), ref.get_normals_buffer())
    drawn = np.isnan(ref.get_color_buffer()).all(axis=-1)
    want = np.where(drawn[..., None], texel.astype(F32), F32(0))
    assert bits_equal(got.get_color_buffer(), want)


@pytest.mark.parametrize("seed", range(24))
def test_depth_and_normals_are_the_vertex_oracles(seed):
    """Random texture and coordinates, composited onto a per-vertex frame: only the colour may differ."""
    m = random_scene(seed)
    base = random_scene(seed + 100, T=50)
    base_arrays = (base._vertices_by_triangles, base._colors_by_triangles, base._normals_by_triangles)
    v, c, n = m._vertices_by_triangles, m._colors_by_triangles, m._normals_by_triangles
    ref = O().OracleFiller(96, 72)
    ref.render_arrays(*base_arrays)
    ref.render_arrays(v, c, n)
    got = textured(96, 72, v, random_uvs(seed, v.shape[0]), n, random_texture(seed, 33, 17), base=base_arrays)
    assert bits_equal(got.get_z_buffer(), ref.get_z_buffer())
    assert bits_equal(got.get_normals_buffer(), ref.get_normals_buffer())


def _pixel_triangle(h, w, px, py, z=F32(1.0)):
    """Camera-space corners that the oracle projects exactly onto pixel centres (px[k], py[k]) of an h x w frame at
    fov 90 (square frames: P00 = P11 = 1), facing the camera (normals (0, 0, -1))."""
    xs, ys = F32(w / 2.0), F32(h / 2.0)
    v = np.zeros((1, 3, 3), F32)
    for k in range(3):
        v[0, k] = ((F32(px[k]) / xs - F32(1)) * z, (F32(py[k]) / ys - F32(1)) * z, z)
    n = np.zeros((1, 3, 3), F32)
    n[..., 2] = -1
    return v, n


@pytest.mark.parametrize("seed", range(12))
def test_pixel_on_a_vertex_gets_the_vertex_texel(seed):
    from oracle import ingest as I
    rng = np.random.default_rng(seed)
    h = w = 128
    tex = random_texture(seed, int(rng.integers(1, 300)), int(rng.integers(1, 300)))
    checked = 0
    for _ in range(20):
        px, py = rng.integers(0, w, 3), rng.integers(0, h, 3)
        v, n = _pixel_triangle(h, w, px, py)
        s = O().project(h, w, O().projection_matrix(h, w), v)
        assert np.array_equal(s[0, :, 0], px.astype(F32)) and np.array_equal(s[0, :, 1], py.astype(F32))
        uv = rng.uniform(-0.1, 1.1, (1, 3, 2)).astype(F32)
        o = textured(h, w, v, uv, n, tex)
        x0, x1, y0, y1 = O().pixel_rect(s[0], h, w)
        for k in range(3):
            if x0 <= px[k] < x1 and y0 <= py[k] < y1 and o.get_z_buffer()[py[k], px[k]] < F32(1e6):
                want = I.vertex_colors(uv[0, k:k + 1], tex)[0]
                assert bits_equal(o.get_color_buffer()[py[k], px[k]], want), (px[k], py[k], uv[0, k])
                checked += 1
    assert checked >= 10


@pytest.mark.skipif(platform.machine() not in ("x86_64", "AMD64"), reason="NumPy's float -> int32 cast is platform-defined")
@pytest.mark.parametrize("tshape", [(1, 1), (1, 7), (7, 1), (61, 47)])
def test_out_of_range_coordinates_follow_the_numpy_rule(tshape):
    """Every covered pixel of triangles whose corner coordinates come from NaN, +-inf, +-1e10, -3, 0, 1, ...: the colour is
    the texel a NumPy float32 restatement names -- barycentrics (oracle_barycentric), u = (u0*b1 + u1*b2) + u2*b3, then
    astype('int32') and the clip."""
    rng = np.random.default_rng(sum(tshape))
    tex = random_texture(tshape[0], *tshape)
    h = w = 64
    P = O().projection_matrix(h, w)
    checked = 0
    for i in range(len(SPECIAL) * 3):
        v, n = _pixel_triangle(h, w, rng.integers(0, w, 3), rng.integers(0, h, 3))
        uv = rng.uniform(-0.5, 1.5, (1, 3, 2)).astype(F32)
        uv[0, i % 3, i % 2] = SPECIAL[i % len(SPECIAL)]
        uv[0, (i + 1) % 3, (i // 2) % 2] = SPECIAL[(i * 7) % len(SPECIAL)]
        o = textured(h, w, v, uv, n, tex)
        s = O().project(h, w, P, v)[0]
        ys, xs = np.nonzero(o.get_z_buffer() < F32(1e6))
        for y, x in zip(ys, xs):
            b = O().barycentric(s, x, y)
            with np.errstate(invalid="ignore", over="ignore"):
                u_ = (uv[0, 0, 0] * b[0] + uv[0, 1, 0] * b[1]) + uv[0, 2, 0] * b[2]
                v_ = (uv[0, 0, 1] * b[0] + uv[0, 1, 1] * b[1]) + uv[0, 2, 1] * b[2]
            assert bits_equal(o.get_color_buffer()[y, x], texel_rule(np.array([u_], F32), np.array([v_], F32), tex)[0]), \
                (i, x, y, u_, v_)
            checked += 1
    assert checked > 100


def test_uv_pairs_equal_uv_triples():
    m = random_scene(3)
    uv = random_uvs(3, m._vertices_by_triangles.shape[0])
    tex = random_texture(3, 20, 30)
    a = textured(50, 40, m._vertices_by_triangles, uv, m._normals_by_triangles, tex)
    b = textured(50, 40, m._vertices_by_triangles, np.ascontiguousarray(uv[..., :2]), m._normals_by_triangles, tex)
    assert bits_equal(a.get_color_buffer(), b.get_color_buffer())


def test_bad_texture_is_refused():
    m = random_scene(1)
    o = TO().TexturedOracleFiller(8, 8)
    for bad in (np.zeros((4, 4, 3), np.float32), np.zeros((4, 4), np.uint8), np.zeros((0, 4, 3), np.uint8)):
        with pytest.raises(ValueError):
            o.render_arrays(m._vertices_by_triangles, m._colors_by_triangles, m._normals_by_triangles, texture=bad)


def test_spherical_uvs_are_latitude_longitude():
    from cython3dmodelrenderer_b200 import synthetic
    s = synthetic.uv_sphere(16, 8)
    uv = synthetic.spherical_uvs(s._vertices_by_triangles, center=(0.0, 0.0, 1.5))
    assert uv.shape == s._vertices_by_triangles.shape[:2] + (2,) and uv.dtype == F32
    assert np.all((uv >= 0) & (uv <= 1))
    lat = np.arcsin(np.clip(s._normals_by_triangles[..., 1], -1, 1)) / np.pi + 0.5
    assert np.allclose(uv[..., 1], lat, atol=1e-5)
