"""The oracle of the two texturing modes (oracle/texture_modes_oracle.py: CRB_TEX_PERSPECTIVE, CRB_TEX_BILINEAR; DESIGN 2), on
the CPU.

The NumPy bilinear rule is checked against a scalar restatement, one float32 operation at a time, on random and adversarial
coordinates and texture shapes; at texel centres it must be the nearest texel.  The perspective composition is checked
against the definition at every covered pixel (prelude, interpolation, division, texel rule), and semantically: on quads
tilted steeply away from the camera its (u, v) are those of the point of the triangle's plane seen through the pixel,
which affine coordinates miss.
"""
import platform

import numpy as np
import pytest

from conftest import bits_equal
from test_texture_oracle import SPECIAL, random_texture, random_uvs, texel_rule

F32 = np.float32
SHAPES = [(1, 1), (1, 7), (7, 1), (2, 2), (4, 16), (64, 32), (256, 256), (709, 709)]
x86 = pytest.mark.skipif(platform.machine() not in ("x86_64", "AMD64"), reason="NumPy's float -> int32 cast is platform-defined")


def O():
    from oracle import oracle
    return oracle


def TM():
    from oracle import texture_modes_oracle
    return texture_modes_oracle


def bilinear_scalar(u, v, tex):
    """CRB_TEX_BILINEAR for one coordinate pair, np.float32 scalars, one rounding per line."""
    th, tw = tex.shape[:2]
    with np.errstate(invalid="ignore", over="ignore"):
        sx = F32(u) * F32(tw)
        sx = sx - F32(0.5)
        sy = F32(1) - F32(v)
        sy = sy * F32(th)
        sy = sy - F32(0.5)
    out = []
    for s, n in ((sx, tw), (sy, th)):
        if np.isnan(s) or s < F32(-1):       # fmax(s, -1): NaN gives -1
            s = F32(-1)
        if s > F32(n):                       # fmin(s, n)
            s = F32(n)
        s0 = np.floor(s)
        f = s - s0
        assert f.dtype == np.float32
        i = int(s0)
        out.append((f, F32(1) - f, min(max(i, 0), n - 1), min(max(i + 1, 0), n - 1)))
    (fx, gx, c0, c1), (fy, gy, r0, r1) = out
    res = np.empty(3, F32)
    for k in range(3):
        t00, t01 = F32(tex[r0, c0, k]), F32(tex[r0, c1, k])
        t10, t11 = F32(tex[r1, c0, k]), F32(tex[r1, c1, k])
        a = t00 * gx
        b = t01 * fx
        top = a + b
        a = t10 * gx
        b = t11 * fx
        bot = a + b
        a = top * gy
        b = bot * fy
        res[k] = a + b
    return res


def adversarial_coordinates(tw):
    """NaN, +-inf, +-1e30, 0 and 1 and one ulp either side of them, texel centres and texel edges of a tw-wide texture."""
    vals = [np.nan, np.inf, -np.inf, 1e30, -1e30, 0.0, -0.0, 1.0, 0.5, -1e-30, 1e-30]
    for x in (0.0, 1.0):
        vals += [np.nextafter(F32(x), F32(-2)), np.nextafter(F32(x), F32(2))]
    for c in sorted({0, 1, tw // 2, max(tw - 2, 0), tw - 1}):
        vals += [(c + 0.5) / tw, c / tw, (c + 1) / tw, np.nextafter(F32(c / tw), F32(2)), np.nextafter(F32((c + 0.5) / tw), F32(-2))]
    return np.array(vals, F32)


@pytest.mark.parametrize("tshape", SHAPES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_bilinear_rule_matches_scalar_restatement(tshape):
    th, tw = tshape
    tex = random_texture(th * 7 + tw, th, tw)
    rng = np.random.default_rng(th * 1000 + tw)
    us = np.concatenate([adversarial_coordinates(tw), rng.uniform(-0.3, 1.3, 200).astype(F32), SPECIAL])
    vs = np.concatenate([adversarial_coordinates(th), rng.uniform(-0.3, 1.3, 200).astype(F32), SPECIAL])
    u, v = np.meshgrid(us, vs)              # every u against every v
    u, v = u.ravel(), v.ravel()
    pick = rng.choice(u.size, min(u.size, 6000), replace=False)
    got = TM().bilinear_texels(u[pick], v[pick], tex)
    assert got.dtype == F32 and got.shape == (pick.size, 3)
    for i, j in enumerate(pick):
        want = bilinear_scalar(u[j], v[j], tex)
        assert bits_equal(got[i], want), (tshape, u[j], v[j], got[i], want)
    assert np.all(np.isfinite(got)) and np.all(got >= 0) and np.all(got <= 255)


@x86
@pytest.mark.parametrize("tshape", [(1, 1), (2, 4), (16, 16), (64, 128), (512, 256)], ids=lambda s: f"{s[0]}x{s[1]}")
def test_bilinear_equals_nearest_at_texel_centres(tshape):
    """Power-of-two textures, u = (c + 0.5) / tw, v = 1 - (r + 0.5) / th: sx = c and sy = r exactly, so the blend is the texel
    the nearest rule names."""
    th, tw = tshape
    tex = random_texture(3, th, tw)
    r, c = np.meshgrid(np.arange(th), np.arange(tw), indexing="ij")
    u = ((c.ravel() + F32(0.5)) / F32(tw)).astype(F32)
    v = (F32(1) - (r.ravel() + F32(0.5)) / F32(th)).astype(F32)
    assert np.array_equal(u * F32(tw) - F32(0.5), c.ravel().astype(F32))
    assert np.array_equal((F32(1) - v) * F32(th) - F32(0.5), r.ravel().astype(F32))
    got = TM().bilinear_texels(u, v, tex)
    assert bits_equal(got, texel_rule(u, v, tex))
    assert bits_equal(got, tex[r.ravel(), c.ravel()].astype(F32))


def _depth_triangle(h, w, px, py, zs):
    """Camera-space corners at depths zs[k] that project near pixels (px[k], py[k]) of an h x w frame at fov 90, facing the
    camera."""
    xs, ys = F32(w / 2.0), F32(h / 2.0)
    v = np.zeros((1, 3, 3), F32)
    for k in range(3):
        z = F32(zs[k])
        v[0, k] = ((F32(px[k]) / xs - F32(1)) * z, (F32(py[k]) / ys - F32(1)) * z, z)
    n = np.zeros((1, 3, 3), F32)
    n[..., 2] = -1
    return v, n


DEPTHS = np.array([0.3, 1.0, 2.5, 7.0, 40.0, 1e-3, -1.0, 0.0], F32)


@x86
@pytest.mark.parametrize("filt", ["nearest", "bilinear"])
@pytest.mark.parametrize("tshape", [(1, 1), (7, 1), (61, 47)], ids=lambda s: f"{s[0]}x{s[1]}")
def test_perspective_composition_follows_the_definition(tshape, filt):
    """Every covered pixel of single triangles with corners at different depths (some at z = 0 or behind the camera) and
    coordinates including NaN, +-inf and +-1e10: the colour is the definition restated in NumPy float32 -- w = 1 / z per corner,
    (u*w, v*w, w) interpolated with the oracle's barycentrics, u = U / W, v = V / W, then the texel rule or the bilinear rule.
    The junk third component of the coordinates has no effect."""
    rng = np.random.default_rng(sum(tshape) + len(filt))
    tex = random_texture(tshape[1], *tshape)
    h = w = 64
    P = O().projection_matrix(h, w)
    checked = 0
    for i in range(40):
        zs = rng.uniform(0.5, 6.0, 3).astype(F32)
        if i % 4 == 3:
            zs[i % 3] = DEPTHS[(i // 4) % len(DEPTHS)]
        v, n = _depth_triangle(h, w, rng.integers(0, w, 3), rng.integers(0, h, 3), zs)
        uv = random_uvs(i, 1, special=(i % 2 == 1))
        o = TM().TexturedOracleFiller(h, w)
        o.render_arrays(v, uv, n, texture=tex, perspective=True, filter=filt)
        uv0 = uv.copy()
        uv0[..., 2] = 0
        o0 = TM().TexturedOracleFiller(h, w)
        o0.render_arrays(v, uv0, n, texture=tex, perspective=True, filter=filt)
        assert bits_equal(o.get_color_buffer(), o0.get_color_buffer())
        s = O().project(h, w, P, v)[0]
        with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
            wk = F32(1) / v[0, :, 2]
            U, V = uv[0, :, 0] * wk, uv[0, :, 1] * wk
        ys, xs = np.nonzero(o.get_z_buffer() < F32(1e6))
        for y, x in zip(ys, xs):
            b = O().barycentric(s, x, y)
            with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
                Ui = (U[0] * b[0] + U[1] * b[1]) + U[2] * b[2]
                Vi = (V[0] * b[0] + V[1] * b[1]) + V[2] * b[2]
                Wi = (wk[0] * b[0] + wk[1] * b[1]) + wk[2] * b[2]
                u_, v_ = np.array([Ui / Wi], F32), np.array([Vi / Wi], F32)
            want = TM().bilinear_texels(u_, v_, tex)[0] if filt == "bilinear" else texel_rule(u_, v_, tex)[0]
            assert bits_equal(o.get_color_buffer()[y, x], want), (i, x, y, u_, v_)
            checked += 1
    assert checked > 300


def test_pixel_uv_and_slots():
    v = np.array([[[0, 0, 2], [1, 0, 4], [0, 1, 0.5]]], F32)
    uv = np.array([[[0.25, 0.75, 99], [1, 0, -5], [0.5, 0.5, 1e6]]], F32)
    s = TM().perspective_slots(v, uv)
    assert s.dtype == F32 and s.shape == (1, 3, 3)
    assert bits_equal(s[0, :, 2], np.array([0.5, 0.25, 2], F32))
    assert bits_equal(s[0, :, 0], np.array([0.125, 0.25, 1], F32)) and bits_equal(s[0, :, 1], np.array([0.375, 0, 1], F32))
    assert bits_equal(TM().perspective_slots(v, uv[..., :2]), s)
    u_, v_ = TM().pixel_uv(s[0], True)
    assert bits_equal(u_, uv[0, :, 0]) and bits_equal(v_, uv[0, :, 1])
    u_, v_ = TM().pixel_uv(s[0], False)
    assert bits_equal(u_, s[0, :, 0]) and bits_equal(v_, s[0, :, 1])


def _tilted_quads():
    """Two textured quads (two triangles each) seen at a grazing angle: a floor running from z = 1 to z = 20, and a wall
    turned about the vertical axis from z = 1.2 to z = 12."""
    floor = np.array([(-2, 0.6, 1), (2, 0.6, 1), (2, 0.6, 20), (-2, 0.6, 20)], F32)
    wall = np.array([(-0.8, -0.7, 1.2), (1.5, -0.7, 12), (1.5, 0.7, 12), (-0.8, 0.7, 1.2)], F32)
    quad_uv = np.array([(0, 0), (1, 0), (1, 1), (0, 1)], F32)
    out = []
    for q in (floor, wall):
        for idx in ((0, 1, 2), (0, 2, 3)):
            out.append((q[list(idx)], quad_uv[list(idx)]))
    return out


@pytest.mark.parametrize("tri", range(4))
def test_perspective_coordinates_are_those_of_the_surface(tri):
    """At each covered pixel well inside the triangle, the point of the triangle's plane that projects to that pixel (screen
    x and y are affine in X/Z and Y/Z: a 3x3 linear system in its barycentrics beta, float64) has coordinates sum(beta_k uv_k).
    The perspective (u, v) of the oracle match them to 1e-4; the affine ones miss by more than 1e-2 somewhere."""
    h, w = 192, 256
    corners, uvk = _tilted_quads()[tri]
    v = corners[None].copy()
    n = np.zeros((1, 3, 3), F32)
    n[..., 2] = -1
    uv = np.concatenate([uvk, np.zeros((3, 1), F32)], axis=1)[None]
    P = O().projection_matrix(h, w).astype(np.float64).ravel()
    slots = {"perspective": TM().perspective_slots(v, uv), "affine": uv}
    got = {}
    for name, c in slots.items():
        o = O().OracleFiller(h, w)
        o.render_arrays(v, c, n)
        got[name] = o
    cov = got["affine"].get_z_buffer() < F32(1e6)
    assert bits_equal(got["affine"].get_z_buffer(), got["perspective"].get_z_buffer())
    s = O().project(h, w, O().projection_matrix(h, w), v)[0]
    V = corners.astype(np.float64)
    Xn = V[:, 0] * P[0] + V[:, 1] * P[4] + V[:, 2] * P[8] + P[12]
    Yn = Xn * P[1] + V[:, 1] * P[5] + V[:, 2] * P[9] + P[13]
    xs, ys = w / 2.0, h / 2.0
    assert np.allclose((Xn / V[:, 2] + 1) * xs, s[:, 0], atol=1e-3) and np.allclose((Yn / V[:, 2] + 1) * ys, s[:, 1], atol=1e-3)
    err = {"perspective": 0.0, "affine": 0.0}
    checked = 0
    for y, x in zip(*np.nonzero(cov)):
        b = O().barycentric(s, x, y)
        if b.min() < 0.02:
            continue
        A = np.stack([Xn - (x / xs - 1) * V[:, 2], Yn - (y / ys - 1) * V[:, 2], np.ones(3)])
        beta = np.linalg.solve(A, np.array([0.0, 0.0, 1.0]))
        want = beta @ uvk.astype(np.float64)
        for name, o in got.items():
            u_, v_ = TM().pixel_uv(o.get_color_buffer()[y, x], name == "perspective")
            err[name] = max(err[name], abs(float(u_) - want[0]), abs(float(v_) - want[1]))
        checked += 1
    assert checked > 500
    assert err["perspective"] < 1e-4, err
    assert err["affine"] > 1e-2, err


def test_refusals():
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller
    v = np.array([[[0, 0, 1], [1, 0, 1], [0, 1, 1]]], F32)
    n = np.zeros_like(v)
    n[..., 2] = -1
    tex = random_texture(1, 4, 4)
    o = TM().TexturedOracleFiller(8, 8)
    for bad in ("cubic", "Bilinear", None, 1):
        with pytest.raises(ValueError):
            o.render_arrays(v, v, n, texture=tex, filter=bad)
        with pytest.raises(ValueError):
            TM().render_textured(o, v, v, n, tex, filter=bad)
        with pytest.raises(ValueError):
            AdvancedPixelBufferFiller(8, 8, texture_filter=bad)
    for bad in ("yes", 1, None, 0.0):
        with pytest.raises(ValueError):
            AdvancedPixelBufferFiller(8, 8, perspective_correct=bad)
    with pytest.raises(ValueError):
        o.render_arrays(v, v, n, perspective=True)          # a mode without a texture
