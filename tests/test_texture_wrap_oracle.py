"""The wrap modes of per-pixel texturing, CRB_TEX_REPEAT and CRB_TEX_MIRROR (DESIGN 2): the CPU oracle
(oracle/texture_wrap_oracle.py) against a scalar restatement of the rule (math.floor, Python's %), against the clamp rule where
both must agree, for periodicity and mirror symmetry, for trilinear filtering, and end to end on a full-screen quad whose
coordinates span several periods."""
import math
import platform

import numpy as np
import pytest

from conftest import bits_equal
from test_texture_oracle import random_texture

F32 = np.float32
SHAPES = [(1, 1), (1, 7), (7, 1), (61, 47), (512, 256)]
WRAPS = ("repeat", "mirror")
x86 = pytest.mark.skipif(platform.machine() not in ("x86_64", "AMD64"), reason="NumPy's float -> int32 cast is platform-defined")


def O():
    from oracle import oracle
    return oracle


def TM():
    from oracle import texture_modes_oracle
    return texture_modes_oracle


def MIP():
    from oracle import texture_mip_oracle
    return texture_mip_oracle


def WR():
    from oracle import texture_wrap_oracle
    return texture_wrap_oracle


# ---- scalar restatement: float32 scalars for every float operation, Python integers for the indices ----------------------

def s_ifloor(x):
    x = F32(x)
    if math.isnan(x) or abs(float(x)) >= 2.0 ** 31:
        x = F32(0)
    return math.floor(float(x))


def s_wrap(k, n, wrap):
    if wrap == "repeat":
        return k % n
    m = k % (2 * n)
    return m if m < n else 2 * n - 1 - m


def s_nearest(u, v, tex, wrap):
    th, tw = tex.shape[:2]
    with np.errstate(all="ignore"):
        col = s_wrap(s_ifloor(F32(u) * F32(tw)), tw, wrap)
        row = s_wrap(s_ifloor((F32(1) - F32(v)) * F32(th)), th, wrap)
    return [F32(x) for x in tex[row, col]]


def s_bilinear(u, v, tex, wrap):
    th, tw = tex.shape[:2]
    with np.errstate(all="ignore"):
        sx = F32(u) * F32(tw) - F32(0.5)
        sy = (F32(1) - F32(v)) * F32(th) - F32(0.5)
    sx, sy = (F32(0) if math.isnan(s) or abs(float(s)) >= 2.0 ** 31 else s for s in (sx, sy))
    x0, y0 = math.floor(float(sx)), math.floor(float(sy))
    fx, fy = sx - F32(x0), sy - F32(y0)
    gx, gy = F32(1) - fx, F32(1) - fy
    c0, c1, r0, r1 = s_wrap(x0, tw, wrap), s_wrap(x0 + 1, tw, wrap), s_wrap(y0, th, wrap), s_wrap(y0 + 1, th, wrap)
    out = []
    for k in range(3):
        t = lambda r, c: F32(tex[r, c, k])      # noqa: E731
        top = t(r0, c0) * gx + t(r0, c1) * fx
        bot = t(r1, c0) * gx + t(r1, c1) * fx
        out.append(top * gy + bot * fy)
    return out


def adversarial(n):
    """NaN, +-inf, +-3e9, +-2^31, -1e-45, -0.0, 2^24 + 1, 0 and 1 and one ulp either side, and integer and half-integer
    texel positions of an n-texel axis over several periods either side of [0, 1] (as texture coordinates)."""
    vals = [np.nan, np.inf, -np.inf, 3e9, -3e9, 2.0 ** 31, -2.0 ** 31, -1e-45, -0.0, 0.0, 1.0, 2.0 ** 24 + 1]
    vals += [2.0 ** 31 / n, -2.0 ** 31 / n, 3e9 / n, -3e9 / n]           # products at the limits
    for x in (0.0, 1.0):
        vals += [np.nextafter(F32(x), F32(-2)), np.nextafter(F32(x), F32(2))]
    for k in sorted({-2 * n - 1, -n - 1, -n, -1, 0, 1, n // 2, n - 1, n, n + 1, 2 * n, 3 * n + 2}):
        vals += [k / n, (k + 0.5) / n, np.nextafter(F32(k / n), F32(-1e9)), np.nextafter(F32((k + 0.5) / n), F32(1e9))]
    return np.array(vals, F32)


def _grid(tshape):
    th, tw = tshape
    us, vs = adversarial(tw), adversarial(th)
    u, v = np.meshgrid(us, vs)
    return u.ravel(), v.ravel()


def _scalar(fn, u, v, tex, wrap):
    return np.array([fn(a, b, tex, wrap) for a, b in zip(u, v)], F32).reshape(-1, 3)


@pytest.mark.parametrize("wrap", WRAPS)
@pytest.mark.parametrize("tshape", SHAPES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_samplers_match_scalar_restatement(tshape, wrap):
    tex = random_texture(tshape[0] * 31 + tshape[1], *tshape)
    u, v = _grid(tshape)
    assert bits_equal(WR().nearest_texels(u, v, tex, wrap), _scalar(s_nearest, u, v, tex, wrap))
    assert bits_equal(WR().bilinear_texels(u, v, tex, wrap), _scalar(s_bilinear, u, v, tex, wrap))


def test_index_rule():
    big = [-2 ** 31, -2 ** 31 + 1, -3 * 2 ** 30, -1, 0, 1, 2 ** 31 - 2, 2 ** 31 - 1]
    for n in (1, 2, 3, 7, 256, 2 ** 30 - 1, 2 ** 30, 2 ** 31 - 1):        # 2n of the last three exceeds int32
        k = np.array(big + list(range(-3 * n - 2, 3 * n + 3)) if n < 64 else big + list(range(-200, 200)), np.int64)
        for wrap in WRAPS:
            got = WR().wrap_index(k, n, wrap)
            assert got.tolist() == [s_wrap(int(x), n, wrap) for x in k], (n, wrap)
            assert ((got >= 0) & (got < n)).all()
    x = np.array([np.nan, np.inf, -np.inf, 3e9, -3e9, 2.0 ** 31, -2.0 ** 31, -1e-45, -0.0, 2.0 ** 24 + 1, -0.5, 2.5,
                  np.nextafter(F32(2.0 ** 31), F32(0)), np.nextafter(F32(-2.0 ** 31), F32(0))], F32)
    got = WR().ifloor(x)
    assert got.tolist() == [s_ifloor(a) for a in x]
    assert got.tolist()[:10] == [0, 0, 0, 0, 0, 0, 0, -1, 0, 2 ** 24]
    assert (got >= -2 ** 31).all() and (got + 1 <= 2 ** 31 - 1).all()


@x86
@pytest.mark.parametrize("wrap", WRAPS)
@pytest.mark.parametrize("tshape", SHAPES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_wrap_equals_clamp_inside_the_texture(tshape, wrap):
    """Nearest where 0 <= u*tw < tw and 0 <= (1-v)*th < th, bilinear where 0 <= sx <= tw-1 and 0 <= sy <= th-1: the clamp
    rule's texel / blend bit for bit.  Just below 0, nearest picks the last column (repeat) or column 0 (mirror)."""
    th, tw = tshape
    tex = random_texture(7, th, tw)
    rng = np.random.default_rng(th + tw)
    u = np.concatenate([rng.uniform(-0.1, 1.1, 20000), adversarial(tw)[:400]]).astype(F32)
    v = np.concatenate([rng.uniform(-0.1, 1.1, 20000), adversarial(th)[:400]]).astype(F32)
    v = np.resize(v, u.size)
    with np.errstate(all="ignore"):
        px, py = u * F32(tw), (F32(1) - v) * F32(th)
        sx, sy = px - F32(0.5), py - F32(0.5)
    inside = (px >= 0) & (px < tw) & (py >= 0) & (py < th)
    assert inside.sum() > 10000
    assert bits_equal(WR().nearest_texels(u[inside], v[inside], tex, wrap), WR().nearest_texels(u[inside], v[inside], tex, "clamp"))
    inner = (sx >= 0) & (sx <= tw - 1) & (sy >= 0) & (sy <= th - 1)
    if tw > 1 and th > 1:
        assert inner.sum() > 10000
    assert bits_equal(WR().bilinear_texels(u[inner], v[inner], tex, wrap), TM().bilinear_texels(u[inner], v[inner], tex))
    below = np.full(1, np.nextafter(F32(0), F32(-1)), F32)
    got = WR().nearest_texels(below, np.full(1, 0.5, F32), tex, wrap)
    assert bits_equal(got, tex[th // 2 if th > 1 else 0, tw - 1 if wrap == "repeat" else 0][None].astype(F32))


@pytest.mark.parametrize("wrap", WRAPS)
@pytest.mark.parametrize("tshape", SHAPES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_bilinear_at_texel_centres_is_wrapped_nearest(tshape, wrap):
    th, tw = tshape
    tex = random_texture(9, th, tw)
    c = np.arange(-2 * tw - 1, 3 * tw + 2)
    r = np.resize(np.arange(-2 * th - 1, 3 * th + 2), c.size)
    u = ((c + 0.5) / tw).astype(F32)
    v = (1 - (r + 0.5) / th).astype(F32)
    with np.errstate(all="ignore"):
        centre = ((u * F32(tw) - F32(0.5)) == c) & (((F32(1) - v) * F32(th) - F32(0.5)) == r)
    assert centre.sum() > c.size // 4
    assert bits_equal(WR().bilinear_texels(u[centre], v[centre], tex, wrap), WR().nearest_texels(u[centre], v[centre], tex, wrap))


@pytest.mark.parametrize("tshape", [(1, 1), (4, 16), (32, 8), (256, 512)], ids=lambda s: f"{s[0]}x{s[1]}")
def test_periodicity_and_mirror_symmetry(tshape):
    """Dyadic coordinates and power-of-two sizes: repeat at u + m equals repeat at u (every filter); the mirror index of k is
    that of -1 - k, and mirror at u + 2m equals mirror at u."""
    th, tw = tshape
    tex = random_texture(11, th, tw)
    j = np.arange(-64, 65)
    u, v = np.meshgrid((j / 64.0).astype(F32), (j[::3] / 64.0).astype(F32))
    u, v = u.ravel(), v.ravel()
    levels = MIP().mip_chain(tex)
    lc = np.resize(np.array([0, 0.25, 0.5, 1, len(levels) - 1], F32), u.size).clip(0, len(levels) - 1)
    for m in (1, -1, 3, -7, 64):
        for wrap, period in (("repeat", m), ("mirror", 2 * m)):
            du, dv = (u + F32(period)).astype(F32), (v - F32(period)).astype(F32)
            assert bits_equal(WR().nearest_texels(du, dv, tex, wrap), WR().nearest_texels(u, v, tex, wrap)), (m, wrap)
            assert bits_equal(WR().bilinear_texels(du, dv, tex, wrap), WR().bilinear_texels(u, v, tex, wrap)), (m, wrap)
            assert bits_equal(WR().trilinear_texels(du, dv, lc, levels, wrap), WR().trilinear_texels(u, v, lc, levels, wrap))
    for n in (tw, th, 1 << 30):
        k = np.arange(-5 * min(n, 64), 5 * min(n, 64) + 1)
        assert np.array_equal(WR().wrap_index(k, n, "mirror"), WR().wrap_index(-1 - k, n, "mirror"))
        assert np.array_equal(WR().wrap_index(k, n, "repeat"), WR().wrap_index(k + n, n, "repeat"))


@pytest.mark.parametrize("wrap", WRAPS)
def test_trilinear_at_level_zero_and_one_texel_levels(wrap):
    """lc == 0 is wrapped bilinear of the texture; every tap of a 1 x 1 level is its texel whatever the coordinate (with
    channels 0, 1 and 128 the blend of that texel with itself is exact, so the colour is the texel)."""
    tex = random_texture(13, 61, 47)
    levels = MIP().mip_chain(tex)
    u, v = _grid((61, 47))
    assert bits_equal(WR().trilinear_texels(u, v, np.zeros(u.size, F32), levels, wrap), WR().bilinear_texels(u, v, tex, wrap))
    one = np.array([[[0, 1, 128]]], np.uint8)
    want = np.tile(one[0, 0].astype(F32), (u.size, 1))
    assert bits_equal(WR().bilinear_texels(u, v, one, wrap), want)
    assert bits_equal(WR().nearest_texels(u, v, one, wrap), want)
    assert bits_equal(WR().trilinear_texels(u, v, np.zeros(u.size, F32), [one], wrap), want)
    sq = np.broadcast_to(one, (8, 8, 3)).copy()      # its last level (lc = 3) is 1 x 1
    chain = MIP().mip_chain(sq)
    assert chain[-1].shape[:2] == (1, 1)
    for lc in (F32(3), F32(2.5)):
        assert bits_equal(WR().trilinear_texels(u, v, np.full(u.size, lc, F32), chain, wrap), want)


def _screen_quad(h, w, uv_lo, uv_hi):
    """Two triangles covering the whole h x w frame at depth 1, fov 90, texture coordinates from uv_lo at the top left to
    uv_hi at the bottom right (u along x, v along y)."""
    z = F32(1.0)
    xs, ys = F32(w / 2.0), F32(h / 2.0)

    def corner(px, py):
        return ((F32(px) / xs - F32(1)) * z, (F32(py) / ys - F32(1)) * z, z)
    tl, tr, bl, br = corner(-1, -1), corner(w + 1, -1), corner(-1, h + 1), corner(w + 1, h + 1)
    v = np.array([[tl, tr, bl], [tr, br, bl]], F32)
    n = np.zeros_like(v)
    n[..., 2] = -1
    a, b = uv_lo, uv_hi
    ttl, ttr, tbl, tbr = (a, a, 0), (b, a, 0), (a, b, 0), (b, b, 0)
    uv = np.array([[ttl, ttr, tbl], [ttr, tbr, tbl]], F32)
    return v, uv, n


@x86
@pytest.mark.parametrize("filt", ["nearest", "bilinear", "trilinear"])
@pytest.mark.parametrize("wrap", WRAPS)
def test_full_screen_quad_spanning_several_periods(wrap, filt):
    """A quad over the whole frame with (u, v) from -3 to 4 at its corners: at every drawn pixel the oracle's colour is the texel (or blend)
    the rule gives for that pixel's interpolated (u, v) -- found here by a plain oracle_render of the coordinates -- and the
    frame shows every period."""
    h, w = 96, 128
    v, uv, n = _screen_quad(h, w, -3.0, 4.0)
    tex = random_texture(17, 13, 11)
    plain = O().OracleFiller(h, w)
    plain.render_arrays(v, uv, n)
    drawn = plain.get_z_buffer() < F32(1e6)
    assert drawn.all()
    uu, vv = plain.get_color_buffer()[..., 0], plain.get_color_buffer()[..., 1]
    assert uu.min() < -2 and uu.max() > 3 and vv.min() < -2 and vv.max() > 3      # the corners lie outside the frame
    o = WR().TexturedOracleFiller(h, w, wrap=wrap)
    o.render_arrays(v, uv, n, texture=tex, filter=filt)
    got = o.get_color_buffer()
    assert bits_equal(o.get_z_buffer(), plain.get_z_buffer()) and bits_equal(o.get_normals_buffer(), plain.get_normals_buffer())
    if filt == "nearest":
        want = _scalar(s_nearest, uu.ravel(), vv.ravel(), tex, wrap)
    elif filt == "bilinear":
        want = _scalar(s_bilinear, uu.ravel(), vv.ravel(), tex, wrap)
    else:       # the quad magnifies (13 x 11 texels over 7 periods on 128 x 96 pixels is less than one texel per pixel)
        assert tex.shape[1] * 7 < w and tex.shape[0] * 7 < h
        want = _scalar(s_bilinear, uu.ravel(), vv.ravel(), tex, wrap)
    assert bits_equal(got.reshape(-1, 3), want)
    periods = {math.floor(float(x)) for x in uu.ravel()}
    assert periods >= set(range(-2, 4))


@pytest.mark.parametrize("filt", ["nearest", "bilinear", "trilinear"])
@pytest.mark.parametrize("persp", [False, True])
def test_clamp_delegates_to_the_existing_oracles(filt, persp):
    from test_gpu_texture import _scene
    m, uv = _scene(5)
    tex = random_texture(5, 61, 47)
    a = WR().TexturedOracleFiller(128, 160)
    a.render_arrays(m._vertices_by_triangles, uv, m._normals_by_triangles, texture=tex, perspective=persp, filter=filt)
    b = MIP().TexturedOracleFiller(128, 160)
    b.render_arrays(m._vertices_by_triangles, uv, m._normals_by_triangles, texture=tex, perspective=persp, filter=filt)
    for x, y in zip((a.get_z_buffer(), a.get_color_buffer(), a.get_normals_buffer()),
                    (b.get_z_buffer(), b.get_color_buffer(), b.get_normals_buffer())):
        assert bits_equal(x, y)


def test_refusals():
    tex = random_texture(1, 4, 4)
    u = np.zeros(3, F32)
    for bad in ("Repeat", "wrap", "border", None):
        with pytest.raises(ValueError):
            WR().nearest_texels(u, u, tex, bad)
        with pytest.raises(ValueError):
            WR().TexturedOracleFiller(8, 8, wrap=bad)
    with pytest.raises(ValueError):
        WR().wrap_index(np.zeros(2, np.int64), 4, "clamp")
