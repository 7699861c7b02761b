"""The oracle of trilinear mip filtering (oracle/texture_mip_oracle.py; DESIGN 2) against its definition, on the CPU: the chain
against a scalar restatement, the log2 substitute, the winner ids against oracle_render's own buffers, the level of detail
against analytic and finite-difference expectations, the bilinear equality at lambda_c == 0, the regimes the GPU tests' scenes
reach, and that the mode removes the aliasing of a minified checkerboard."""
import numpy as np
import pytest

from conftest import load_indexed
from test_gpu_texture import SEEDS, _base, _scene
from test_texture_filter_oracle import _depth_triangle
from test_texture_oracle import random_texture, random_uvs

F32 = np.float32


def O():
    from oracle import oracle
    return oracle


def TM():
    from oracle import texture_modes_oracle
    return texture_modes_oracle


def MIP():
    from oracle import texture_mip_oracle
    return texture_mip_oracle


def mip_scalar(level, r, c):
    """Texel (r, c) of the next level, restated texel by texel."""
    h, w = level.shape[:2]
    r0, r1, c0, c1 = min(2 * r, h - 1), min(2 * r + 1, h - 1), min(2 * c, w - 1), min(2 * c + 1, w - 1)
    return [(int(level[r0, c0, k]) + int(level[r0, c1, k]) + int(level[r1, c0, k]) + int(level[r1, c1, k]) + 2) >> 2
            for k in range(3)]


@pytest.mark.parametrize("tshape", [(1, 1), (1, 7), (7, 1), (5, 3), (709, 709), (333, 4097), (2048, 2048)],
                         ids=lambda s: f"{s[0]}x{s[1]}")
def test_mip_chain_matches_scalar_restatement(tshape):
    th, tw = tshape
    levels = MIP().mip_chain(random_texture(th + tw, th, tw))
    assert len(levels) == MIP().levels_of(th, tw) == 1 + int(np.floor(np.log2(max(th, tw))))
    assert levels[-1].shape[:2] == (1, 1)
    rng = np.random.default_rng(th * tw)
    for k in range(1, len(levels)):
        prev, cur = levels[k - 1], levels[k]
        assert cur.shape[:2] == (max(1, prev.shape[0] >> 1), max(1, prev.shape[1] >> 1))
        if cur.shape[0] * cur.shape[1] <= 4096:
            pts = [(r, c) for r in range(cur.shape[0]) for c in range(cur.shape[1])]
        else:     # every edge texel (where odd sizes clamp) and a random sample
            hh, ww = cur.shape[:2]
            pts = [(r, c) for r in (0, hh - 1) for c in range(ww)] + [(r, c) for c in (0, ww - 1) for r in range(hh)]
            pts += list(zip(rng.integers(0, hh, 2000), rng.integers(0, ww, 2000)))
        for r, c in pts:
            assert list(cur[r, c]) == mip_scalar(prev, int(r), int(c)), (tshape, k, r, c)
    packed = MIP().pack_chain(levels)
    assert packed.size == sum(t.shape[0] * t.shape[1] for t in levels) < 2 ** 31
    t0 = levels[0].reshape(-1, 3).astype(np.uint32)
    assert np.array_equal(packed[:t0.shape[0]], t0[:, 0] | (t0[:, 1] << 8) | (t0[:, 2] << 16))


def test_log2_substitute():
    L2 = MIP().log2_substitute
    ks = np.arange(-149, 128)
    p = np.ldexp(np.ones(ks.size, F32), ks).astype(F32)       # every power of two of float32, subnormals included
    assert (p > 0).all() and np.isfinite(p).all()
    assert np.array_equal(L2(p), ks.astype(F32))
    x = np.sort(np.random.default_rng(0).uniform(-40, 40, 200000)).astype(np.float64)
    r2 = np.exp2(x).astype(F32)
    y = L2(r2)
    assert (np.diff(y) >= 0).all()
    assert np.abs(y - np.log2(r2.astype(np.float64))).max() < 0.0861
    dense = np.nextafter(F32(1), F32(2)) * np.arange(1, 100000, dtype=F32)
    assert (np.diff(L2(np.sort(dense))) >= 0).all()
    sub = np.array([1e-45, 3e-40, 1.17e-38], F32)
    assert np.array_equal(np.diff(L2(sub)) > 0, [True, True])
    spec = L2(np.array([0.0, -0.0, np.inf, np.nan], F32))
    assert spec[0] == -np.inf and spec[1] == -np.inf and spec[2] == np.inf and np.isnan(spec[3])


def _edge_scenes(h, w):
    import test_gpu_edges as E
    for i, name in enumerate(sorted(E.FAMILIES)):
        m = E.family(name, h, w)
        yield f"family {name}", m._vertices_by_triangles, m._normals_by_triangles, random_uvs(50 + i, m._vertices_by_triangles.shape[0]), E.FOV


def _seeded_scenes():
    for seed in SEEDS:
        m, uv = _scene(seed)
        yield f"seed {seed}", m._vertices_by_triangles, m._normals_by_triangles, uv, 90.0


def _all_scenes(h, w):
    yield from _seeded_scenes()
    yield from _edge_scenes(h, w)


@pytest.mark.parametrize("composite", [False, True])
def test_winner_ids_restate_the_oracles_depth_and_normals(composite):
    h, w = 200, 333
    for what, v, n, uv, fov in _all_scenes(h, w):
        o = O().OracleFiller(h, w, fov=fov)
        if composite:
            o.render_arrays(*_base())
        z_before = o.get_z_buffer().copy()
        # the pixels this render draws, by the NaN-colour render of texture_oracle
        scratch = O().OracleFiller(h, w, fov=fov)
        scratch.z_buffer[...] = z_before
        scratch.render_arrays(v, np.full(v.shape, np.nan, F32), n)
        drawn = np.isnan(scratch.color_buffer[..., 0])
        o.render_arrays(v, np.zeros(v.shape, F32), n)
        ids = MIP().winner_ids(h, w, o.proj_mat.ravel(), v, n, o.get_z_buffer())
        assert np.array_equal(ids >= 0, drawn), what
        z, nb = MIP().restate(h, w, o.proj_mat.ravel(), v, n, ids)
        assert np.array_equal(z[drawn].view(np.uint32), o.get_z_buffer()[drawn].view(np.uint32)), what
        assert np.array_equal(nb[drawn].view(np.uint32), o.get_normals_buffer()[drawn].view(np.uint32)), what
        assert drawn.sum() > 0, what


def _quad(h, w, x0, y0, x1, y1, zs=(1.0, 1.0, 1.0, 1.0)):
    """Two triangles covering pixels [x0, x1) x [y0, y1) with corner depths zs (top-left, top-right, bottom-left, bottom-right)
    and texture coordinates (0,1) ... (1,0) across them."""
    a, _ = _depth_triangle(h, w, (x0, x1, x0), (y0, y0, y1), (zs[0], zs[1], zs[2]))
    b, _ = _depth_triangle(h, w, (x1, x1, x0), (y0, y1, y1), (zs[1], zs[3], zs[2]))
    v = np.concatenate([a, b])
    n = np.zeros_like(v)
    n[..., 2] = -1
    uv = np.array([[[0, 1, 0], [1, 1, 0], [0, 0, 0]], [[1, 1, 0], [1, 0, 0], [0, 0, 0]]], F32)
    return v, uv, n


@pytest.mark.parametrize("k", range(0, 7))
def test_screen_aligned_minification_gives_lambda_k(k):
    """A facing quad 32 pixels wide showing a 32 * 2^k texture: lambda is k up to the float32 rounding of the gradients."""
    h = w = 128
    size = 32 << k
    v, uv, n = _quad(h, w, 40, 40, 72, 72)
    tex = random_texture(k, size, size)
    for persp in (False, True):
        o = O().OracleFiller(h, w)
        ids, lam, lc = MIP().render_textured(o, v, uv, n, tex, perspective=persp, return_lod=True)
        assert lam.size > 800
        assert np.abs(lam - k).max() < 2e-3, (k, persp, lam.min(), lam.max())


def test_perspective_lambda_agrees_with_finite_differences():
    """Steeply tilted quads: lambda against 0.5 * log2 of the footprint of central differences (float64) of the perspective
    (u, v) = (U / W, V / W), within the log2 substitute's 0.043 and the differences' error."""
    h = w = 256
    cases = [(1.0, 1.0, 12.0, 12.0), (1.0, 20.0, 1.0, 20.0), (0.5, 3.0, 8.0, 40.0)]
    for zs in cases:
        v, uv, n = _quad(h, w, 20, 30, 230, 220, zs)
        tex = random_texture(1, 512, 512)
        o = O().OracleFiller(h, w)
        ids, lam, lc = MIP().render_textured(o, v, uv, n, tex, perspective=True, return_lod=True)
        ys, xs = np.nonzero(ids >= 0)
        scr = O().project(h, w, o.proj_mat.ravel(), v).astype(np.float64)
        slots = TM().perspective_slots(v, uv).astype(np.float64)

        def uv_at(t, px, py):
            x0, y0, x1, y1, x2, y2 = (scr[t, k, j] for k in range(3) for j in range(2))
            d = (x1 - x2) * (y0 - y2) - (y1 - y2) * (x0 - x2)
            b0 = ((x1 - x2) * (py - y2) - (y1 - y2) * (px - x2)) / d
            b1 = ((x2 - x0) * (py - y0) - (y2 - y0) * (px - x0)) / d
            b2 = 1 - b0 - b1
            U, V, W = ((slots[t, 0, j] * b0 + slots[t, 1, j] * b1 + slots[t, 2, j] * b2) for j in range(3))
            return U / W, V / W
        t = ids[ys, xs]
        e = 1e-3
        (ua, va), (ub, vb) = uv_at(t, xs + e, ys), uv_at(t, xs - e, ys)
        (uc, vc), (ud, vd) = uv_at(t, xs, ys + e), uv_at(t, xs, ys - e)
        ux, vx, uy, vy = (ua - ub) / (2 * e), (va - vb) / (2 * e), (uc - ud) / (2 * e), (vc - vd) / (2 * e)
        r2 = np.maximum((ux * 512) ** 2 + (vx * 512) ** 2, (uy * 512) ** 2 + (vy * 512) ** 2)
        want = 0.5 * np.log2(r2)
        assert lam.size > 10000
        assert np.abs(lam - want).max() < 0.05, (zs, np.abs(lam - want).max())
        assert lam.max() - lam.min() > 1.0, zs      # the quads are tilted enough for lambda to vary across them


def _lods(h, w, scenes, tshape, persp):
    out = []
    for what, v, n, uv, fov in scenes:
        o = O().OracleFiller(h, w, fov=fov)
        ids, lam, lc = MIP().render_textured(o, v, uv, n, random_texture(3, *tshape), perspective=persp, return_lod=True)
        out.append((what, o, ids, lam, lc))
    return out


@pytest.mark.parametrize("persp", [False, True])
def test_trilinear_is_bilinear_where_lambda_c_is_zero(persp):
    h, w = 200, 333
    for tshape in ((1, 7), (709, 709)):
        tex = random_texture(3, *tshape)
        for what, v, n, uv, fov in _all_scenes(h, w):
            o = O().OracleFiller(h, w, fov=fov)
            ids, lam, lc = MIP().render_textured(o, v, uv, n, tex, perspective=persp, return_lod=True)
            b = TM().TexturedOracleFiller(h, w, fov=fov)
            b.render_arrays(v, uv, n, texture=tex, perspective=persp, filter="bilinear")
            drawn = ids >= 0
            zero = np.zeros((h, w), bool)
            zero[drawn] = lc == 0
            assert np.array_equal(o.get_color_buffer()[zero].view(np.uint32), b.get_color_buffer()[zero].view(np.uint32)), what
            assert np.array_equal(o.get_z_buffer().view(np.uint32), b.get_z_buffer().view(np.uint32)), what
            if tshape == (1, 7):
                assert zero[drawn].sum() == 0 or (lc == 0).any()


def test_scene_families_reach_every_regime():
    """lambda_c == 0, a fractional lambda inside every level interval of a 709^2 chain, lambda clamped at the top level, and
    NaN lambda, over the scenes the GPU tests render (seeded, edge families, 256^2 T-Rex orbit views)."""
    from cython3dmodelrenderer_b200 import synthetic, views as VW
    h, w = 256, 256
    m = load_indexed("trex")
    uv = synthetic.spherical_uvs(m._vertices_by_triangles)
    views = VW.orbit_views(128, first=0, count=8, stride=16)
    trex = []
    for k in (0, 4):
        vk, nk = VW.transform_arrays_host(views[k], m._vertices_by_triangles, m._normals_by_triangles)
        trex.append((f"trex view {k}", vk, nk, uv, 45.0))
    for persp in (False, True):
        lam = np.concatenate([r[3] for r in _lods(h, w, list(_all_scenes(h, w)) + trex, (709, 709), persp)])
        top = MIP().levels_of(709, 709) - 1
        assert (np.nan_to_num(lam, nan=-1) <= 0).any(), persp
        for lv in range(top):
            assert ((lam > lv) & (lam < lv + 1)).any(), (persp, lv)
        assert (lam > top).any(), persp
        assert np.isnan(lam).any(), persp


def test_trilinear_removes_checkerboard_aliasing():
    """A floor receding from depth 1.2 to 30 with a one-texel checkerboard of 512^2: in the far half of its pixels (by depth)
    bilinear sampling still swings between the two squares, while trilinear averages the footprint.  Oracle numbers (256^2
    frame, perspective-correct): far-half variance of a channel 1897 bilinear against 0 trilinear (lambda >= 1.2 there, and
    every level from 1 on is uniform grey); the bar is a hundredth."""
    h = w = 256
    q = np.array([[-1, -0.6, 1.2], [1, -0.6, 1.2], [-1, -0.6, 30], [1, -0.6, 30]], F32)
    t = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [1, 1, 0]], F32)
    v, uv = np.stack([q[[0, 1, 2]], q[[1, 3, 2]]]), np.stack([t[[0, 1, 2]], t[[1, 3, 2]]])
    n = np.zeros_like(v)
    n[..., 2] = -1
    r, c = np.indices((512, 512))
    tex = np.repeat((((r + c) & 1) * 255).astype(np.uint8)[..., None], 3, axis=2)
    var = {}
    for filt in ("bilinear", "trilinear"):
        o = MIP().TexturedOracleFiller(h, w)
        o.render_arrays(v, uv, n, texture=tex, perspective=True, filter=filt)
        z = o.get_z_buffer()
        drawn = z < F32(1e6)
        far = drawn & (z > np.median(z[drawn]))
        assert far.sum() > 3000
        var[filt] = float(o.get_color_buffer()[far][:, 0].astype(np.float64).var())
    assert var["bilinear"] > 1000 and var["trilinear"] < 0.01 * var["bilinear"], var


def test_refusals():
    with pytest.raises(ValueError):
        MIP().TexturedOracleFiller(8, 8).render_arrays(*_base(), filter="trilinear")
    with pytest.raises(ValueError):
        MIP().mip_chain(np.zeros((4, 4, 3), np.float32))
