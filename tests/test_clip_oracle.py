"""Near-plane clipping (oracle/clip_oracle.py; CRB_CLIP_NEAR, DESIGN 2) on the CPU: the NumPy clip against a scalar
restatement of the rule on adversarial corners, its properties, and the defect it removes, drawn with the pinned oracle."""
import numpy as np
import pytest

F32 = np.float32


def CL():
    from oracle import clip_oracle
    return clip_oracle


def scalar_clip(v, c, n, z_near):
    """The rule, one triangle at a time, with float32 scalars: the polygon walk, I(i, o), the pieces."""
    zn = F32(z_near)
    pieces, parents = [], []
    for t in range(len(v)):
        A = [np.concatenate([v[t, k], n[t, k], c[t, k]]).astype(F32) for k in range(3)]
        inside = [bool(A[k][2] >= zn) for k in range(3)]
        poly = []
        for a in range(3):
            b = (a + 1) % 3
            if inside[a]:
                poly.append(A[a])
            if inside[a] != inside[b]:
                i, o = (A[a], A[b]) if inside[a] else (A[b], A[a])
                with np.errstate(all="ignore"):
                    s = F32(F32(zn - i[2]) / F32(o[2] - i[2]))
                    p = np.array([F32(i[k] + F32(s * F32(o[k] - i[k]))) for k in range(9)], F32)
                p[2] = zn
                poly.append(p)
        assert len(poly) in (0, 3, 4)
        if len(poly) >= 3:
            pieces.append([poly[0], poly[1], poly[2]]); parents.append(t)
        if len(poly) == 4:
            pieces.append([poly[0], poly[2], poly[3]]); parents.append(t)
    P = np.array(pieces, F32).reshape(-1, 3, 9)
    return P[:, :, 0:3], P[:, :, 6:9], P[:, :, 3:6], np.array(parents, np.int64)


def same(a, b):
    a, b = np.asarray(a, F32), np.asarray(b, F32)
    return a.shape == b.shape and bool(np.all((a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))))


def adversarial(seed, T, zn):
    """Triangles whose corners sit on zn, one ulp either side, on both sides of it, at NaN and +-inf, plus slivers."""
    rng = np.random.default_rng(seed)
    zn = F32(zn)
    v = rng.uniform(-2, 2, (T, 3, 3)).astype(F32)
    v[..., 2] = rng.uniform(-3, 3, (T, 3)).astype(F32) + zn
    special = np.array([zn, np.nextafter(zn, F32(np.inf)), np.nextafter(zn, F32(-np.inf)), F32(0), -F32(0), -zn, F32(2) * zn,
                        np.nan, np.inf, -np.inf, F32(1e30), F32(-1e30)], F32)
    m = rng.random((T, 3)) < 0.4
    v[..., 2][m] = rng.choice(special, size=int(m.sum()))
    v[:T // 8, :, 2] = zn                                             # all three on the plane
    sl = slice(T // 8, T // 4)                                        # slivers: corners 1 and 2 nearly equal
    v[sl, 2] = v[sl, 1] + rng.uniform(-1e-6, 1e-6, v[sl, 1].shape).astype(F32)
    n = rng.standard_normal((T, 3, 3)).astype(F32)
    c = (rng.random((T, 3, 3)) * 255).astype(F32)
    return v, c, n


@pytest.mark.parametrize("zn", [0.1, 0.5, 1.0, 1e-30, 3e4, 1e30])
@pytest.mark.parametrize("seed", range(3))
def test_clip_equals_scalar_rule(seed, zn):
    v, c, n = adversarial(seed, 400, zn)
    got, want = CL().clip(v, c, n, zn), scalar_clip(v, c, n, zn)
    for g, w in zip(got[:3], want[:3]):
        assert same(g, w)
    assert np.array_equal(got[3], want[3])


def test_crossing_at_s_zero_and_one():
    # corner 0 on the plane (inside, s = 0 for the edge to an outside corner), corner 2 one ulp below it (s = 1 from corner 1)
    zn = F32(0.5)
    below = np.nextafter(zn, F32(-1))
    v = np.array([[[0, 0, zn], [1, 0, 2], [0, 1, below]]], F32)
    c = np.arange(9, dtype=F32).reshape(1, 3, 3)
    n = -np.ones((1, 3, 3), F32)
    pv, pc, pn, parent = CL().clip(v, c, n, zn)
    assert list(parent) == [0, 0]
    for g, w in zip((pv, pc, pn), scalar_clip(v, c, n, zn)[:3]):
        assert same(g, w)
    assert np.all(pv[..., 2] >= zn)


@pytest.mark.parametrize("seed", range(4))
def test_properties(seed):
    zn = F32(0.25)
    v, c, n = adversarial(seed, 300, zn)
    pv, pc, pn, parent = CL().clip(v, c, n, zn)
    # every piece corner is at z >= zn, or derives from a NaN (a NaN z is outside, a crossing towards it is NaN-derived)
    z = pv[..., 2]
    assert np.all((z >= zn) | np.isnan(pv).any(axis=2) | np.isnan(v[parent]).any(axis=(1, 2))[:, None])
    # all-inside triangles come back unchanged, bit for bit, as piece 0 and no piece 1
    with np.errstate(invalid="ignore"):
        allin = np.all(v[..., 2] >= zn, axis=1)
    for t in np.flatnonzero(allin):
        k = np.flatnonzero(parent == t)
        assert len(k) == 1 and same(pv[k[0]], v[t]) and same(pc[k[0]], c[t]) and same(pn[k[0]], n[t])
    # the two pieces of a quad share the diagonal p0-p2: piece 1's (p0, p2) are piece 0's (p0, p2)
    for t in np.unique(parent):
        k = np.flatnonzero(parent == t)
        if len(k) == 2:
            assert same(pv[k[1], 0], pv[k[0], 0]) and same(pv[k[1], 1], pv[k[0], 2])
            assert same(pc[k[1], 1], pc[k[0], 2]) and same(pn[k[1], 1], pn[k[0], 2])
    # a triangle entirely outside has no piece
    with np.errstate(invalid="ignore"):
        allout = ~np.any(v[..., 2] >= zn, axis=1)
    assert not np.isin(np.flatnonzero(allout), parent).any()


def test_all_inside_scene_unchanged():
    from conftest import random_scene
    m = random_scene(11, T=500)
    v = m._vertices_by_triangles.copy()
    v[..., 2] = np.abs(v[..., 2]) + F32(0.5)
    pv, pc, pn, parent = CL().clip(v, m._colors_by_triangles, m._normals_by_triangles, 0.5)
    assert np.array_equal(parent, np.arange(len(v)))
    assert same(pv, v) and same(pc, m._colors_by_triangles) and same(pn, m._normals_by_triangles)


def _floor():
    """A floor triangle under the camera running from z = 3 to z = -1, facing the camera (normals -z)."""
    v = np.array([[[-2, -0.5, 3], [2, -0.5, 3], [0, -0.5, -1]]], F32)
    n = np.tile(np.array([0, 0, -1], F32), (1, 3, 1))
    c = np.full((1, 3, 3), 200, F32)
    return v, c, n


def test_floor_stays_below_the_horizon():
    from oracle import oracle as O
    v, c, n = _floor()
    # without clipping the corner behind the camera projects mirrored: the floor reaches into the sky (upper rows, which
    # are the high row indices of the buffers: rows count from the bottom, run.py:26 flips them)
    o = O.OracleFiller(64, 64, fov=60)
    o.render_arrays(v, c, n)
    rows = np.flatnonzero((o.z_buffer < 1e6).any(axis=1))
    assert rows.size and rows.max() > 32
    # with clipping: the floor covers rows below the horizon (row 32 is the horizon of a camera at height 0.5 looking along z)
    oc, ids = CL().render(64, 64, v, c, n, fov=60, z_near=0.1)
    rows = np.flatnonzero((oc.z_buffer < 1e6).any(axis=1))
    assert rows.size and rows.max() < 32
    assert set(np.unique(ids)) == {-1, 0}
    assert np.array_equal(ids >= 0, oc.z_buffer < 1e6)


def test_scene_behind_the_camera_draws_nothing():
    from oracle import oracle as O
    v = np.array([[[-0.5, -0.5, -2], [0.5, -0.5, -2], [0, 0.5, -2]]], F32)
    n = np.tile(np.array([0, 0, -1], F32), (1, 3, 1))
    c = np.full((1, 3, 3), 200, F32)
    o = O.OracleFiller(64, 64, fov=60)
    o.render_arrays(v, c, n)
    assert int((o.z_buffer < 1e6).sum()) > 0                 # the defect: drawn at depth just above 1
    oc, ids = CL().render(64, 64, v, c, n, fov=60, z_near=0.1)
    assert int((oc.z_buffer < 1e6).sum()) == 0 and np.all(ids == -1)


def test_tie_order_follows_pieces():
    """Two coplanar copies of a straddling triangle: the later parent wins every pixel, both pieces included."""
    v, c, n = _floor()
    v2, c2, n2 = (np.concatenate([a, a]) for a in (v, c, n))
    c2[1] = 50
    oc, ids = CL().render(64, 64, v2, c2, n2, fov=60, z_near=0.1)
    drawn = oc.z_buffer < 1e6
    assert drawn.any() and np.all(ids[drawn] == 1) and np.allclose(oc.color_buffer[drawn], 50, atol=1e-3)
