"""Scenes in batched views (oracle/scene_oracle.py; crb_render_scene_views, DESIGN 2) on the CPU: the oracle against a scalar
per-triangle restatement of the rule, the two equivalences with crb_render_views_ids, and the helpers views.scene_views and
views.concat_meshes."""
import numpy as np
import pytest

from conftest import random_scene

F32 = np.float32


def SC():
    from oracle import scene_oracle
    return scene_oracle


def VW():
    from cython3dmodelrenderer_b200 import views
    return views


def same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    if a.dtype == F32:
        a, b = a.view(np.uint32), np.asarray(b, F32).view(np.uint32)
    return a.shape == b.shape and bool(np.all(a == b))


def random_pose(rng, pad=0.0):
    """A rigid {R, p, q, pad}: a random rotation (QR of a Gaussian matrix), a pivot and a translation"""
    q, r = np.linalg.qr(rng.standard_normal((3, 3)))
    R = q * np.sign(np.diag(r))
    if np.linalg.det(R) < 0:
        R[:, 0] = -R[:, 0]
    M = VW().view_matrix(R, p=rng.uniform(-0.3, 0.3, 3), q=rng.uniform(-0.3, 0.3, 3) + np.array([0.0, 0.0, 1.2]))
    M[15] = F32(pad)
    return M


def small_scene(seed=3, T=240, K=5):
    """Interleaved (non-contiguous) object indices, some outside [0, K), and per-view poses with hidden objects (pads of 1,
    NaN and -0, the last one shown)"""
    rng = np.random.default_rng(seed)
    m = random_scene(seed, T=T)
    v = m._vertices_by_triangles.copy()
    v[..., 2] -= F32(1.0)                                      # object space about the origin; the poses put them at z ~ 1.2
    tri_obj = rng.integers(0, K, T).astype(np.int32)
    tri_obj[::17] = K                                          # out of range
    tri_obj[5::23] = -1
    V = 3
    views = np.stack([np.stack([random_pose(rng) for _ in range(K)]) for _ in range(V)])
    views[0, 1, 15] = F32(1.0)
    views[1, 2, 15] = F32(np.nan)
    views[2, 3, 15] = -F32(0.0)
    views[2, 0, 15] = F32(-1e-30)
    return v, m._colors_by_triangles, m._normals_by_triangles, tri_obj, views


def scalar_camera_space(v, c, n, tri_obj, views_v):
    """The rule one triangle at a time with float32 scalars: view_point / view_normal of the triangle's object transform"""
    K = len(views_v)
    out_v, out_c, out_n, kept = [], [], [], []
    for t in range(len(v)):
        k = int(tri_obj[t])
        if not 0 <= k < K or not views_v[k, 15] == 0:
            continue
        M = [F32(x) for x in views_v[k]]
        tv, tn = np.empty((3, 3), F32), np.empty((3, 3), F32)
        for j in range(3):
            d = [F32(v[t, j, i] - M[9 + i]) for i in range(3)]
            for r in range(3):
                tv[j, r] = F32(F32(F32(F32(M[3 * r] * d[0]) + F32(M[3 * r + 1] * d[1])) + F32(M[3 * r + 2] * d[2])) + M[12 + r])
                tn[j, r] = F32(F32(F32(M[3 * r] * n[t, j, 0]) + F32(M[3 * r + 1] * n[t, j, 1])) + F32(M[3 * r + 2] * n[t, j, 2]))
        out_v.append(tv); out_n.append(tn); out_c.append(c[t]); kept.append(t)
    sh = lambda a: np.array(a, F32).reshape(-1, 3, 3)
    return sh(out_v), sh(out_c), sh(out_n), np.array(kept, np.int64)


@pytest.mark.parametrize("view", [0, 1, 2])
def test_camera_space_against_scalar_restatement(view):
    v, c, n, tri_obj, views = small_scene()
    got = SC().camera_space(v, c, n, tri_obj, views[view])
    want = scalar_camera_space(v, c, n, tri_obj, views[view])
    for g, w, name in zip(got, want, ("v", "c", "n", "kept")):
        assert same(g, w), f"view {view}: {name} differs"
    assert 0 < len(got[3]) < len(v)
    with np.errstate(invalid="ignore"):
        hidden = ~(views[view, :, 15] == 0)
    assert not np.isin(tri_obj[got[3]], np.flatnonzero(hidden)).any()


@pytest.mark.parametrize("view", [0, 1, 2])
def test_render_against_scalar_restatement(view):
    """The oracle's frame equals oracle_render of the scalar camera-space triangles, and tri_id maps through the kept indices"""
    from oracle import ids_oracle as ID
    v, c, n, tri_obj, views = small_scene()
    o, ids, bary = SC().render(128, 160, v, c, n, tri_obj, views[view], fov=60.0)
    sv, sc, sn, kept = scalar_camera_space(v, c, n, tri_obj, views[view])
    w = ID.IdsOracleFiller(128, 160, fov=60.0)
    w.render_arrays(sv, sc, sn)
    for a, b in ((o.z_buffer, w.z_buffer), (o.color_buffer, w.color_buffer), (o.normals_buffer, w.normals_buffer), (bary, w.bary)):
        assert same(a, b)
    assert same(ids, np.where(w.tri_id >= 0, kept[np.maximum(w.tri_id, 0)], -1))
    assert (ids >= 0).sum() > 500
    assert np.all(np.isin(ids[ids >= 0], kept))


def test_render_with_near_clip_against_clip_oracle():
    from oracle import clip_oracle as CL
    v, c, n, tri_obj, views = small_scene()
    views = views.copy()
    views[..., 14] -= F32(1.0)                                 # objects straddle z_near
    o, ids, _ = SC().render(96, 96, v, c, n, tri_obj, views[0], fov=90.0, z_near=0.2, near_clip=True)
    sv, sc, sn, kept = scalar_camera_space(v, c, n, tri_obj, views[0])
    w, wids = CL.render(96, 96, sv, sc, sn, fov=90.0, z_near=0.2)
    assert same(o.z_buffer, w.z_buffer) and same(o.color_buffer, w.color_buffer) and same(o.normals_buffer, w.normals_buffer)
    assert same(ids, np.where(wids >= 0, kept[np.maximum(wids, 0)], -1))
    assert (ids >= 0).sum() > 100


def test_nothing_shown():
    v, c, n, tri_obj, views = small_scene()
    hidden = views[0].copy()
    hidden[:, 15] = F32(1.0)
    o, ids, bary = SC().render(64, 64, v, c, n, tri_obj, hidden)
    assert (ids == -1).all() and (o.z_buffer == F32(1e6)).all() and (bary == 0).all()


def views_ids_oracle(h, w, v, c, n, view, fov):
    """One view of crb_render_views_ids: oracle_render of transform_arrays_host(view), with tri_id and bary"""
    from oracle import ids_oracle as ID
    tv, tn = VW().transform_arrays_host(view, v, n)
    o = ID.IdsOracleFiller(h, w, fov=fov)
    o.render_arrays(tv, c, tn)
    return o


def test_equivalence_one_object_is_render_views_ids():
    v, c, n, _, _ = small_scene()
    cams = VW().orbit_views(4)
    tri_obj = np.zeros(len(v), np.int32)
    for k in range(4):
        view = cams[k].copy()
        view[14] += F32(0.5)
        o, ids, bary = SC().render(96, 128, v, c, n, tri_obj, view[None], fov=45.0)
        w = views_ids_oracle(96, 128, v, c, n, view, 45.0)
        for a, b in ((o.z_buffer, w.z_buffer), (o.color_buffer, w.color_buffer), (o.normals_buffer, w.normals_buffer),
                     (ids, w.tri_id), (bary, w.bary)):
            assert same(a, b), f"view {k}"


def test_equivalence_equal_transforms_is_render_views_ids():
    v, c, n, tri_obj, _ = small_scene()
    tri_obj = tri_obj % 5                                      # every triangle in range
    cams = VW().orbit_views(3)
    for k in range(3):
        view = cams[k].copy()
        view[14] += F32(0.5)
        o, ids, bary = SC().render(96, 128, v, c, n, tri_obj, np.repeat(view[None], 5, axis=0), fov=45.0)
        w = views_ids_oracle(96, 128, v, c, n, view, 45.0)
        for a, b in ((o.z_buffer, w.z_buffer), (o.color_buffer, w.color_buffer), (o.normals_buffer, w.normals_buffer),
                     (ids, w.tri_id), (bary, w.bary)):
            assert same(a, b), f"view {k}"


def test_scene_views_composes_camera_and_pose():
    """scene_views against the two transforms applied one after the other in float64, and the pad carried through"""
    rng = np.random.default_rng(11)
    V, K = 4, 6
    cams = np.stack([random_pose(rng) for _ in range(V)])
    poses = np.stack([random_pose(rng, pad=1.0 if k == 2 else 0.0) for k in range(K)])
    per_view = np.stack([np.stack([random_pose(rng) for _ in range(K)]) for _ in range(V)])
    pts = rng.uniform(-1, 1, (50, 3))

    def apply(M, x):
        M = np.asarray(M, np.float64)
        return (M[:9].reshape(3, 3) @ (x - M[9:12]).T).T + M[12:15]

    for P in (poses, per_view):
        S = VW().scene_views(cams, P)
        assert S.shape == (V, K, 16) and S.dtype == F32
        for vi in range(V):
            for k in range(K):
                pk = P[k] if P.ndim == 2 else P[vi, k]
                want = apply(cams[vi], apply(pk, pts))
                assert np.abs(apply(S[vi, k], pts) - want).max() < 1e-5
                assert same(S[vi, k, 15:], pk[15:])
    # the camera alone: an identity pose gives back the camera's R and q (p = 0)
    ident = VW().view_matrix(p=(0.0, 0.0, 0.0))
    S = VW().scene_views(cams, ident[None])
    assert np.allclose(S[:, 0, :9], cams[:, :9], atol=1e-7)
    assert np.allclose(S[:, 0, 12:15], (cams[:, :9].reshape(V, 3, 3).astype(np.float64) @ -cams[:, 9:12, None].astype(np.float64))[..., 0]
                       + cams[:, 12:15], atol=1e-6)


def test_concat_meshes():
    rng = np.random.default_rng(2)
    meshes = [tuple(rng.standard_normal((t, 3, 3)).astype(F32) for _ in range(3)) for t in (5, 1, 300)]
    v, c, n, tri_obj = VW().concat_meshes(meshes)
    assert v.shape == c.shape == n.shape == (306, 3, 3) and v.dtype == c.dtype == n.dtype == F32
    assert tri_obj.dtype == np.int32 and tri_obj.tolist() == [0] * 5 + [1] + [2] * 300
    for k, i in ((0, 0), (1, 5), (2, 6)):
        assert same(v[i], meshes[k][0][0]) and same(c[i], meshes[k][1][0]) and same(n[i], meshes[k][2][0])
    with pytest.raises(ValueError):
        VW().concat_meshes([])
