"""Batched views under general camera transforms, word for word against the oracle.

A view is 16 floats {R (9, row-major), p (3), q (3), pad}: v' = R (v - p) + q and n' = R n, each component evaluated as
((r0*d0 + r1*d1) + r2*d2) + q in float32 with one rounding per operation (views.py, crender_b200.h).  crender_b200.cu
evaluates it in view_point and view_normal (the vertices, the shade record's normals, k_transform_view), again by hand in the
z row of the normals the cull reads (once for full-frame fillers, once for band fillers), and a third time in the z row that
CRB_TEX_PERSPECTIVE divides by.  Orbit views about the y axis have R[1] = R[3] = R[5] = R[7] = 0, R[4] = 1 and q = p on the
z axis, so a wrong index among those zeros, x and y of p or q swapped, p and q exchanged or a reassociated sum all give the
values of the right transform there (test_orbit_views_cannot_tell_these_mistakes_apart).  The view families below can.

CPU: transform_arrays_host against R (v - p) + q in float64, within the float32 error bound, on every family; NumPy mutants
of the transform, each of which the families tell apart from it.  GPU: transform_view, and render_views (z, colour, normals,
uint8, fused Guro) on the T-Rex, random scenes and the edge families of test_gpu_edges, across batching, the rasterizer
shapes, band fillers, the row exchange and the six texture modes -- every view against the oracle fed the camera-space
arrays of transform_arrays_host.
"""
from fractions import Fraction

import numpy as np
import pytest

from conftest import bits_equal, load_indexed, random_scene, same_f32

F32 = np.float32
Z_FAR = 1000.0
LARGE_SHIFT = np.array([10007.25, -9871.5, 11003.125])      # where the "large_offset" views expect the model
LIGHT = [0.3, -0.2, 1.0]
SIZES = [(256, 256), (200, 333)]


def VW():
    from cython3dmodelrenderer_b200 import views
    return views


def O():
    from oracle import oracle
    return oracle


# ---------------------------------------------------------------------------------------------------- view families
def _rotation(rng):
    """A uniformly distributed rotation: the matrix of a normalised Gaussian quaternion (float64)."""
    w, x, y, z = (lambda q: q / np.linalg.norm(q))(rng.standard_normal(4))
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])


def _look_at(eye, target, up):
    """Rows (right, up, forward) of a camera at `eye` that looks at `target` along its +z (det +1)."""
    f = (target - eye) / np.linalg.norm(target - eye)
    r = np.cross(up, f)
    r /= np.linalg.norm(r)
    return np.stack([r, np.cross(f, r), f])


def _frame(v, fov):
    """(centre, radius, distance) of a model: the median corner, the 75th percentile of the distance to it (the edge-case
    families have far outliers), and the camera distance at which that radius fills 70 % of the half-frame."""
    pts = np.asarray(v, np.float64).reshape(-1, 3)
    c = np.median(pts, axis=0)
    r = max(float(np.percentile(np.linalg.norm(pts - c, axis=1), 75)), 1e-3)
    return c, r, r / (0.7 * np.tan(np.radians(fov) / 2))


def view_families(v, fov, seed=0):
    """name -> [V,16] float32 views of each family, for a model with corners `v` [T,3,3] seen with `fov`.  The
    "large_offset" views expect the model moved by LARGE_SHIFT (large_offset_vertices)."""
    VM = VW().view_matrix
    rng = np.random.default_rng(seed)
    c, r, D = _frame(v, fov)

    def off(s):          # a vector off every axis
        return rng.uniform(0.05, 0.15, 3) * rng.choice([-1.0, 1.0], 3) * s

    def place():         # q: the model in front of the camera at distance D, off the z axis
        return np.array([0.0, 0.0, D]) + off(0.4 * r) * [1, 1, 0]

    fam = {"rotation": [VM(_rotation(rng), c + off(r), place()) for _ in range(6)]}

    looks = []
    dirs = [rng.standard_normal(3) for _ in range(3)] + [np.array([1e-3, 1.0, 2e-3]), np.array([-3e-4, -1.0, 1e-4])]
    for d in dirs:          # random eyes, and two near the poles, where the (slightly rolled) up vector is nearly the view axis
        eye = c + D * d / np.linalg.norm(d)
        looks.append(VM(_look_at(eye, c, np.array([0.15, 1.0, -0.1])), eye, off(0.3 * r)))
    d = rng.standard_normal(3)
    d /= np.linalg.norm(d)
    looks.append(VM(_look_at(c + D * d, c, -d + 1e-4 * rng.standard_normal(3)), c + D * d, off(0.3 * r)))
    fam["look_at"] = looks

    u = rng.standard_normal(3)
    u /= np.linalg.norm(u)
    mats = [np.diag([0.6, 1.7, 1.2]) @ _rotation(rng),                                  # anisotropic scale
            np.array([[1.0, 0.35, -0.2], [0.0, 1.0, 0.45], [0.1, 0.0, 1.0]]) @ _rotation(rng),   # shear
            np.diag([-1.0, 1.0, 1.0]) @ _rotation(rng),                                 # mirror: det < 0
            (np.eye(3) - 2 * np.outer(u, u)) @ _rotation(rng),                          # reflection in a general plane
            _rotation(rng) @ (np.eye(3) - (1 - 1e-6) * np.outer(u, u))]                 # nearly singular: u scaled by 1e-6
    fam["non_orthonormal"] = [VM(R, c + off(r), place()) for R in mats]

    # camera plane: q.z = -(z row without q) of the corner at the middle depth puts it exactly on z = 0, one ulp of q.z more
    # or less just in front of or just behind the camera; then, scaled in x and y to stay in view, across and beyond z_far
    R, p, q = _rotation(rng), c + off(r), place()
    with np.errstate(all="ignore"):
        s = np.sort(VW().transform_arrays_host(VM(R, p, (0, 0, 0)), v, v)[0][..., 2].ravel())
    s = s[s.size // 2]
    planes = [VM(R, p, (q[0], q[1], qz)) for qz in (-s, np.nextafter(-s, F32(np.inf)), np.nextafter(-s, F32(-np.inf)))]
    k = Z_FAR / D
    Rk = np.diag([k, k, 1.0]) @ R
    planes += [VM(Rk, p, (k * q[0], k * q[1], Z_FAR - float(s))), VM(Rk, p, (k * q[0], k * q[1], Z_FAR + 4 * r))]
    fam["camera_plane"] = planes

    # -0.0 and subnormal entries in place of the zeros of rotations about z and about x
    a, b = 0.7, -1.1
    m1 = VM([[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]], c + off(r), place())
    m1[[2, 5, 6, 7]] = (F32(-0.0), F32(1e-40), F32(-1e-45), F32(-0.0))
    m2 = VM([[1, 0, 0], [0, np.cos(b), -np.sin(b)], [0, np.sin(b), np.cos(b)]], c + off(r), place())
    m2[[1, 2, 3, 6, 12]] = (F32(-0.0), F32(2e-39), F32(-3e-42), F32(-0.0), F32(-0.0))
    fam["special"] = [m1, m2]

    nf = [VM(_rotation(rng), c + off(r), place()) for _ in range(3)]
    nf[0][4], nf[1][8], nf[2][12] = F32(np.nan), F32(np.inf), F32(-np.inf)
    fam["non_finite"] = nf

    # p around 1e4, next to the moved model: v - p cancels.  A camera near the model (q of model size), and q around 1e4
    # with R scaled to keep the model in view at depth 9e3 and 4e4
    cs = c + LARGE_SHIFT
    fam["large_offset"] = [VM(_rotation(rng), cs + off(r), place()), VM(_rotation(rng), cs + off(r), place()),
                           VM(9000.0 / D * _rotation(rng), cs + off(r), (1500.5, -1200.25, 9000.0)),
                           VM(40000.0 / D * _rotation(rng), cs + off(r), (-9000.5, 8000.25, 40000.0))]
    return {name: np.stack(m).astype(F32) for name, m in fam.items()}


def large_offset_vertices(v):
    return (np.asarray(v, np.float64) + LARGE_SHIFT).astype(F32)


def general_batch(fams):
    """Every family but large_offset in one batch, the non-finite views spread between the others: (views, labels)."""
    views, labels = [], []
    spread = list(fams["non_finite"])
    for name in ("rotation", "look_at", "non_orthonormal", "camera_plane", "special"):
        for m in fams[name]:
            views.append(m)
            labels.append(name)
        if spread and name != "special":
            views.append(spread.pop(0))
            labels.append("non_finite")
    assert not spread
    return np.stack(views), labels


def transform(view, v, n):
    with np.errstate(all="ignore"):
        return VW().transform_arrays_host(view, v, n)


# ---------------------------------------------------------------------------------------------------- mutants
def _swap(M, i, j):
    M = np.array(M, F32).ravel().copy()
    M[[i, j]] = M[[j, i]]
    return M


def _set(M, i, j):
    """M with entry i read where entry j belongs."""
    M = np.array(M, F32).ravel().copy()
    M[j] = M[i]
    return M


def _transposed(M):
    M = np.array(M, F32).ravel().copy()
    M[:9] = M[:9].reshape(3, 3).T.ravel()
    return M


def _reassociated(M, v, n, order):
    """The transform with each row summed as r0*d0 + (r1*d1 + r2*d2) ("right") or as (r0*d0 + r1*d1) + (r2*d2 + q) ("q")."""
    M = np.asarray(M, F32).ravel()
    v, n = np.asarray(v, F32), np.asarray(n, F32)
    d = [v[..., k] - M[9 + k] for k in range(3)]
    vo, no = np.empty_like(v), np.empty_like(n)
    with np.errstate(all="ignore"):
        for r in range(3):
            a, b, c = (M[3 * r + k] * d[k] for k in range(3))
            na, nb, nc = (M[3 * r + k] * n[..., k] for k in range(3))
            vo[..., r] = (a + (b + c)) + M[12 + r] if order == "right" else (a + b) + (c + M[12 + r])
            no[..., r] = na + (nb + nc) if order == "right" else (na + nb) + nc
    return vo, no


# name -> (view, v, n) -> (v', n'); each a mistake the kernel could make in view_point / view_normal
MUTANTS = {
    "transposed R": lambda M, v, n: transform(_transposed(M), v, n),
    "M[5] <-> M[7]": lambda M, v, n: transform(_swap(M, 5, 7), v, n),
    "M[1] <-> M[3]": lambda M, v, n: transform(_swap(M, 1, 3), v, n),
    "z row reads M[5] for M[7]": lambda M, v, n: transform(_set(M, 5, 7), v, n),
    "p <-> q": lambda M, v, n: transform(np.concatenate([M[:9], M[12:15], M[9:12], M[15:]]), v, n),
    "q x <-> y": lambda M, v, n: transform(_swap(M, 12, 13), v, n),
    "p x <-> y": lambda M, v, n: transform(_swap(M, 9, 10), v, n),
    "r0*d0 + (r1*d1 + r2*d2)": lambda M, v, n: _reassociated(M, v, n, "right"),
    "(r0*d0 + r1*d1) + (r2*d2 + q)": lambda M, v, n: _reassociated(M, v, n, "q"),
}
# the mutants orbit views cannot tell apart from the transform (except for the sign of a zero)
ORBIT_BLIND = ("M[5] <-> M[7]", "M[1] <-> M[3]", "z row reads M[5] for M[7]", "p <-> q", "q x <-> y", "p x <-> y",
               "r0*d0 + (r1*d1 + r2*d2)")


def kept(view, n):
    """The cull of setup_chunk: a triangle is kept unless the float sum of its view-space normals' z is >= 0 (NaN: kept)."""
    with np.errstate(all="ignore"):
        z = transform(view, n, n)[1][..., 2]
        return ~(((z[:, 0] + z[:, 1]) + z[:, 2]) >= 0)


def _round_f32(x):
    """The float32 nearest to the Fraction x (ties to even)."""
    c = F32(float(x))
    cands = [y for y in (np.nextafter(c, F32(-np.inf)), c, np.nextafter(c, F32(np.inf))) if np.isfinite(y)]
    return min(cands, key=lambda y: (abs(Fraction(float(y)) - x), int(np.asarray(y).view(np.uint32)) & 1))


def fma_contracted(M, pts):
    """view_point with both product-sums contracted into FMAs, fma(r2, d2, fma(r1, d1, r0*d0)) + q, rounded exactly
    (Fractions) at corners pts [N,3]: what nvcc emits without -fmad=false."""
    M = np.asarray(M, F32).ravel()
    out = np.empty(pts.shape, F32)
    F = lambda x: Fraction(float(x))     # noqa: E731
    for i, p in enumerate(np.asarray(pts, F32)):
        d = [p[k] - M[9 + k] for k in range(3)]
        for r in range(3):
            s = M[3 * r] * d[0]
            s = _round_f32(F(M[3 * r + 1]) * F(d[1]) + F(s))
            s = _round_f32(F(M[3 * r + 2]) * F(d[2]) + F(s))
            out[i, r] = s + M[12 + r]
    return out


# ---------------------------------------------------------------------------------------------------- CPU tests
def _cpu_cases():
    """(label, corners, normals, views) of the T-Rex and a random scene: every family, large_offset on the moved model."""
    out = []
    for name, m, fov in (("trex", load_indexed("trex"), 45.0), ("scene3", random_scene(3, T=400), 90.0)):
        v, n = m._vertices_by_triangles, m._normals_by_triangles
        fams = view_families(v, fov)
        for fam, views in fams.items():
            out.append((f"{name}/{fam}", large_offset_vertices(v) if fam == "large_offset" else v, n, views))
    return out


def test_families_are_what_they_claim():
    fams = view_families(load_indexed("trex")._vertices_by_triangles, 45.0)
    for name in ("rotation", "look_at", "non_orthonormal", "camera_plane", "large_offset"):
        R, p, q = fams[name][:, :9], fams[name][:, 9:12], fams[name][:, 12:15]
        assert (R != 0).all() and (p[:, :2] != 0).all() and (q[:, :2] != 0).all(), name
    for name in ("rotation", "look_at"):
        R = fams[name][:, :9].reshape(-1, 3, 3).astype(np.float64)
        assert np.allclose(R @ R.transpose(0, 2, 1), np.eye(3), atol=1e-6) and np.allclose(np.linalg.det(R), 1, atol=1e-6)
    R = fams["non_orthonormal"][:, :9].reshape(-1, 3, 3).astype(np.float64)
    det = np.linalg.det(R)
    assert (det[2:4] < 0).all() and abs(det[4]) < 1e-5 and not np.allclose(R[0] @ R[0].T, np.eye(3), atol=0.1)
    assert (np.abs(fams["large_offset"][:, 9:12]) > 1000).all() and (np.abs(fams["large_offset"][2:, 12:15]) > 1000).all()
    sp = fams["special"][:, :15]
    assert (np.signbit(sp) & (sp == 0)).sum() >= 4 and ((sp != 0) & (np.abs(sp) < np.finfo(F32).tiny)).sum() >= 4
    nf = fams["non_finite"]
    assert np.isnan(nf[0, 4]) and nf[1, 8] == np.inf and nf[2, 12] == -np.inf
    # the camera-plane views put corners exactly on z = 0, one ulp in front and behind, and beyond z_far
    m = load_indexed("trex")
    z = [transform(M, m._vertices_by_triangles, m._normals_by_triangles)[0][..., 2] for M in fams["camera_plane"]]
    tiny = np.finfo(F32).eps
    assert (z[0] == 0).any() and (z[0] < 0).any() and (z[0] > 0).any()
    assert ((z[1] > 0) & (z[1] < tiny)).any() and ((z[2] < 0) & (z[2] > -tiny)).any()
    assert (z[3] > Z_FAR).any() and (z[3] < Z_FAR).any() and (z[4] > Z_FAR).mean() > 0.9


def test_restatement_is_the_transform_within_float32_rounding():
    """transform_arrays_host against R (v - p) + q and R n in float64 (products of two floats are exact there): a component
    of v' is d_k = v_k - p_k rounded, three products and three sums -- each term rounded at most five times -- so it is
    within gamma_5 * (sum |r_k (v_k - p_k)| + |q|) of the exact value, n' within gamma_3 * sum |r_k n_k|, plus the
    absolute error of subnormal results.  Non-finite values must be non-finite alike (same NaN / +-inf)."""
    u = 2.0 ** -24
    gamma = lambda k: k * u / (1 - k * u)          # noqa: E731
    eta = 8 * 2.0 ** -149
    for label, v, n, views in _cpu_cases():
        v64, n64 = v.astype(np.float64), n.astype(np.float64)
        for i, M in enumerate(views):
            R = M[:9].astype(np.float64).reshape(3, 3)
            p, q = M[9:12].astype(np.float64), M[12:15].astype(np.float64)
            got_v, got_n = transform(M, v, n)
            with np.errstate(all="ignore"):
                d = v64 - p
                exact_v = d @ R.T + q
                bound_v = gamma(5) * (np.abs(d) @ np.abs(R).T + np.abs(q)) + eta
                exact_n = n64 @ R.T
                bound_n = gamma(3) * (np.abs(n64) @ np.abs(R).T) + eta
            for what, got, exact, bound in (("v", got_v, exact_v, bound_v), ("n", got_n, exact_n, bound_n)):
                fin = np.isfinite(exact)
                assert np.array_equal(np.isnan(got), np.isnan(exact)), f"{label} view {i} {what}: NaN pattern"
                assert np.array_equal(got[np.isinf(exact)], exact[np.isinf(exact)].astype(F32)), f"{label} view {i} {what}"
                err = np.abs(got[fin].astype(np.float64) - exact[fin])
                assert (err <= bound[fin]).all(), f"{label} view {i} {what}: error {err.max()!r} over the bound"
            if "non_finite" not in label:
                assert np.isfinite(got_v).all() and np.isfinite(got_n).all(), f"{label} view {i}"


def _differs(a, b):
    a, b = np.ascontiguousarray(a, F32), np.ascontiguousarray(b, F32)
    return int((a.view(np.uint32) != b.view(np.uint32)).sum())


def _fma_sample_differs(views, v, rng, count):
    pts = np.asarray(v, F32).reshape(-1, 3)
    diff = 0
    for M in views:
        if not np.isfinite(M).all():
            continue
        s = pts[rng.choice(len(pts), count, replace=False)]
        want = transform(M, s[:, None, :], s[:, None, :])[0][:, 0]
        diff += _differs(fma_contracted(M, s), want)
    return diff


def test_general_views_tell_every_mutant_apart():
    """Each mistake changes at least one output word of the families (the random rotations alone too); the cull's z row
    read wrong changes at least one cull decision; FMA contraction changes a word of a sample of corners."""
    cases = _cpu_cases()
    for name, mutant in MUTANTS.items():
        total, rotation = 0, 0
        for label, v, n, views in cases:
            for M in views:
                want_v, want_n = transform(M, v, n)
                got_v, got_n = mutant(M, v, n)
                d = _differs(got_v, want_v) + _differs(got_n, want_n)
                total += d
                rotation += d if label.endswith("/rotation") else 0
        assert total > 0 and rotation > 0, f"the view families cannot tell '{name}' apart"
    # only the cull reads the z row wrong (full-frame or band filler): some triangle is culled differently
    flips = sum(int((kept(_set(M, 5, 7), n) != kept(M, n)).sum()) for _, _, n, views in cases for M in views)
    assert flips > 0
    # only the perspective texture's depth (CRB_TEX_PERSPECTIVE, w = 1 / z) reads the z row wrong
    with np.errstate(all="ignore"):
        dw = sum(_differs(F32(1) / transform(_set(M, 5, 7), v, n)[0][..., 2], F32(1) / transform(M, v, n)[0][..., 2])
                 for _, v, n, views in cases for M in views)
    assert dw > 0
    rng = np.random.default_rng(5)
    assert sum(_fma_sample_differs(views, v, rng, 24) for _, v, _, views in cases) > 0


def test_orbit_views_cannot_tell_these_mistakes_apart():
    """The views the rest of the suite renders -- orbit_views(128) about the y axis, q = p = (0, 0, 1) -- give the values of
    the right transform under the index swaps, the p / q exchange, the x / y swaps and r0*d0 + (r1*d1 + r2*d2), and keep the
    same triangles in the cull: only the sign of a zero may change.  They do catch a transposed R, FMA contraction, and q
    added to the z row's last product first (three nonzero terms there)."""
    m = load_indexed("trex")
    v, n = m._vertices_by_triangles, m._normals_by_triangles
    orbit = VW().orbit_views(128)
    for name in ORBIT_BLIND:
        for k, M in enumerate(orbit):
            want_v, want_n = transform(M, v, n)
            got_v, got_n = MUTANTS[name](M, v, n)
            assert np.array_equal(got_v, want_v) and np.array_equal(got_n, want_n), f"orbit view {k} tells '{name}' apart"
    assert all(np.array_equal(kept(_set(M, 5, 7), n), kept(M, n)) for M in orbit)
    for name in ("transposed R", "(r0*d0 + r1*d1) + (r2*d2 + q)"):
        assert sum(_differs(MUTANTS[name](M, v, n)[0], transform(M, v, n)[0]) for M in orbit) > 0, name
    assert _fma_sample_differs(orbit, v, np.random.default_rng(6), 8) > 0


# ---------------------------------------------------------------------------------------------------- GPU tests
def _model(name, h, w):
    """(TriModel, fov): the T-Rex, a random scene (seed 10: partly behind the camera, 14: snapped to a grid), or the
    edge-case families of test_gpu_edges built for h x w."""
    if name == "trex":
        return load_indexed("trex"), 45.0
    if name.startswith("scene"):
        return random_scene(int(name[5:]), T=400), 90.0
    import test_gpu_edges as E
    return E.concat(*(E.family(k, h, w) for k in "ACDEFG")), E.FOV


_BATCHES = {}


def batches(name, h, w):
    """[(batch, TriModel, views [V,16], labels)]: the general batch, and large_offset on the moved model."""
    key = (name, h, w)
    if key not in _BATCHES:
        from conftest import TriModel
        m, fov = _model(name, h, w)
        fams = view_families(m._vertices_by_triangles, fov)
        views, labels = general_batch(fams)
        moved = TriModel(large_offset_vertices(m._vertices_by_triangles), m._colors_by_triangles, m._normals_by_triangles)
        _BATCHES[key] = (fov, [("general", m, views, labels),
                               ("large_offset", moved, fams["large_offset"], ["large_offset"] * len(fams["large_offset"]))])
    return _BATCHES[key]


_ORACLE = {}


def oracle_views(key, m, views, h, w, fov, light=None):
    """Per view: the oracle's (z, colour, normals) of transform_arrays_host's arrays, colour lit by `light` if given."""
    k = key + (h, w)
    if k not in _ORACLE:
        frames = []
        for M in views:
            vk, nk = transform(M, m._vertices_by_triangles, m._normals_by_triangles)
            o = O().OracleFiller(h, w, fov=fov)
            o.render_arrays(vk, m._colors_by_triangles, nk)
            frames.append(tuple(a.copy() for a in (o.get_z_buffer(), o.get_color_buffer(), o.get_normals_buffer())))
        _ORACLE[k] = frames
    if light is None:
        return _ORACLE[k]
    return [(z, O().guro(c.copy(), nrm, light), nrm) for z, c, nrm in _ORACLE[k]]


def _u8(colour):
    with np.errstate(invalid="ignore"):
        return colour[::-1].astype("uint8")


def _device(m):
    import torch
    return tuple(torch.from_numpy(np.ascontiguousarray(a)).cuda()
                 for a in (m._vertices_by_triangles, m._colors_by_triangles, m._normals_by_triangles))


def _check_out(out, want, labels, what, names=("z", "color", "normals"), rows=slice(None)):
    from test_gpu_edges import _assert_same
    for k, frame in enumerate(want):
        got = tuple(out[name][k].cpu().numpy() for name in names)
        ref = tuple(frame[("z", "color", "normals").index(name)][rows] for name in names)
        for name, g, r in zip(names, got, ref):
            _assert_same((g,), (r,), f"{what} view {k} ({labels[k]}) {name}")
        if "color_u8" in out:
            assert np.array_equal(out["color_u8"][k].cpu().numpy(), _u8(frame[1][rows])), f"{what} uint8 view {k} ({labels[k]})"


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["trex", "scene10", "edges"])
def test_transform_view_equals_restatement(name):
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller
    h, w = SIZES[0]
    fov, bs = batches(name, h, w)
    f = AdvancedPixelBufferFiller(h, w, fov=fov)
    for batch, m, views, labels in bs:
        dv, _, dn = _device(m)
        for k, M in enumerate(views):
            want_v, want_n = transform(M, m._vertices_by_triangles, m._normals_by_triangles)
            gv, gn = (a.cpu().numpy() for a in f.transform_view(dv, dn, M))
            # NaN bits are the instruction set's (x86 0xFFC00000 / payload, GPU 0x7FFFFFFF): only the non-finite views make NaN
            same = same_f32 if labels[k] == "non_finite" else bits_equal
            assert same(gv, want_v) and same(gn, want_n), f"{name} {batch} view {k} ({labels[k]})"


@pytest.mark.gpu
@pytest.mark.parametrize("size", SIZES, ids=lambda s: f"{s[0]}x{s[1]}")
@pytest.mark.parametrize("name", ["trex", "scene3", "scene10", "scene14", "edges"])
def test_render_views_general_views(name, size):
    """z, colour, normals and the fused uint8 image of every view; then colour-only with the fused Guro pass under a
    general light direction."""
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller
    h, w = size
    fov, bs = batches(name, h, w)
    covered = 0
    for batch, m, views, labels in bs:
        dv, dc, dn = _device(m)
        f = AdvancedPixelBufferFiller(h, w, fov=fov)
        out = f.render_views(dv, dc, dn, views, chunk=3, color_u8_out=True)
        want = oracle_views((name, batch), m, views, h, w, fov)
        _check_out(out, want, labels, f"{name} {batch} {h}x{w}")
        covered += sum(int((z < F32(1e5)).sum()) for z, _, _ in want)
        lit = f.render_views(dv, dc, dn, views, want=("color",), guro_light=LIGHT, color_u8_out=True, chunk=5)
        assert set(lit) == {"color", "color_u8"}
        _check_out(lit, oracle_views((name, batch), m, views, h, w, fov, LIGHT), labels, f"{name} {batch} lit {h}x{w}",
                   names=("color",))
    assert covered > 20 * h * w // 100


@pytest.mark.gpu
def test_render_views_trex_1024():
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller
    h = w = 1024
    fov, bs = batches("trex", 256, 256)
    _, m, views, labels = bs[0]
    pick = list(range(0, len(views), 3))
    views, labels = views[pick], [labels[i] for i in pick]
    dv, dc, dn = _device(m)
    out = AdvancedPixelBufferFiller(h, w, fov=fov).render_views(dv, dc, dn, views, chunk=4, color_u8_out=True,
                                                                guro_light=LIGHT)
    want = oracle_views(("trex", "general", tuple(pick)), m, views, h, w, fov, LIGHT)
    _check_out(out, want, labels, "trex 1024")
    assert sum(int((z < F32(1e5)).sum()) for z, _, _ in want) > len(views) * 20000


@pytest.mark.gpu
def test_batching_of_general_views():
    """chunk in {1, 3, V, > V} (V = 11), the launch pipeline off and on, defer_join then join(), and `want` subsets."""
    import torch
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller, _lib
    h, w = SIZES[1]
    fov, bs = batches("trex", h, w)
    _, m, views, labels = bs[0]
    views, labels = views[:11], labels[:11]
    assert "non_finite" in labels
    want = oracle_views(("trex", "general", "first11"), m, views, h, w, fov)
    dv, dc, dn = _device(m)
    for pipe in (0, 1):
        for chunk in (1, 3, 11, 16):
            f = AdvancedPixelBufferFiller(h, w, fov=fov)
            f.set_option(_lib.CRB_OPT_CHUNK_PIPELINE, pipe)
            _check_out(f.render_views(dv, dc, dn, views, chunk=chunk, color_u8_out=True), want, labels,
                       f"pipeline {pipe} chunk {chunk}")
    g = AdvancedPixelBufferFiller(h, w, fov=fov)
    g.render_views(dv, dc, dn, views, chunk=1)      # sizes the pair list for every view: calls without check_status never retry
    dviews = torch.from_numpy(views).cuda()
    first = g.render_views(dv, dc, dn, dviews[:5], chunk=1, check_status=False, defer_join=True, color_u8_out=True)
    second = g.render_views(dv, dc, dn, dviews[5:], chunk=1, check_status=False, defer_join=True, color_u8_out=True)
    g.join()
    _check_out(first, want[:5], labels[:5], "deferred, first batch")
    _check_out(second, want[5:], labels[5:], "deferred, second batch")
    for sub in (("z",), ("normals",), ("color", "normals")):
        out = g.render_views(dv, dc, dn, views, want=sub, chunk=4)
        assert set(out) == set(sub)
        _check_out(out, want, labels, f"want={sub}", names=sub)


@pytest.mark.gpu
def test_hundreds_of_views_small_frames():
    """300 random rotations and look-at cameras at 32x48: ten launches of 32 views and 43 of 7, the slab of every view
    at its own offset."""
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller
    h, w = 32, 48
    m, fov = _model("trex", h, w)
    views = []
    for seed in range(30):
        fams = view_families(m._vertices_by_triangles, fov, seed=100 + seed)
        views += list(fams["rotation"]) + list(fams["look_at"][:4])
    views = np.stack(views[:300])
    assert len(views) == 300
    labels = ["rotation/look_at"] * len(views)
    want = oracle_views(("trex", "hundreds"), m, views, h, w, fov)
    dv, dc, dn = _device(m)
    f = AdvancedPixelBufferFiller(h, w, fov=fov)
    for chunk in (32, 7):
        _check_out(f.render_views(dv, dc, dn, views, chunk=chunk, color_u8_out=True), want, labels, f"chunk {chunk}")


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [1, 2, 3])
def test_rasterizer_shapes_general_views(shape):
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller, _lib
    h, w = SIZES[0]
    for name in ("trex", "edges"):
        fov, bs = batches(name, h, w)
        for batch, m, views, labels in bs:
            f = AdvancedPixelBufferFiller(h, w, fov=fov)
            f.set_option(_lib.CRB_OPT_RASTER_SHAPE, shape)
            out = f.render_views(*_device(m), views, chunk=4, color_u8_out=True)
            _check_out(out, oracle_views((name, batch), m, views, h, w, fov), labels, f"shape {shape} {name} {batch}")


@pytest.mark.gpu
@pytest.mark.parametrize("size", SIZES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_band_fillers_general_views(size):
    """render_views on band fillers (the banded cull): bands not aligned to tiles, one-row bands, the first and last rows;
    each band equals the oracle's rows."""
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller
    h, w = size
    bands = [(0, 37), (37, 133), (133, h), (5, 6), (h - 1, h), (h // 2 - 9, h // 2 + 23)]
    for name in ("trex", "scene10"):
        fov, bs = batches(name, h, w)
        for batch, m, views, labels in bs:
            want = oracle_views((name, batch), m, views, h, w, fov)
            dv, dc, dn = _device(m)
            for r0, r1 in bands:
                f = AdvancedPixelBufferFiller(h, w, fov=fov, band=(r0, r1))
                out = f.render_views(dv, dc, dn, views, chunk=3)
                _check_out(out, want, labels, f"{name} {batch} band {r0}:{r1} {h}x{w}", rows=slice(r0, r1))


@pytest.mark.gpu
@pytest.mark.parametrize("size", SIZES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_row_exchange_general_views(size):
    """crb_set_u8_exchange with two row bands whose bases are local device buffers: per view, the two bands concatenated
    are the local color_u8_out image, and the oracle's."""
    import torch
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller
    h, w = size
    hb = h // 2
    fov, bs = batches("trex", h, w)
    _, m, views, labels = bs[0]
    V = len(views)
    dv, dc, dn = _device(m)
    f = AdvancedPixelBufferFiller(h, w, fov=fov)
    local = f.render_views(dv, dc, dn, views, want=(), chunk=4, color_u8_out=True)["color_u8"]
    recv = [torch.full((V, hb, w, 3), 7, dtype=torch.uint8, device="cuda") for _ in range(2)]
    f.render_views(dv, dc, dn, views, want=(), chunk=4, u8_exchange=(hb, [b.data_ptr() for b in recv]))
    torch.cuda.synchronize()
    got = torch.cat(recv, dim=1)
    want = oracle_views(("trex", "general"), m, views, h, w, fov)
    for k in range(V):
        assert torch.equal(got[k], local[k]), f"view {k} ({labels[k]}): exchanged bands differ from the local image"
        assert np.array_equal(got[k].cpu().numpy(), _u8(want[k][1])), f"view {k} ({labels[k]}): differs from the oracle"


TEX_MODES = [(flt, persp) for flt in ("nearest", "bilinear", "trilinear") for persp in (False, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", TEX_MODES, ids=lambda m: m[0] + ("_persp" if m[1] else ""))
def test_textured_general_views(mode):
    """Per-pixel texturing under every family, fused Guro and uint8 included, against texture_modes_oracle (nearest,
    bilinear) and texture_mip_oracle (trilinear) on the transformed arrays.  Perspective-correct coordinates divide by
    the transformed z (the z row evaluated a third time in setup_chunk)."""
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller, synthetic
    from test_texture_oracle import random_texture
    flt, persp = mode
    if flt == "trilinear":
        from oracle.texture_mip_oracle import TexturedOracleFiller
    else:
        from oracle.texture_modes_oracle import TexturedOracleFiller
    h, w = SIZES[0]
    tex = random_texture(11, 709, 709)
    for batch, m, views, labels in batches("trex", h, w)[1]:
        fov = 45.0
        uv = synthetic.spherical_uvs(load_indexed("trex")._vertices_by_triangles)
        dv, _, dn = _device(m)
        f = AdvancedPixelBufferFiller(h, w, fov=fov, texture_filter=flt, perspective_correct=persp)
        out = f.render_views(dv, uv, dn, views, chunk=3, color_u8_out=True, guro_light=LIGHT, texture=tex)
        want = []
        for M in views:
            vk, nk = transform(M, m._vertices_by_triangles, m._normals_by_triangles)
            o = TexturedOracleFiller(h, w, fov=fov)
            with np.errstate(all="ignore"):
                o.render_arrays(vk, uv, nk, texture=tex, perspective=persp, filter=flt)
            z, c, nrm = (a.copy() for a in (o.get_z_buffer(), o.get_color_buffer(), o.get_normals_buffer()))
            O().guro(c, nrm, LIGHT)
            want.append((z, c, nrm))
        _check_out(out, want, labels, f"{flt} persp={persp} {batch}")
