"""The tile rasterizer's shortcuts at their admission thresholds, against the oracle, bit for bit.

k_setup (cython3dmodelrenderer_b200/csrc/crender_b200.cu, setup_chunk) admits each triangle to a few fast paths, each
correct because of an error analysis in a comment there:
  FL_SPAN  closed-form conservative row span (span_bound): all three denominators in [1e-30, 1e30], coordinates finite
           and <= 2^18 (SPAN_COORD_MAX); everything else tests each pixel of a rectangle row against thresholds
  FL_REJ   division-free rejection of barycentric k: |l_k3| in [L3_MIN, L3_MAX], with FL_NEG flipping its sign
  FL_FDIV  div_rn_by instead of div.rn: denominators in [2^-40, 2^40], numerators >= 2^-40 (fdiv_ok_lo)
and the band pre-pass (k_band_chunks) lists a 256-triangle chunk from rcp.approx screen y in a widened band.
Random scenes put almost every triangle on the same side of each of these tests.  The scene families below are built
in camera space from target screen coordinates so that they land on both sides of them; `classify` restates k_setup's
decisions on the oracle's projection, and test_edge_families_reach_their_regimes checks that every family really
reaches the regime it is aimed at.  Then the GPU renders every family on every path and switch, fresh and composited,
in batched views and in row bands, and must give the oracle's bits.

The uint8 stage (to_u8) is checked on colours outside [0, 255], where NumPy's `astype('uint8')` on x86-64 yields the
low byte of cvttss2si's result: INT_MIN (low byte 0) for NaN and everything outside int range.
"""
import os
import platform

import numpy as np
import pytest

from conftest import ROOT, TriModel, bits_equal, random_scene

F32 = np.float32
SIZES = [(256, 256), (200, 333)]
FOV = 90.0
SPAN_COORD_MAX = F32(2.0 ** 18)
L3_MIN, L3_MAX = F32(1e-30), F32(1e30)
FDIV_LO, FDIV_HI = F32(2.0 ** -40), F32(2.0 ** 40)
Z_INIT = F32(1e6)


def O():
    from oracle import oracle
    return oracle


# ---------------------------------------------------------------------------------------------------- classifier
def numerators(s, px, py):
    """The three barycentric numerators at pixel (px, py) of screen-space triangles s [T,3,3], in shade_fragment's
    operation order (crender_b200.cu, shade_fragment; mu:34)."""
    x0, y0, x1, y1, x2, y2 = (s[:, k // 2, k % 2] for k in range(6))
    px, py = F32(px), F32(py)
    n1 = (x1 - x2) * (py - y2) - (y1 - y2) * (px - x2)
    n2 = (x2 - x0) * (py - y0) - (y2 - y0) * (px - x0)
    n3 = (x0 - x1) * (py - y1) - (y0 - y1) * (px - x1)
    return n1, n2, n3


def classify(h, w, fov, v, n):
    """k_setup's per-triangle decisions (crender_b200.cu, setup_chunk) on the oracle's projection (pinned bit-equal to the
    reference), restated in float32 NumPy: elementwise float32 operations round once and never contract, as -fmad=false.
    Returns a dict of per-triangle arrays."""
    o = O()
    s = o.project(h, w, o.projection_matrix(h, w, fov), v)
    with np.errstate(all="ignore"):
        rects = np.array([o.pixel_rect(t, h, w) for t in s], dtype=np.int64).reshape(-1, 4)
        # pyx:202-211: not culled (float sum of the normals' z, NaN is not culled) and a non-empty rectangle
        nz = np.asarray(n, dtype=F32)[:, :, 2]
        culled = ((nz[:, 0] + nz[:, 1]) + nz[:, 2]) >= 0
        drawn = (rects[:, 0] < rects[:, 1]) & (rects[:, 2] < rects[:, 3]) & ~culled
        x, y = s[..., 0], s[..., 1]
        # denominators of mu:12-21 in the kernel's order (setup_chunk, "l03 = (x[1] - x[2]) * ...")
        l03 = (x[:, 1] - x[:, 2]) * (y[:, 0] - y[:, 2]) - (y[:, 1] - y[:, 2]) * (x[:, 0] - x[:, 2])
        l13 = (x[:, 2] - x[:, 0]) * (y[:, 1] - y[:, 0]) - (y[:, 2] - y[:, 0]) * (x[:, 1] - x[:, 0])
        l23 = (x[:, 0] - x[:, 1]) * (y[:, 2] - y[:, 1]) - (y[:, 0] - y[:, 1]) * (x[:, 2] - x[:, 1])
        l3 = np.stack([l03, l13, l23], axis=1)
        a = np.abs(l3)
        rej = (a >= L3_MIN) & (a <= L3_MAX)                          # FL_REJ << k
        neg = rej & (l3 < 0)                                         # FL_NEG << k
        cmax = np.fmax.reduce(np.fmax(np.abs(x), np.abs(y)), axis=1, initial=F32(0))   # fmaxf: NaN never wins
        finite_xy = np.all((x - x == 0) & (y - y == 0), axis=1)
        span = rej.all(axis=1) & finite_xy & (cmax <= SPAN_COORD_MAX)    # FL_SPAN
        fdiv = (np.fmin.reduce(a, axis=1) >= FDIV_LO) & (np.fmax.reduce(a, axis=1) <= FDIV_HI)   # FL_FDIV (fminf / fmaxf)
    return dict(s=s, rect=rects, drawn=drawn, l3=l3, rej=rej, neg=neg, cmax=cmax, finite_xy=finite_xy, span=span, fdiv=fdiv)


# ---------------------------------------------------------------------------------------------------- scene families
def _camera(h, w, fov, xs, ys, z):
    """Camera-space x, y whose projection lands near screen (xs, ys) at camera depth z (float64 inverse of pyx:116-130)."""
    P = O().projection_matrix(h, w, fov).astype(np.float64)
    xs, ys, z = (np.asarray(a, dtype=np.float64) for a in (xs, ys, z))
    return (xs / (w / 2.0) - 1.0) * z / P[0, 0], (ys / (h / 2.0) - 1.0) * z / P[1, 1]


def _model(v, rng, nz=-1.0):
    v = np.ascontiguousarray(v, dtype=F32)
    n = np.zeros_like(v)
    n[..., 2] = F32(nz)
    c = (rng.random(v.shape) * 255).astype(F32)
    return TriModel(v, c, n)


def _tris(h, w, xs, ys, z):
    """[T,3,3] camera-space triangles from screen targets xs, ys [T,3] and camera depths z [T,3]."""
    x, y = _camera(h, w, FOV, xs, ys, z)
    return np.stack([x, y, np.asarray(z, dtype=np.float64)], axis=-1).astype(F32)


def _slivers(h, w, rng, T, rmin, rmax):
    """Long thin triangles: a 0.5-4 px wide base on screen, an apex at distance rmin..rmax px, shallow, steep and random."""
    p = np.stack([rng.uniform(0, w, T), rng.uniform(0, h, T)], axis=1)
    th = rng.uniform(0, 2 * np.pi, T)
    th[0::4] = rng.choice([0.0, np.pi], T)[0::4] + rng.uniform(-1e-3, 1e-3, len(th[0::4]))            # shallow
    th[1::4] = rng.choice([0.5, 1.5], T)[1::4] * np.pi + rng.uniform(-1e-3, 1e-3, len(th[1::4]))      # steep
    R = np.exp(rng.uniform(np.log(rmin), np.log(rmax), T))
    d = np.stack([np.cos(th), np.sin(th)], axis=1)
    nrm = np.stack([-d[:, 1], d[:, 0]], axis=1) * rng.uniform(0.25, 2.0, (T, 1))
    apex = p + R[:, None] * d
    pts = np.stack([p - nrm, p + nrm, apex], axis=1)
    # keep the apex coordinate itself inside [rmin, rmax] (cmax is a max over |x|, |y|)
    z = np.repeat(rng.uniform(1.0, 4.0, (T, 1)), 3, axis=1)
    return _tris(h, w, pts[..., 0], pts[..., 1], z)


def family_A(h, w):
    """Far slivers inside the span limit: apex 2^10..2^18 px away, most beyond 2^17."""
    rng = np.random.default_rng(1)
    v = np.concatenate([_slivers(h, w, rng, 40, 2.0 ** 10, 2.0 ** 17), _slivers(h, w, rng, 60, 2.0 ** 17 + 2 * w, 2.0 ** 18 - 2 * w)])
    return _model(v, rng)


def family_B(h, w):
    """The same just outside the span limit: apex 2^18..2^22 px away."""
    rng = np.random.default_rng(2)
    return _model(_slivers(h, w, rng, 60, 2.0 ** 18 + 2 * w, 2.0 ** 22 - 2 * w), rng)


def family_C(h, w):
    """Huge denominators: one or two vertices near the camera plane (z = +-1e-6 .. +-1e-12), or far enough out for the
    projection to overflow, next to an ordinary on-screen base."""
    rng = np.random.default_rng(3)
    T = 60
    xs = rng.uniform(0.2 * w, 0.8 * w, (T, 3))
    ys = rng.uniform(0.2 * h, 0.8 * h, (T, 3))
    z = np.repeat(rng.uniform(1.0, 3.0, (T, 1)), 3, axis=1)
    v = _tris(h, w, xs, ys, z)
    for t in range(T):
        # the far vertex goes to negative screen x and y: beyond int range on the positive side, (int)ceil gives INT_MIN
        # and the pixel rectangle is empty (pyx:165-175)
        sg = rng.choice([-1.0, 1.0])
        zt = F32(sg * 10.0 ** rng.uniform(-12, -6))
        v[t, 2, 2] = zt
        v[t, 2, :2] = (-sg * rng.uniform(0.01, 0.3, 2)).astype(F32)
        if t % 3 == 1:                                    # two near-plane vertices far apart: denominators beyond 1e30
            v[t, 1, 2] = F32(-zt)
            v[t, 1, :2] = (sg * rng.uniform(1, 50, 2)).astype(F32)
            v[t, 2, :2] = (-sg * rng.uniform(1e2, 1e3, 2)).astype(F32)
        if t % 6 == 2:                                    # X / z overflows: infinite screen coordinate
            v[t, 2, 2] = F32(1e-38 * sg)
    return _model(v, rng)


def family_D(h, w):
    """Tiny denominators: triangles a few quanta of the screen lattice wide (2^-24 * w/2 near an edge of the screen,
    so every difference and product is exact) around the corner pixels, some collinear (zero denominators), some with a
    vertex exactly on the pixel centre (zero numerators).  On that lattice a denominator or numerator is a multiple of
    (2^-24 * w/2)^2 = 2^-34 at w = 256, so the ones below 2^-40 (FL_FDIV off, fdiv_ok_lo false) are exact zeros."""
    rng = np.random.default_rng(4)
    tris = []
    for cx, cy in ((0, 0), (w - 1, 0), (0, h - 1), (w - 1, h - 1), (1, 1)):
        for k in range(24):
            q = rng.integers(-3, 4, (3, 2)).astype(np.float64)
            if k % 4 == 0:
                q[0] = 0.0                                # a vertex on the pixel centre
            if k % 4 == 1:
                q[2] = 2 * q[1] - q[0]                    # collinear lattice points: all three denominators 0
            tris.append(np.stack([cx + q[:, 0] * 2.0 ** -24 * (w / 2.0), cy + q[:, 1] * 2.0 ** -24 * (h / 2.0)], axis=1))
    pts = np.asarray(tris)
    z = np.ones(pts.shape[:2])
    return _model(_tris(h, w, pts[..., 0], pts[..., 1], z), rng)


def family_E(h, w):
    """Pixel lattice: meshes with every vertex on a pixel centre (numerators exactly 0 and -0.0 on shared inclusive edges),
    a duplicate at the same depth (ties broken by index), and screen-covering triangles with vertices at +-2^17."""
    rng = np.random.default_rng(5)
    tris = []
    for (gx, gy, step, zc) in ((3, 5, 7, 1.0), (40, 60, 13, 2.0), (w // 2 - 20, h // 2 - 30, 5, 1.0)):
        for i in range(5):
            for j in range(5):
                a, b = (gx + i * step, gy + j * step), (gx + (i + 1) * step, gy + j * step)
                c, d = (gx + i * step, gy + (j + 1) * step), (gx + (i + 1) * step, gy + (j + 1) * step)
                tris += [((a, b, d), zc), ((a, d, c), zc)]
    tris += tris[:20]                                     # identical copies later in the list: they win the ties
    big = 2 ** 17
    for zc, pts in ((4.0, ((-big, 7), (big, 3), (5, big))), (0.5, ((9, -big), (-big, big), (big, big))),
                    (2.0, ((-big, -big), (big, -big), (11, 13)))):
        tris.append((pts, zc))
    xs = np.array([[p[0] for p in t] for t, _ in tris], dtype=np.float64)
    ys = np.array([[p[1] for p in t] for t, _ in tris], dtype=np.float64)
    z = np.array([[zc] * 3 for _, zc in tris])
    return _model(_tris(h, w, xs, ys, z), rng)


def _needles(h, w, rng, T, reach):
    p0 = np.stack([rng.integers(0, w, T), rng.integers(0, h, T)], axis=1).astype(np.float64)
    d = rng.integers(-reach, reach + 1, (T, 2)).astype(np.float64)
    d[np.all(d == 0, axis=1)] = (1.0, 3.0)
    k = rng.integers(2, 6, T)[:, None]
    pts = np.stack([p0, p0 + d, p0 + k * d], axis=1)
    pts[:, 2] += rng.integers(-4, 5, (T, 2)) * 2.0 ** -17
    z = np.repeat(rng.uniform(1.0, 3.0, (T, 1)), 3, axis=1)
    return _tris(h, w, pts[..., 0], pts[..., 1], z)


def family_F(h, w):
    """Needles: three nearly collinear points through pixel centres, one moved by a few lattice quanta, so that the three
    denominators (equal in exact arithmetic) round to different signs or to an exact zero.  Short ones, and long ones
    (far vertex thousands of pixels out) picked by `classify` for denominators of mixed sign: there the rounding noise in
    the numerators of covered pixels is far above the rejection guard band REJ_EPS, so a denominator normalised with the
    wrong sign rejects pixels it must not."""
    rng = np.random.default_rng(6)
    short = _needles(h, w, rng, 400, 40)
    cand = _needles(h, w, rng, 20000, 2000)
    cl = classify(h, w, FOV, cand, np.full_like(cand, -1.0))
    sg = np.sign(cl["l3"])
    keep = np.flatnonzero(cl["drawn"] & (sg.max(axis=1) > 0) & (sg.min(axis=1) < 0))[:100]
    return _model(np.concatenate([short, cand[keep]]), rng)


def _depth_search(h, w, z0, want):
    """Float camera depths next to z0 for a vertex at (0, 0, z): that vertex projects onto the pixel centre (w/2, h/2)
    with depth Z / z; returns (z, depth) pairs around `want`."""
    o = O()
    P = o.projection_matrix(h, w, FOV)
    zs = np.array([z0], dtype=F32)
    for _ in range(40):
        zs = np.unique(np.concatenate([zs, np.nextafter(zs, F32(np.inf)), np.nextafter(zs, F32(-np.inf))]))
    v = np.zeros((len(zs), 3, 3), F32)
    v[:, :, 2] = zs[:, None]
    dep = o.project(h, w, P, v)[:, 0, 2]
    return zs, dep


def family_G(h, w):
    """Depth extremes, each in its own part of the screen: triangles between the camera and z_near (negative depth),
    +-inf depth from a vertex at (0, 0, tiny z) -- it projects onto the centre pixel, finite --, depth 0 (camera z ==
    z_near) in overlapping copies, and vertices on the pixel centres (w/4, h/4), (w/4, 3h/8) and (3w/8, h/4) whose depth is
    just below, just above and (where a float camera z gives it) equal to the clear value 1e6."""
    rng = np.random.default_rng(7)
    U = lambda lo, hi, n, k: rng.uniform(lo * k, hi * k, (n, 3))
    tris = [_tris(h, w, U(0.55, 0.95, 24, w), U(0.05, 0.45, 24, h), rng.uniform(0.02, 0.09, (24, 3))),   # in front of z_near
            _tris(h, w, U(0.05, 0.4, 8, w), U(0.55, 0.95, 8, h), np.full((8, 3), 0.1))]                  # depth 0
    inf = _tris(h, w, U(0.55, 0.95, 8, w), U(0.55, 0.95, 8, h), np.full((8, 3), 2.0))
    inf[:, 0] = 0.0
    inf[:, 0, 2] = np.array([1e-40, -1e-40, 1e-45, -1e-45] * 2, dtype=F32)            # depth Z / z = -inf / +inf
    tris.append(inf)
    zs, dep = _depth_search(h, w, F32(-0.1 * 1000.0 / 999.9 / 1e6), Z_INIT)
    pick = [zs[dep < Z_INIT][np.argmax(dep[dep < Z_INIT])], zs[dep > Z_INIT][np.argmin(dep[dep > Z_INIT])]]
    pick += list(zs[dep == Z_INIT][:1])
    for zc, (fx, fy) in zip(pick, ((-0.5, -0.5), (-0.5, -0.25), (-0.25, -0.5))):
        # depth does not depend on x, y (P[0,2] = P[1,2] = 0); x = -z/2 gives x / z = -1/2 exactly: screen w/4
        t = np.full((2, 3, 3), zc, F32)
        t[:, :, 0] = F32(fx) * zc
        t[:, :, 1] = F32(fy) * zc
        t[0, 1, 0] -= F32(3e-10)   # z < 0: the other vertices land 0.4 px right of / below the pixel centre
        t[0, 2, 1] -= F32(3e-10)
        t[1, 1, 1] -= F32(3e-10)
        t[1, 2, 0] -= F32(3e-10)
        tris.append(t)
    m = _model(np.concatenate(tris), rng)
    m.clear_depth_found = bool((dep == Z_INIT).any())
    return m


H_ROWS = (37, 45, 61, 100)


def _y_near_row(h, w, r, z, above):
    """Camera y at depth z whose projected screen y is the lattice point next to row r, above it or below it."""
    o = O()
    P = o.projection_matrix(h, w, FOV)
    _, y0 = _camera(h, w, FOV, 0.0, float(r), float(z))
    ys = np.array([F32(y0)], F32)
    for _ in range(24):
        ys = np.unique(np.concatenate([ys, np.nextafter(ys, F32(np.inf)), np.nextafter(ys, F32(-np.inf))]))
    v = np.zeros((len(ys), 3, 3), F32)
    v[:, :, 1] = ys[:, None]
    v[:, :, 2] = F32(z)
    sy = o.project(h, w, P, v)[:, 0, 1]
    sel = sy > r if above else sy < r
    i = np.argmin(np.where(sel, np.abs(sy - r), np.inf))
    return ys[i]


def family_H(h, w):
    """Band edges: triangles whose bottom (or top) edge is horizontal one lattice step below (above) a row in H_ROWS, the
    far vertex at moderate |y| or at |y| near 1e9.  Each 256-triangle chunk holds copies of ONE such triangle at
    different x, so that the chunk pre-pass is the deciding test for the chunk.  Most chunks are the case the pre-pass's
    approximate reciprocal can get wrong, at many camera depths: a bottom edge one lattice step below a band's first row,
    which the band must list although the edge is within one rounding of the row."""
    rng = np.random.default_rng(8)
    chunks = []
    for r in H_ROWS:
        for j in range(32):
            z = F32(rng.uniform(1.1, 3.9))
            above = j % 2 == 0 or j >= 8                      # horizontal edge just below row r (max y): the band starting at r gets one row
            ye = _y_near_row(h, w, r, z, above=above)
            far = 1e9 * (0.999 if j % 4 < 2 else 1.001)
            ytip = (r - 9.0 if above else r + 9.0) if not 4 <= j < 8 else (-far if above else far)
            _, yt = _camera(h, w, FOV, 0.0, ytip, float(z))
            x0 = rng.uniform(2, w - 30, 256)
            xs = np.stack([x0, x0 + 20, x0 + 10], axis=1)
            xc, _ = _camera(h, w, FOV, xs, 0.0, float(z))
            v = np.empty((256, 3, 3), F32)
            v[:, :, 0] = xc
            v[:, 0, 1] = ye
            v[:, 1, 1] = ye
            v[:, 2, 1] = F32(yt)
            v[:, :, 2] = z
            chunks.append(v)
    return _model(np.concatenate(chunks), rng)


FAMILIES = {"A": family_A, "B": family_B, "C": family_C, "D": family_D, "E": family_E, "F": family_F, "G": family_G,
            "H": family_H}
_CACHE = {}


def family(name, h, w):
    key = (name, h, w)
    if key not in _CACHE:
        _CACHE[key] = FAMILIES[name](h, w)
    return _CACHE[key]


def concat(*models):
    return TriModel(*(np.ascontiguousarray(np.concatenate([getattr(m, a) for m in models])) for a in
                      ("_vertices_by_triangles", "_colors_by_triangles", "_normals_by_triangles")))


# ---------------------------------------------------------------------------------------------------- CPU tests
def _covered_fragments(cl, pick):
    """(triangle, numerators) for every pixel of the picked triangles' rectangles where no barycentric is negative."""
    out = []
    s = cl["s"]
    for t in np.flatnonzero(pick):
        x0, x1, y0, y1 = cl["rect"][t]
        for py in range(y0, y1):
            for px in range(x0, x1):
                with np.errstate(all="ignore"):
                    nn = np.array([a[0] for a in numerators(s[t:t + 1], px, py)])
                    b = nn / cl["l3"][t]
                if not (b < 0).any():
                    out.append((t, nn))
    return out


def test_edge_families_reach_their_regimes():
    h, w = SIZES[0]
    C = {k: (family(k, h, w), classify(h, w, FOV, family(k, h, w)._vertices_by_triangles, family(k, h, w)._normals_by_triangles))
         for k in FAMILIES}
    big = np.float32(2.0 ** 17)
    _, a = C["A"]
    assert int((a["drawn"] & a["span"] & (a["cmax"] > big)).sum()) >= 20
    _, b = C["B"]
    d = b["drawn"]
    assert d.sum() >= 20 and b["rej"][d].all() and not b["span"][d].any()
    assert ((b["cmax"][d] > SPAN_COORD_MAX) & (b["cmax"][d] <= F32(2.0 ** 22))).all()
    _, c = C["C"]
    d = c["drawn"]
    a3 = np.abs(c["l3"])
    huge = (a3 > FDIV_HI) & (a3 <= L3_MAX)
    assert (d & huge.any(axis=1) & ~c["fdiv"]).sum() >= 5 and c["rej"][huge & d[:, None]].all()
    assert (d & ((a3 > L3_MAX) | np.isnan(a3)).any(axis=1)).sum() >= 3          # the -inf threshold
    _, dd = C["D"]
    d = dd["drawn"]
    assert (d & (np.fmin.reduce(np.abs(dd["l3"]), axis=1) < FDIV_LO)).sum() >= 5
    frags = _covered_fragments(dd, d)
    assert sum(1 for _, nn in frags if (np.abs(nn) < FDIV_LO).any()) >= 5
    _, e = C["E"]
    assert e["drawn"].sum() >= 100 and (e["drawn"] & (e["cmax"] == big)).sum() == 3
    mf, f = C["F"]
    l3 = f["l3"]
    sgn = np.sign(l3)
    mixed = (sgn.max(axis=1) > 0) & (sgn.min(axis=1) < 0)
    one_zero = (l3 == 0).sum(axis=1) == 1
    assert (f["drawn"] & (mixed | one_zero)).sum() >= 20
    o = O().OracleFiller(h, w, fov=FOV)
    o.render_model(mf)
    assert int((o.get_z_buffer() < 1e5).sum()) >= 50
    mg, g = C["G"]
    o = O().OracleFiller(h, w, fov=FOV)
    o.render_model(mg)
    z = o.get_z_buffer()
    assert (z < 0).any() and np.isneginf(z).any() and (z == 0).any()
    s = g["s"][-6:] if mg.clear_depth_found else g["s"][-4:]   # the clear-value vertices: below / above / at 1e6
    px = [(w // 4, h // 4), (w // 4, 3 * h // 8), (3 * w // 8, h // 4)]
    for k in range(len(s) // 2):
        assert (s[2 * k:2 * k + 2, 0, 0] == px[k][0]).all() and (s[2 * k:2 * k + 2, 0, 1] == px[k][1]).all()
    assert (s[0:2, 0, 2] < Z_INIT).all() and (s[2:4, 0, 2] > Z_INIT).all() and (s[4:, 0, 2] == Z_INIT).all()
    assert z[h // 4, w // 4] == s[0, 0, 2] and z[3 * h // 8, w // 4] == Z_INIT
    if mg.clear_depth_found:      # drawn: an equal depth overwrites (pyx:223)
        assert z[h // 4, 3 * w // 8] == Z_INIT and o.get_color_buffer()[h // 4, 3 * w // 8].any()
    assert np.isinf(g["s"][..., 2]).any(axis=1).sum() >= 4 and np.isposinf(g["s"][..., 2]).any()
    print(f"family G: a vertex with depth exactly 1e6 {'was' if mg.clear_depth_found else 'was not'} found")
    mh, hh = C["H"]
    sy = hh["s"][..., 1]
    edge = sy[:, 0]                                       # vertices 0 and 1 form the horizontal edge
    assert (sy[:, 1] == edge).all()
    assert all(((edge > r) & (edge - r < 1e-4)).sum() == 256 * 28 and ((edge < r) & (r - edge < 1e-4)).sum() == 256 * 4
               for r in H_ROWS)
    assert hh["drawn"].sum() >= 0.9 * len(hh["drawn"])
    assert (np.abs(sy) >= 9.9e8).any(axis=1).sum() >= 256 * 8


@pytest.mark.skipif(platform.machine() not in ("x86_64", "AMD64"), reason="NumPy's float -> uint8 cast is platform-defined")
def test_uint8_cast_known_answers():
    """run.py:26's `astype('uint8')` on x86-64 (cvttss2si, then the low byte) -- what to_u8 restates."""
    vals = np.array([3e9, 2.0 ** 31, 1e30, np.inf, -3e9, -np.inf, np.nan, 300.7, -3.5, 1e6], F32)
    with np.errstate(invalid="ignore"):
        got = vals.astype("uint8")
    assert got.tolist() == [0, 0, 0, 0, 0, 0, 0, 44, 253, 64]


# ---------------------------------------------------------------------------------------------------- GPU tests
def _buffers(f):
    return f.get_z_buffer().copy(), f.get_color_buffer().copy(), f.get_normals_buffer().copy()


def _assert_same(got, want, what):
    for name, g, w in zip(("z", "color", "normals"), got, want):
        if not bits_equal(g, w):
            bad = np.argwhere(g.view(np.uint32) != w.view(np.uint32))
            raise AssertionError(f"{what}: {name} differs at {len(bad)} words, first {bad[:5].tolist()}: "
                                 f"got {g[tuple(bad[0])]!r} want {w[tuple(bad[0])]!r}")


def _mv(m):
    return m._vertices_by_triangles, m._colors_by_triangles, m._normals_by_triangles


@pytest.fixture(scope="module")
def oracle_frames():
    """Oracle frames, each rendered once per module: (family, h, w, composited) -> (z, colour, normals)."""
    cache = {}

    def get(name, h, w, composite=False):
        key = (name, h, w, composite)
        if key not in cache:
            o = O().OracleFiller(h, w, fov=FOV)
            if composite:
                o.render_model(random_scene(17, T=300))
            o.render_model(family(name, h, w))
            cache[key] = _buffers(o)
        return cache[key]
    return get


CONFIGS = {"default": {}, "atomic": {}, "shape1": {"RASTER_SHAPE": 1}, "shape2": {"RASTER_SHAPE": 2},
           "shape3": {"RASTER_SHAPE": 3}, "split_heavy0": {"SPLIT_HEAVY": 0}, "wide_kernel0": {"WIDE_KERNEL": 0},
           "tma0": {"TMA": 0}}


@pytest.mark.gpu
@pytest.mark.parametrize("size", SIZES, ids=lambda s: f"{s[0]}x{s[1]}")
@pytest.mark.parametrize("config", sorted(CONFIGS))
@pytest.mark.parametrize("name", sorted(FAMILIES))
def test_edge_families_bit_exact(name, config, size, oracle_frames):
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller, _lib
    h, w = size
    m = family(name, h, w)
    path = "atomic" if config == "atomic" else "tiled"
    for composite in (False, True):
        f = AdvancedPixelBufferFiller(h, w, fov=FOV)
        for opt, val in CONFIGS[config].items():
            f.set_option(getattr(_lib, "CRB_OPT_" + opt), val)
        if composite:
            f.render_model(random_scene(17, T=300))
        f.render_arrays(*_mv(m), path=path)
        _assert_same(_buffers(f), oracle_frames(name, h, w, composite), f"family {name} {config} {h}x{w} composite={composite}")


@pytest.mark.gpu
@pytest.mark.parametrize("size", SIZES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_edge_families_in_batched_views(size):
    """render_views with chunk < views, views at and near identity, fused uint8 output: per view, the oracle fed the
    camera-space arrays the view transform produces."""
    import torch
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller, views as VW
    h, w = size
    m = concat(*(family(k, h, w) for k in ("A", "C", "D", "E", "F", "G")))
    views = np.stack([VW.view_matrix(), VW.view_matrix(VW.rot_y(1e-6), p=(0.0, 0.0, 1.0)),
                      VW.view_matrix(VW.rot_y(-3e-4), p=(0.0, 0.0, 2.0)), VW.view_matrix(q=(1e-4, -2e-4, 0.0))])
    dv, dc, dn = (torch.from_numpy(a).cuda() for a in _mv(m))
    f = AdvancedPixelBufferFiller(h, w, fov=FOV)
    out = f.render_views(dv, dc, dn, views, chunk=3, color_u8_out=True)
    for k in range(len(views)):
        vk, nk = VW.transform_arrays_host(views[k], m._vertices_by_triangles, m._normals_by_triangles)
        gv, gn = f.transform_view(dv, dn, views[k])
        gv, gn = gv.cpu().numpy(), gn.cpu().numpy()
        assert bits_equal(gv, vk) and bits_equal(gn, nk)
        o = O().OracleFiller(h, w, fov=FOV)
        o.render_arrays(gv, m._colors_by_triangles, gn)
        got = tuple(out[n][k].cpu().numpy() for n in ("z", "color", "normals"))
        _assert_same(got, _buffers(o), f"view {k} {h}x{w}")
        with np.errstate(invalid="ignore"):
            want_u8 = o.get_color_buffer()[::-1].astype("uint8")
        assert np.array_equal(out["color_u8"][k].cpu().numpy(), want_u8), f"uint8 view {k}"


@pytest.mark.gpu
@pytest.mark.parametrize("prepass", [1, 0])
@pytest.mark.parametrize("size", SIZES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_edge_families_in_bands(size, prepass):
    """Row bands (not aligned to tiles, one-row bands, the first and last row, bands starting and ending at the rows H's
    edges touch) over families H, A and E, with and without the chunk pre-pass: each band equals the oracle's rows."""
    import torch
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller, _lib
    h, w = size
    m = concat(family("H", h, w), family("A", h, w), family("E", h, w))
    o = O().OracleFiller(h, w, fov=FOV)
    o.render_model(m)
    want = _buffers(o)
    dv, dc, dn = (torch.from_numpy(a).cuda() for a in _mv(m))
    cuts = sorted({0, 1, 2, h - 1, h} | set(H_ROWS) | {r + 1 for r in H_ROWS} | {r - 1 for r in H_ROWS} | {h // 2 + 3})
    bands = list(zip(cuts[:-1], cuts[1:])) + [(0, h), (H_ROWS[0], H_ROWS[-1]), (5, H_ROWS[1])]
    for r0, r1 in bands:
        f = AdvancedPixelBufferFiller(h, w, fov=FOV, band=(r0, r1))
        f.set_option(_lib.CRB_OPT_BAND_PREPASS, prepass)
        f.render_arrays(dv, dc, dn)
        _assert_same(_buffers(f), tuple(a[r0:r1] for a in want), f"band {r0}:{r1} prepass={prepass} {h}x{w}")


@pytest.mark.gpu
def test_largest_supported_dimensions():
    """65535 x 33 and 33 x 65535: the 16-bit rectangle packing at its limit and tile index 2047; 65536 is refused."""
    import ctypes
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller, _lib
    for h, w in ((65535, 33), (33, 65535)):
        rng = np.random.default_rng(h)
        T = 24
        if h > w:
            ys = np.stack([rng.uniform(0, h, T), rng.uniform(0, h, T), rng.uniform(-10, h + 10, T)], axis=1)
            xs = np.stack([np.full(T, -2.0), np.full(T, w + 2.0), rng.uniform(0, w, T)], axis=1)
        else:
            xs = np.stack([rng.uniform(0, w, T), rng.uniform(0, w, T), rng.uniform(-10, w + 10, T)], axis=1)
            ys = np.stack([np.full(T, -2.0), np.full(T, h + 2.0), rng.uniform(0, h, T)], axis=1)
        xs[0], ys[0] = (w - 3, w + 5, w - 3), (h - 3, h - 3, h + 5)         # covers the last pixel (w-1, h-1)
        m = _model(_tris(h, w, xs, ys, np.repeat(rng.uniform(1, 3, (T, 1)), 3, axis=1)), rng)
        o = O().OracleFiller(h, w, fov=FOV)
        o.render_model(m)
        z = o.get_z_buffer()
        assert (z[h - 1, w - 1] < 1e5) and (z < 1e5).sum() > 1000
        for path in ("tiled", "atomic"):
            f = AdvancedPixelBufferFiller(h, w, fov=FOV)
            f.render_arrays(*_mv(m), path=path)
            _assert_same(_buffers(f), _buffers(o), f"{h}x{w} {path}")
            del f
    L = _lib.load_library()
    for h, w in ((65536, 33), (33, 65536)):
        handle = ctypes.c_void_p()
        assert L.crb_create(h, w, FOV, 0.1, 1000.0, 0, ctypes.byref(handle)) == _lib.CRB_ERR_INVALID
        with pytest.raises(_lib.CrenderError):
            AdvancedPixelBufferFiller(h, w, fov=FOV)


U8_VALUES = np.array([3e9, 2.0 ** 31, 1e30, np.inf, -3e9, -np.inf, np.nan, 300.7, -3.5, 1e6, 255.9, -0.5, 2147483520.0,
                      -2147483648.0, 65535.5, 1e9], F32)


def _u8_model(h, w):
    """A grid of small quads, each flat in one colour from U8_VALUES or from (255, 2^31); normals of magnitude up to 1e9."""
    rng = np.random.default_rng(9)
    cols = np.concatenate([U8_VALUES, np.exp(rng.uniform(np.log(256.0), np.log(2.0 ** 31), 40)).astype(F32),
                           -np.exp(rng.uniform(0, np.log(2.0 ** 31), 8)).astype(F32)])
    tris, cs = [], []
    g = int(np.ceil(np.sqrt(len(cols))))
    sx, sy = w / g, h / g
    for i, c in enumerate(cols):
        x0, y0 = (i % g) * sx + 0.3, (i // g) * sy + 0.3
        for t in (((x0, y0), (x0 + sx, y0), (x0 + sx, y0 + sy)), ((x0, y0), (x0 + sx, y0 + sy), (x0, y0 + sy))):
            tris.append(t)
            cs.append(c)
    pts = np.asarray(tris)
    v = _tris(h, w, pts[..., 0], pts[..., 1], np.ones(pts.shape[:2]))
    c = np.repeat(np.asarray(cs, F32)[:, None, None], 3, axis=1).repeat(3, axis=2)
    c[:, :, 1] *= F32(0.5)
    n = rng.standard_normal(v.shape).astype(F32)
    n[..., 2] = -np.abs(n[..., 2]) - F32(0.5)
    n *= np.exp(rng.uniform(0, np.log(1e9), (len(v), 3, 1))).astype(F32)
    return TriModel(np.ascontiguousarray(v), np.ascontiguousarray(c), np.ascontiguousarray(n))


@pytest.mark.gpu
@pytest.mark.parametrize("entry", ["color_u8_flipped", "render_views", "host_image_pipeline"])
@pytest.mark.parametrize("lit", [False, True])
def test_uint8_stage_on_out_of_range_colours(lit, entry):
    import torch
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller, HostImagePipeline, views as VW
    h, w = 96, 128
    m = _u8_model(h, w)
    light = [0.2, -0.1, 1.0]
    o = O().OracleFiller(h, w, fov=FOV)
    o.render_model(m)
    if lit:
        O().guro(o.get_color_buffer(), o.get_normals_buffer(), light)
    col = o.get_color_buffer()
    assert (col >= 2.0 ** 31).any() and (col < 0).any() and np.isnan(col).any() and ((col > 255) & (col < 2.0 ** 31)).any()
    with np.errstate(invalid="ignore"):
        want = col[::-1].astype("uint8")
    if entry == "color_u8_flipped":
        f = AdvancedPixelBufferFiller(h, w, fov=FOV)
        f.render_model(m)
        if lit:
            l = -np.asarray(light, dtype="float32")
            f.illuminate_guro(l / np.linalg.norm(l))
        got = f.color_u8_flipped().cpu().numpy()
    elif entry == "render_views":
        f = AdvancedPixelBufferFiller(h, w, fov=FOV)
        dv, dc, dn = (torch.from_numpy(a).cuda() for a in _mv(m))
        got = f.render_views(dv, dc, dn, VW.view_matrix()[None], color_u8_out=True,
                             guro_light=light if lit else None)["color_u8"][0].cpu().numpy()
    else:
        pipe = HostImagePipeline(h, w, fov=FOV, depth=1, light=light if lit else None)
        got = pipe.result(pipe.submit(torch.from_numpy(np.stack(_mv(m))).pin_memory())).copy()
    bad = np.argwhere(got != want)
    assert bad.size == 0, (f"{len(bad)} bytes differ, first {bad[:5].tolist()}: got {got[tuple(bad[0])]} want "
                           f"{want[tuple(bad[0])]} from colour {col[::-1][tuple(bad[0])]!r}")


@pytest.mark.ref
@pytest.mark.parametrize("name", ["C", "D", "F", "G"])
def test_oracle_equals_reference_build_on_edge_families(name, capfd):
    """The oracle against the reference's own build on the families random scenes never reach (where oracle/_ref exists)."""
    import sys
    from oracle import build_ref
    if not build_ref.built():
        pytest.skip("the reference's own build (oracle/_ref) is not present")
    ref = os.path.join(ROOT, "oracle", "_ref")
    if ref not in sys.path:
        sys.path.insert(0, ref)
    from crender.cy.pixel_buffer_filler import AdvancedPixelBufferFiller
    for h, w in SIZES:
        m = family(name, h, w)
        o = O().OracleFiller(h, w, fov=FOV)
        o.render_model(m)
        r = AdvancedPixelBufferFiller(h, w, fov=FOV, n_threads=1)
        r.render_model(m)
        capfd.readouterr()
        _assert_same(_buffers(r), _buffers(o), f"family {name} {h}x{w}")
