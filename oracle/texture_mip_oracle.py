"""CPU oracle of trilinear mip filtering, CRB_TEX_TRILINEAR (DESIGN 2) -- an extension of this project, like
oracle/texture_modes_oracle.py, which it builds on and leaves as it is.

TEST INFRASTRUCTURE ONLY.  The mode is defined by composing pinned pieces with NumPy statements of the new parts:

  1. the colour slots (u, v, -), or with perspective texture_modes_oracle.perspective_slots' (u*w, v*w, w), go through
     oracle_render unchanged, which leaves each winning fragment's interpolated slots in the colour buffer;
  2. winner_ids: the triangle that wrote each pixel last.  The level of detail needs the triangle, and interpolating a
     per-triangle constant through the colour slots does not return it exactly.  Under the sequential z-test (an equal depth
     overwrites) the last writer of a pixel is the highest-index triangle of the render that draw_triangle would draw there --
     not culled, the pixel inside its rectangle, every barycentric >= 0, depth not NaN -- whose depth == the final z;
  3. lod: the barycentric gradients from the projected corners, the derivatives of (u, v), the footprint, the piecewise-linear
     log2 (log2_substitute) and the clamped level, in NumPy float32;
  4. mip_chain: the chain in NumPy integers, each level sampled with texture_modes_oracle.bilinear_texels and the two levels
     blended in float32.

tests/test_texture_mip_oracle.py checks the pieces against the definition.
"""
import numpy as np

from oracle import oracle as O
from oracle import texture_modes_oracle as TM
from oracle import texture_oracle as TX

F32 = np.float32
INT_MIN = np.int64(-2147483648)


def mip_chain(texture):
    """The mip chain of a uint8 [th,tw,3] texture as a list of uint8 [h_k,w_k,3] levels, level 0 the texture: level k+1 is
    max(1, h_k >> 1) x max(1, w_k >> 1), per channel (t[r0][c0] + t[r0][c1] + t[r1][c0] + t[r1][c1] + 2) >> 2 with
    r0 = min(2r, h_k - 1), r1 = min(2r + 1, h_k - 1), columns alike."""
    t = TX._check_texture(texture)
    levels = [t]
    while t.shape[0] > 1 or t.shape[1] > 1:
        h, w = t.shape[:2]
        r, c = np.arange(max(1, h >> 1)), np.arange(max(1, w >> 1))
        r0, r1 = np.minimum(2 * r, h - 1), np.minimum(2 * r + 1, h - 1)
        c0, c1 = np.minimum(2 * c, w - 1), np.minimum(2 * c + 1, w - 1)
        a = t.astype(np.int32)
        s = a[r0][:, c0] + a[r0][:, c1] + a[r1][:, c0] + a[r1][:, c1] + 2
        t = (s >> 2).astype(np.uint8)
        levels.append(t)
    return levels


def pack_chain(levels):
    """The levels packed as crb_pack_texture_mips stores them: B | G << 8 | R << 16, row-major, back to back (uint32)."""
    out = []
    for t in levels:
        a = t.reshape(-1, 3).astype(np.uint32)
        out.append(a[:, 0] | (a[:, 1] << 8) | (a[:, 2] << 16))
    return np.concatenate(out)


def log2_substitute(r2):
    """L2(r2) = (k - 1) + (2f - 1) for r2 = f * 2^k, f in [0.5, 1) (frexp); 0 -> -inf, +inf -> +inf, NaN -> NaN (float32)."""
    r2 = np.asarray(r2, F32)
    f, k = np.frexp(r2)
    with np.errstate(invalid="ignore"):
        out = (k - 1).astype(F32) + (F32(2) * f - F32(1))
    out = np.where(r2 == 0, F32(-np.inf), out)
    return np.where(np.isposinf(r2), F32(np.inf), out).astype(F32)


def levels_of(th, tw):
    """L = 1 + floor(log2(max(th, tw)))."""
    return int(max(th, tw)).bit_length()


def lod(scr, slots, colour, perspective, th, tw):
    """(lambda, lambda_c) of pixels: scr [N,3,3] the projected corners of each pixel's triangle, slots [N,3,3] its colour slots,
    colour [N,3] the pixel's interpolated slots, (th, tw) the texture's size (float32, one rounding per operation)."""
    scr, slots, colour = (np.asarray(a, F32) for a in (scr, slots, colour))
    x0, y0, x1, y1, x2, y2 = (scr[:, k, j] for k in range(3) for j in range(2))
    with np.errstate(all="ignore"):
        l03 = (x1 - x2) * (y0 - y2) - (y1 - y2) * (x0 - x2)      # oracle_barycentric's denominators
        l13 = (x2 - x0) * (y1 - y0) - (y2 - y0) * (x1 - x0)
        l23 = (x0 - x1) * (y2 - y1) - (y0 - y1) * (x2 - x1)
        gx = ((y2 - y1) / l03, (y0 - y2) / l13, (y1 - y0) / l23)
        gy = ((x1 - x2) / l03, (x2 - x0) / l13, (x0 - x1) / l23)

        def d(j, g):
            return (slots[:, 0, j] * g[0] + slots[:, 1, j] * g[1]) + slots[:, 2, j] * g[2]

        ux, vx, uy, vy = d(0, gx), d(1, gx), d(0, gy), d(1, gy)
        if perspective:
            u, v = TM.pixel_uv(colour, True)
            W = colour[:, 2]
            wx, wy = d(2, gx), d(2, gy)
            ux, vx = (ux - u * wx) / W, (vx - v * wx) / W
            uy, vy = (uy - u * wy) / W, (vy - v * wy) / W
        p, q, r, s = ux * F32(tw), vx * F32(th), uy * F32(tw), vy * F32(th)
        r2 = np.fmax(p * p + q * q, r * r + s * s)
        lam = F32(0.5) * log2_substitute(r2)
    lc = np.fmin(np.fmax(lam, F32(0)), F32(levels_of(th, tw) - 1))      # fmax: NaN -> 0
    return lam.astype(F32), lc.astype(F32)


def trilinear_texels(u, v, lc, levels):
    """Colour of pixels at (u, v) with clamped level lc [N]: bilinear samples of levels floor(lc) and min(floor(lc) + 1, L-1),
    blended c0*(1 - fr) + c1*fr, fr = lc - floor(lc) (float BGR [N,3])."""
    u, v, lc = (np.asarray(a, F32).ravel() for a in (u, v, lc))
    l0 = np.floor(lc).astype(np.int64)
    fr = (lc - l0.astype(F32))[:, None]
    l1 = np.minimum(l0 + 1, len(levels) - 1)
    c0, c1 = np.zeros((u.size, 3), F32), np.zeros((u.size, 3), F32)
    for lv in np.unique(np.concatenate([l0, l1])):
        for ls, c in ((l0, c0), (l1, c1)):
            sel = ls == lv
            if sel.any():
                c[sel] = TM.bilinear_texels(u[sel], v[sel], levels[lv])
    return c0 * (F32(1) - fr) + c1 * fr


def _ceil_to_int(x):
    c = np.ceil(np.asarray(x, np.float64))
    with np.errstate(invalid="ignore"):
        ok = (c > -2147483649.0) & (c < 2147483648.0)
    return np.where(ok, np.nan_to_num(c), INT_MIN).astype(np.int64)


def winner_ids(h, w, P, v, n, z_final, max_candidates=1 << 22):
    """Index of the triangle of this render that wrote each pixel last ([h,w] int64, -1 where none did), for the [T,3,3]
    vertices / normals `v`, `n` rendered with projection P into a buffer whose depth is now `z_final`."""
    scr = O.project(h, w, P, v)
    n = np.asarray(n, F32)
    with np.errstate(invalid="ignore"):
        culled = ((n[:, 0, 2] + n[:, 1, 2]) + n[:, 2, 2]) >= 0           # pyx:202-204 (only the sign of the float sum)
    x, y = scr[..., 0], scr[..., 1]
    xl = np.fmin(np.fmin(np.fmin(F32(w), x[:, 0]), x[:, 1]), x[:, 2])   # oracle_pixel_rect: NaN never wins a comparison
    xr = np.fmax(np.fmax(np.fmax(F32(0), x[:, 0]), x[:, 1]), x[:, 2])
    yt = np.fmin(np.fmin(np.fmin(F32(h), y[:, 0]), y[:, 1]), y[:, 2])
    yb = np.fmax(np.fmax(np.fmax(F32(0), y[:, 0]), y[:, 1]), y[:, 2])
    r0, r1 = (np.clip(_ceil_to_int(a), 0, w) for a in (xl, xr))
    r2, r3 = (np.clip(_ceil_to_int(a), 0, h) for a in (yt, yb))
    nx, ny = np.maximum(r1 - r0, 0), np.maximum(r3 - r2, 0)
    cnt = np.where(culled, 0, nx * ny)
    win = np.full(h * w, -1, np.int64)
    zf = np.asarray(z_final, F32).ravel()
    tris = np.flatnonzero(cnt)
    csum = np.cumsum(cnt[tris])
    start = 0
    while start < tris.size:
        base = csum[start - 1] if start else 0
        stop = max(start + 1, int(np.searchsorted(csum, base + max_candidates, side="right")))
        t = tris[start:stop]
        k = cnt[t]
        rep = np.repeat(t, k)
        local = np.arange(int(k.sum())) - np.repeat(np.cumsum(k) - k, k)
        px = r0[rep] + local // ny[rep]
        py = r2[rep] + local % ny[rep]
        s = scr[rep]
        b = _bary(s, px, py)
        b0, b1, b2 = b[:, 0], b[:, 1], b[:, 2]
        with np.errstate(all="ignore"):
            z = (s[:, 0, 2] * b0 + s[:, 1, 2] * b1) + s[:, 2, 2] * b2
            pix = py * w + px
            keep = ~((b0 < 0) | (b1 < 0) | (b2 < 0)) & ~np.isnan(z) & (z == zf[pix])
        np.maximum.at(win, pix[keep], rep[keep])
        start = stop
    return win.reshape(h, w)


def restate(h, w, P, v, n, ids):
    """z [h,w] and normals [h,w,3] of the pixels ids >= 0, restated from their winning triangles (the self-check of
    winner_ids against oracle_render); NaN elsewhere."""
    scr = O.project(h, w, P, v)
    n = np.asarray(n, F32)
    ys, xs = np.nonzero(ids >= 0)
    t = ids[ys, xs]
    z = np.full((h, w), np.nan, F32)
    nb = np.full((h, w, 3), np.nan, F32)
    b = _bary(scr[t], xs, ys)
    with np.errstate(all="ignore"):
        z[ys, xs] = (scr[t, 0, 2] * b[:, 0] + scr[t, 1, 2] * b[:, 1]) + scr[t, 2, 2] * b[:, 2]
        for j in range(3):
            nb[ys, xs, j] = (n[t, 0, j] * b[:, 0] + n[t, 1, j] * b[:, 1]) + n[t, 2, j] * b[:, 2]
    return z, nb


def _bary(s, xs, ys):
    """oracle_barycentric (mu:5-34) of pixels (xs, ys) in projected triangles s [N,3,3], float32 [N,3]."""
    fx, fy = xs.astype(F32), ys.astype(F32)
    X0, Y0, X1, Y1, X2, Y2 = (s[:, k, j] for k in range(3) for j in range(2))
    with np.errstate(all="ignore"):
        l01, l02, l11, l12, l21, l22 = X1 - X2, Y1 - Y2, X2 - X0, Y2 - Y0, X0 - X1, Y0 - Y1
        return np.stack([(l01 * (fy - Y2) - l02 * (fx - X2)) / (l01 * (Y0 - Y2) - l02 * (X0 - X2)),
                         (l11 * (fy - Y0) - l12 * (fx - X0)) / (l11 * (Y1 - Y0) - l12 * (X1 - X0)),
                         (l21 * (fy - Y1) - l22 * (fx - X1)) / (l21 * (Y2 - Y1) - l22 * (X2 - X1))], axis=1)


def render_textured(filler, v, uv, n, texture, perspective=False, levels=None, return_lod=False):
    """Composites the trilinear textured render of [T,3,3] v / n with texture coordinates `uv` into an OracleFiller's buffers,
    from affine or (perspective=True) perspective-correct coordinates.  return_lod: also (ids, lambda, lambda_c) of the drawn
    pixels, row-major."""
    tex = TX._check_texture(texture)
    levels = mip_chain(tex) if levels is None else levels
    slots = TM.perspective_slots(v, uv) if perspective else np.ascontiguousarray(TX._uv_triples(uv), dtype=F32)
    filler.render_arrays(v, slots, n)
    ids = winner_ids(filler.h, filler.w, filler.proj_mat.ravel(), v, n, filler.z_buffer)
    drawn = ids >= 0
    t = ids[drawn]
    c = filler.color_buffer
    col = c[drawn]
    scr = O.project(filler.h, filler.w, filler.proj_mat.ravel(), v)
    lam, lc = lod(scr[t], slots[t], col, perspective, *tex.shape[:2])
    u_, v_ = TM.pixel_uv(col, perspective)
    c[drawn] = trilinear_texels(u_, v_, lc, levels)
    if return_lod:
        return ids, lam, lc


class TexturedOracleFiller(TM.TexturedOracleFiller):
    """texture_modes_oracle.TexturedOracleFiller whose render_arrays also takes filter="trilinear"."""

    def render_arrays(self, v, c, n, texture=None, perspective=False, filter="nearest"):
        if filter == "trilinear":
            if texture is None:
                raise ValueError("filter='trilinear' needs a texture")
            return render_textured(self, v, c, n, texture, perspective=perspective)
        return super().render_arrays(v, c, n, texture=texture, perspective=perspective, filter=filter)
