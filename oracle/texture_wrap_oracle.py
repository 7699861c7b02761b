"""CPU oracle of the wrap modes of per-pixel texturing, CRB_TEX_REPEAT and CRB_TEX_MIRROR (DESIGN 2) -- an extension of this
project, like oracle/texture_modes_oracle.py and oracle/texture_mip_oracle.py, which it builds on and leaves as they are.

TEST INFRASTRUCTURE ONLY.  The modes are defined by composing the same pinned pieces as the clamped oracles:

  1. the colour slots (u, v, -), or with perspective texture_modes_oracle.perspective_slots' (u*w, v*w, w), go through
     oracle_render unchanged, which leaves each winning fragment's interpolated slots in the colour buffer;
  2. the pixels this render drew: for nearest and bilinear the NaN-colour scratch render of texture_oracle, for trilinear
     texture_mip_oracle.winner_ids and its level of detail (lod), which the wrap mode does not change;
  3. texture_modes_oracle.pixel_uv;
  4. the wrapped samplers below (ifloor, wrap_index; nearest_texels, bilinear_texels, trilinear_texels over mip_chain levels).

wrap="clamp" delegates to the clamped oracles unchanged.  tests/test_texture_wrap_oracle.py checks the samplers against a
scalar restatement and the composition against the definition.
"""
import numpy as np

from oracle import ingest as I
from oracle import oracle as O
from oracle import texture_mip_oracle as MIP
from oracle import texture_modes_oracle as TM
from oracle import texture_oracle as TX

F32 = np.float32
WRAPS = ("clamp", "repeat", "mirror")
FILTERS = ("nearest", "bilinear", "trilinear")
_LIMIT = F32(2.0 ** 31)


def _check_wrap(wrap, allow_clamp=True):
    if wrap not in (WRAPS if allow_clamp else WRAPS[1:]):
        raise ValueError(f"wrap must be one of {WRAPS if allow_clamp else WRAPS[1:]}, got {wrap!r}")


def wrap_arg(x):
    """The float an index is floored from: NaN and |x| >= 2^31 become F(0) (float32)."""
    x = np.asarray(x, F32)
    with np.errstate(invalid="ignore"):
        return np.where(np.abs(x) < _LIMIT, x, F32(0)).astype(F32)


def ifloor(x):
    """ifloor(x) = int(floor(wrap_arg(x))) as int64; the result and the result + 1 fit int32."""
    return np.floor(wrap_arg(x)).astype(np.int64)


def wrap_index(k, n, wrap):
    """Integer indices k wrapped into [0, n) (int64): repeat k mod n, mirror m = k mod 2n then m < n ? m : 2n - 1 - m (floor
    modulo, np.mod)."""
    _check_wrap(wrap, allow_clamp=False)
    k = np.asarray(k, np.int64)
    n = int(n)
    if wrap == "repeat":
        return np.mod(k, n)
    m = np.mod(k, 2 * n)
    return np.where(m < n, m, 2 * n - 1 - m)


def nearest_texels(u, v, texture, wrap):
    """Nearest texels (float BGR [N,3]) of coordinates u, v [N]: col = wrap(ifloor(u*tw)), row = wrap(ifloor((1 - v)*th)).
    wrap="clamp": the texel rule of model.py:147-150 (ingest_vertex_colors)."""
    _check_wrap(wrap)
    tex = TX._check_texture(texture)
    u, v = np.asarray(u, F32).ravel(), np.asarray(v, F32).ravel()
    if wrap == "clamp":
        return I.vertex_colors(np.ascontiguousarray(np.stack([u, v], axis=1)), tex)
    th, tw = tex.shape[:2]
    with np.errstate(invalid="ignore", over="ignore"):
        col = wrap_index(ifloor(u * F32(tw)), tw, wrap)
        row = wrap_index(ifloor((F32(1) - v) * F32(th)), th, wrap)
    return tex[row, col].astype(F32)


def bilinear_texels(u, v, texture, wrap):
    """Bilinear blend (float BGR [N,3]) of coordinates u, v [N]: sx = u*tw - 0.5 (NaN or |sx| >= 2^31 -> 0), x0 = floor(sx),
    columns wrap(x0) and wrap(x0 + 1), rows alike, blended as texture_modes_oracle.bilinear_texels does.  wrap="clamp": that
    function itself."""
    _check_wrap(wrap)
    if wrap == "clamp":
        return TM.bilinear_texels(u, v, texture)
    tex = TX._check_texture(texture)
    th, tw = tex.shape[:2]
    u, v = np.asarray(u, F32).ravel(), np.asarray(v, F32).ravel()
    with np.errstate(invalid="ignore", over="ignore"):
        sx = wrap_arg(u * F32(tw) - F32(0.5))
        sy = wrap_arg((F32(1) - v) * F32(th) - F32(0.5))
    x0, y0 = np.floor(sx), np.floor(sy)
    fx, fy = sx - x0, sy - y0
    ix, iy = x0.astype(np.int64), y0.astype(np.int64)
    c0, c1 = wrap_index(ix, tw, wrap), wrap_index(ix + 1, tw, wrap)
    r0, r1 = wrap_index(iy, th, wrap), wrap_index(iy + 1, th, wrap)
    gx, gy = (F32(1) - fx)[:, None], (F32(1) - fy)[:, None]
    fx, fy = fx[:, None], fy[:, None]
    t = tex.astype(F32)
    top = t[r0, c0] * gx + t[r0, c1] * fx
    bot = t[r1, c0] * gx + t[r1, c1] * fx
    return top * gy + bot * fy


def trilinear_texels(u, v, lc, levels, wrap):
    """texture_mip_oracle.trilinear_texels with each level sampled by the wrapped bilinear rule on its own size."""
    _check_wrap(wrap)
    if wrap == "clamp":
        return MIP.trilinear_texels(u, v, lc, levels)
    u, v, lc = (np.asarray(a, F32).ravel() for a in (u, v, lc))
    l0 = np.floor(lc).astype(np.int64)
    fr = (lc - l0.astype(F32))[:, None]
    l1 = np.minimum(l0 + 1, len(levels) - 1)
    c0, c1 = np.zeros((u.size, 3), F32), np.zeros((u.size, 3), F32)
    for lv in np.unique(np.concatenate([l0, l1])):
        for ls, c in ((l0, c0), (l1, c1)):
            sel = ls == lv
            if sel.any():
                c[sel] = bilinear_texels(u[sel], v[sel], levels[lv], wrap)
    return c0 * (F32(1) - fr) + c1 * fr


def render_textured(filler, v, uv, n, texture, filter="nearest", perspective=False, wrap="clamp"):
    """Composites the textured render of [T,3,3] v / n with texture coordinates `uv` into an OracleFiller's buffers, sampled
    with `filter` and `wrap` from affine or (perspective=True) perspective-correct coordinates."""
    if filter not in FILTERS:
        raise ValueError(f"filter must be one of {FILTERS}, got {filter!r}")
    _check_wrap(wrap)
    if wrap == "clamp":
        if filter == "trilinear":
            return MIP.render_textured(filler, v, uv, n, texture, perspective=perspective)
        return TM.render_textured(filler, v, uv, n, texture, perspective=perspective, filter=filter)
    tex = TX._check_texture(texture)
    slots = TM.perspective_slots(v, uv) if perspective else np.ascontiguousarray(TX._uv_triples(uv), dtype=F32)
    if filter == "trilinear":
        filler.render_arrays(v, slots, n)
        ids = MIP.winner_ids(filler.h, filler.w, filler.proj_mat.ravel(), v, n, filler.z_buffer)
        drawn = ids >= 0
        c = filler.color_buffer
        col = c[drawn]
        scr = O.project(filler.h, filler.w, filler.proj_mat.ravel(), v)
        _, lc = MIP.lod(scr[ids[drawn]], slots[ids[drawn]], col, perspective, *tex.shape[:2])
        u_, v_ = TM.pixel_uv(col, perspective)
        c[drawn] = trilinear_texels(u_, v_, lc, MIP.mip_chain(tex), wrap)
        return
    scratch = O.OracleFiller(filler.h, filler.w, n_threads=filler.n_threads)
    scratch.proj_mat = filler.proj_mat
    scratch.z_buffer[...] = filler.z_buffer
    filler.render_arrays(v, slots, n)
    scratch.render_arrays(v, np.full(np.shape(v), np.nan, np.float32), n)
    drawn = np.isnan(scratch.color_buffer[..., 0])
    c = filler.color_buffer
    u_, v_ = TM.pixel_uv(c[drawn], perspective)
    c[drawn] = (bilinear_texels if filter == "bilinear" else nearest_texels)(u_, v_, tex, wrap)


class TexturedOracleFiller(MIP.TexturedOracleFiller):
    """texture_mip_oracle.TexturedOracleFiller whose textured renders address texels with `wrap` ("clamp", "repeat" or
    "mirror"), given to the constructor like the GPU filler's texture_wrap."""

    def __init__(self, *args, wrap="clamp", **kw):
        _check_wrap(wrap)
        super().__init__(*args, **kw)
        self.wrap = wrap

    def render_arrays(self, v, c, n, texture=None, perspective=False, filter="nearest"):
        if texture is None or self.wrap == "clamp":
            return super().render_arrays(v, c, n, texture=texture, perspective=perspective, filter=filter)
        return render_textured(self, v, c, n, texture, filter=filter, perspective=perspective, wrap=self.wrap)
