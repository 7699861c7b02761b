"""CPU oracle of the two modes of per-pixel texturing, CRB_TEX_PERSPECTIVE and CRB_TEX_BILINEAR (DESIGN 2) -- an extension of
this project, like oracle/texture_oracle.py, which it builds on and leaves as it is.

TEST INFRASTRUCTURE ONLY.  The modes are defined by composing the same pinned pieces as the textured oracle:

  1. perspective=True: a NumPy float32 prelude (perspective_slots) puts (u*w, v*w, w), w = 1 / z with z the camera-space
     depth of the arrays passed, into the colour slots of each corner;
  2. oracle_render, unchanged, interpolates them (visibility, depth and normals do not depend on the colours);
  3. pixel_uv: at every pixel this render drew, (u, v) = (U, V), or with perspective (U / W, V / W);
  4. filter="nearest": ingest_vertex_colors, the texel rule of model.py:147-150 (as in texture_oracle); filter="bilinear":
     bilinear_texels, a NumPy float32 statement of the bilinear rule.

Nearest sampling of affine coordinates is texture_oracle.render_textured itself.  tests/test_texture_filter_oracle.py checks
the composition against the definitions.
"""
import numpy as np

from oracle import ingest as I
from oracle import oracle as O
from oracle import texture_oracle as TX

F32 = np.float32
FILTERS = ("nearest", "bilinear")


def perspective_slots(v, uv):
    """The colour slots of CRB_TEX_PERSPECTIVE: per corner (u*w, v*w, w), w = 1 / z with z the camera-space depth of `v` (the z
    the projection divides by), float32 [T,3,3].  `uv`: [T,3,2] or [T,3,3] (a third component is ignored)."""
    v = np.asarray(v, F32)
    uv = TX._uv_triples(uv)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        w = F32(1) / v[..., 2]
        return np.ascontiguousarray(np.stack([uv[..., 0] * w, uv[..., 1] * w, w], axis=-1), dtype=F32)


def pixel_uv(colour, perspective):
    """(u, v) of drawn pixels from their interpolated colour slots [..., 3]: (c0, c1), or with perspective (c0 / c2, c1 / c2)."""
    c = np.asarray(colour, F32)
    if not perspective:
        return c[..., 0].copy(), c[..., 1].copy()
    with np.errstate(divide="ignore", invalid="ignore"):
        return c[..., 0] / c[..., 2], c[..., 1] / c[..., 2]


def bilinear_texels(u, v, texture):
    """CRB_TEX_BILINEAR (DESIGN 2) in NumPy float32: float BGR [N,3] for coordinates u, v [N] of a uint8 [th,tw,3] texture."""
    tex = TX._check_texture(texture)
    th, tw = tex.shape[:2]
    u, v = np.asarray(u, F32).ravel(), np.asarray(v, F32).ravel()
    with np.errstate(invalid="ignore", over="ignore"):
        sx = u * F32(tw) - F32(0.5)
        sy = (F32(1) - v) * F32(th) - F32(0.5)
    sx = np.fmin(np.fmax(sx, F32(-1)), F32(tw))     # fmax: NaN -> -1
    sy = np.fmin(np.fmax(sy, F32(-1)), F32(th))
    x0, y0 = np.floor(sx), np.floor(sy)
    fx, fy = sx - x0, sy - y0                      # (exact unless -1 < s < 0: rounded there, as on the GPU)
    ix, iy = x0.astype(np.int64), y0.astype(np.int64)
    c0, c1 = np.clip(ix, 0, tw - 1), np.clip(ix + 1, 0, tw - 1)
    r0, r1 = np.clip(iy, 0, th - 1), np.clip(iy + 1, 0, th - 1)
    gx, gy = (F32(1) - fx)[:, None], (F32(1) - fy)[:, None]
    fx, fy = fx[:, None], fy[:, None]
    t = tex.astype(F32)
    top = t[r0, c0] * gx + t[r0, c1] * fx
    bot = t[r1, c0] * gx + t[r1, c1] * fx
    return top * gy + bot * fy


def render_textured(filler, v, uv, n, texture, perspective=False, filter="nearest"):
    """Composites the textured render of [T,3,3] v / n with texture coordinates `uv` into an OracleFiller's buffers, sampled
    with `filter` from affine or (perspective=True) perspective-correct coordinates."""
    if filter not in FILTERS:
        raise ValueError(f"filter must be one of {FILTERS}, got {filter!r}")
    if not perspective and filter == "nearest":
        return TX.render_textured(filler, v, uv, n, texture)
    tex = TX._check_texture(texture)
    slots = perspective_slots(v, uv) if perspective else TX._uv_triples(uv)
    scratch = O.OracleFiller(filler.h, filler.w, n_threads=filler.n_threads)
    scratch.proj_mat = filler.proj_mat
    scratch.z_buffer[...] = filler.z_buffer
    filler.render_arrays(v, slots, n)
    scratch.render_arrays(v, np.full(np.shape(v), np.nan, np.float32), n)
    drawn = np.isnan(scratch.color_buffer[..., 0])
    c = filler.color_buffer
    u_, v_ = pixel_uv(c[drawn], perspective)
    if filter == "bilinear":
        c[drawn] = bilinear_texels(u_, v_, tex)
    else:
        c[drawn] = I.vertex_colors(np.ascontiguousarray(np.stack([u_, v_], axis=1)), tex)


class TexturedOracleFiller(TX.TexturedOracleFiller):
    """texture_oracle.TexturedOracleFiller whose render_arrays also takes `perspective=` and `filter=`."""

    def render_arrays(self, v, c, n, texture=None, perspective=False, filter="nearest"):
        if texture is None:
            if perspective or filter != "nearest":
                raise ValueError("perspective / filter need a texture")
            return O.OracleFiller.render_arrays(self, v, c, n)
        return render_textured(self, v, c, n, texture, perspective=perspective, filter=filter)
