"""CPU oracle of per-pixel texturing (CRB_TEXTURE), an extension of this project -- not a restatement of the reference.

TEST INFRASTRUCTURE ONLY, like the rest of oracle/.  The reference textures vertices only (model.py:147-150: one texel per
texture-coordinate vertex, blended by the rasterizer).  This module DEFINES the per-pixel mode (DESIGN 2) by composing two
pinned pieces, unchanged:

  1. oracle_render (crender_oracle.c, pinned against the reference build by tests/test_oracle_pinning.py), run with the
     texture coordinates (u, v, w) in the colour slots.  Visibility does not depend on the colours, so it draws exactly
     the per-vertex frame's fragments, with z and normals bit for bit the per-vertex ones, and leaves the winning
     fragment's interpolated (u, v, w) = ((c0*b1 + c1*b2) + c2*b3, ...) in the colour buffer;
  2. ingest_vertex_colors (ingest_oracle.c, pinned by tests/test_ingest_oracle.py), the texel rule of model.py:147-150,
     applied to that (u, v) at every pixel this render drew.

The pixels a render draws are found by a second oracle_render of the same triangles with NaN colours into a scratch copy
of the depth buffer (colour and normals cleared): its colour is NaN exactly where a fragment of this render won.
tests/test_texture_oracle.py checks the composition against the definition.
"""
import numpy as np

from oracle import ingest as I
from oracle import oracle as O


def _check_texture(texture):
    tex = np.ascontiguousarray(texture)
    if tex.dtype != np.uint8 or tex.ndim != 3 or tex.shape[2] != 3 or tex.shape[0] < 1 or tex.shape[1] < 1:
        raise ValueError("texture must be a uint8 [h,w,3] image")
    return tex


def _uv_triples(uv):
    """[T,3,2] or [T,3,3] float32 texture coordinates -> [T,3,3] (a third component is ignored by the rule)."""
    uv = np.asarray(uv)
    if uv.dtype == np.float32 and uv.ndim == 3 and uv.shape[1:] == (3, 2):
        uv = np.concatenate([uv, np.zeros(uv.shape[:2] + (1,), np.float32)], axis=2)
    return uv


def render_textured(filler, v, uv, n, texture):
    """Composites the textured render of [T,3,3] v / n with texture coordinates `uv` into an OracleFiller's buffers."""
    tex = _check_texture(texture)
    uv = _uv_triples(uv)
    scratch = O.OracleFiller(filler.h, filler.w, n_threads=filler.n_threads)
    scratch.proj_mat = filler.proj_mat
    scratch.z_buffer[...] = filler.z_buffer
    filler.render_arrays(v, uv, n)
    scratch.render_arrays(v, np.full(np.shape(v), np.nan, np.float32), n)
    drawn = np.isnan(scratch.color_buffer[..., 0])
    c = filler.color_buffer
    c[drawn] = I.vertex_colors(np.ascontiguousarray(c[drawn][:, :2]), tex)


class TexturedOracleFiller(O.OracleFiller):
    """OracleFiller whose render_arrays also takes `texture=` (uint8 [th,tw,3], BGR): `c` then holds texture coordinates
    by triangle, [T,3,3] (third component ignored) or [T,3,2]."""

    def render_arrays(self, v, c, n, texture=None):
        if texture is None:
            return super().render_arrays(v, c, n)
        return render_textured(self, v, c, n, texture)
