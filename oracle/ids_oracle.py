"""CPU oracle of the id outputs (crb_bind_id_buffers, crb_render_views_ids; DESIGN 2) -- an extension of this project.

TEST INFRASTRUCTURE ONLY.  Composed of pinned pieces, nothing new:

  1. oracle_render (OracleFiller.render_arrays) draws the call and leaves its z buffer;
  2. texture_mip_oracle.winner_ids gives each pixel's last writer of the call under the sequential z-test (-1: the call wrote
     nothing there);
  3. texture_mip_oracle._bary restates mu:5-34 for that triangle at that pixel.

Across calls the buffers keep the previous ids and barycentrics where a call writes nothing, like z, colour and normals.
tests/test_ids_oracle.py checks the composition against oracle_render's buffers.
"""
import numpy as np

from oracle import oracle as O
from oracle import texture_mip_oracle as MIP

F32 = np.float32


class IdsOracleFiller(O.OracleFiller):
    """OracleFiller that also keeps tri_id [h,w] int64 and bary [h,w,3] float32 (fresh: -1 and +0)."""

    def __init__(self, h, w, fov=90.0, z_near=0.1, z_far=1000.0, n_threads=1):
        super().__init__(h, w, fov, z_near, z_far, n_threads)
        self.tri_id = np.full((self.h, self.w), -1, np.int64)
        self.bary = np.zeros((self.h, self.w, 3), F32)

    def render_arrays(self, v, c, n, base=0):
        super().render_arrays(v, c, n)
        ids = MIP.winner_ids(self.h, self.w, self.proj_mat.ravel(), v, n, self.z_buffer)
        ys, xs = np.nonzero(ids >= 0)
        t = ids[ys, xs]
        scr = O.project(self.h, self.w, self.proj_mat.ravel(), v)
        self.tri_id[ys, xs] = base + t
        self.bary[ys, xs] = MIP._bary(scr[t], xs, ys)
        return ids

    def render_model(self, model, base=0):
        return self.render_arrays(model._vertices_by_triangles.copy(), model._colors_by_triangles.copy(),
                                  model._normals_by_triangles.copy(), base=base)


def restate(attr, tri_id, bary, base=0):
    """Per-corner attribute `attr` [T,3,k] of one call (projected corners' z: O.project(...)[..., 2:3]; normals; colours)
    interpolated at the pixels with base <= tri_id < base + T, from their barycentrics: (a0*b1 + a1*b2) + a2*b3 in float32
    (shade_fragment's left-associated sums); NaN elsewhere."""
    tri_id = np.asarray(tri_id)
    ys, xs = np.nonzero((tri_id >= base) & (tri_id < base + len(attr)))
    t = tri_id[ys, xs] - base
    b = np.asarray(bary, F32)[ys, xs]
    a = np.asarray(attr, F32)[t]
    out = np.full(tri_id.shape + (a.shape[2],), np.nan, F32)
    with np.errstate(all="ignore"):
        out[ys, xs] = (a[:, 0] * b[:, 0:1] + a[:, 1] * b[:, 1:2]) + a[:, 2] * b[:, 2:3]
    return out
