"""CPU oracle of near-plane clipping (CRB_CLIP_NEAR, AdvancedPixelBufferFiller(near_clip=True); DESIGN 2) -- an extension of
this project.

TEST INFRASTRUCTURE ONLY.  clip() is a NumPy float32 statement of the clip rule; everything else is composed of pinned pieces:

  1. camera space: the arrays as passed, or for batched views views.transform_arrays_host;
  2. clip() replaces each triangle t by its pieces (t, 0), (t, 1) in that order, absent pieces dropped (only the relative order
     of the pieces matters for the tie rule, and dropping keeps it), and returns each piece's parent;
  3. the pieces are rendered by oracle_render (OracleFiller.render_arrays) or the texture / supersampling oracles, exactly as a
     call without the bit;
  4. texture_mip_oracle.winner_ids on the pieces, mapped through the parents, gives tri_id.

tests/test_clip_oracle.py checks clip() against a scalar restatement of the rule.
"""
import numpy as np

from oracle import oracle as O
from oracle import texture_mip_oracle as MIP

F32 = np.float32


def clip(v, c, n, z_near):
    """Pieces of the [T,3,3] float32 camera-space arrays v, c, n clipped at zn = F(z_near): (pv, pc, pn, parent), the pieces'
    [P,3,3] arrays in the order (0,0), (0,1), (1,0), ... with absent ones dropped, and parent [P] int64."""
    v, c, n = (np.asarray(a, F32).reshape(-1, 3, 3) for a in (v, c, n))
    T = v.shape[0]
    zn = F32(z_near)
    A = np.concatenate([v, n, c], axis=2)                 # [T,3,9]: position, normal, colour of each corner
    with np.errstate(invalid="ignore"):
        inside = A[:, :, 2] >= zn                         # NaN: outside
    # the six candidate corners of the polygon walk, in order: for edge (a, b) corner a itself, then the crossing point
    cand = np.empty((T, 6, 9), F32)
    keep = np.zeros((T, 6), bool)
    for a in range(3):
        b = (a + 1) % 3
        cand[:, 2 * a] = A[:, a]
        keep[:, 2 * a] = inside[:, a]
        ia = inside[:, a][:, None]
        Ai, Ao = np.where(ia, A[:, a], A[:, b]), np.where(ia, A[:, b], A[:, a])   # inside end, outside end
        with np.errstate(all="ignore"):
            s = (zn - Ai[:, 2:3]) / (Ao[:, 2:3] - Ai[:, 2:3])
            x = Ai + s * (Ao - Ai)
        x[:, 2] = zn
        cand[:, 2 * a + 1] = x
        keep[:, 2 * a + 1] = inside[:, a] != inside[:, b]
    count = keep.sum(axis=1)                              # 0, 3 or 4
    order = np.argsort(~keep, axis=1, kind="stable")[:, :4]
    poly = np.take_along_axis(cand, order[:, :, None], axis=1)     # [T,4,9]; corners beyond `count` are unused
    pieces = np.stack([poly[:, [0, 1, 2]], poly[:, [0, 2, 3]]], axis=1)     # [T,2,3,9]
    present = np.stack([count >= 3, count == 4], axis=1)                  # [T,2]
    sel = pieces[present]
    parent = np.repeat(np.arange(T), 2).reshape(T, 2)[present]
    pv, pn, pc = (np.ascontiguousarray(sel[:, :, k:k + 3]) for k in (0, 3, 6))
    return pv, pc, pn, parent.astype(np.int64)


def clipped_ids(o, pv, pn, parent, base=0):
    """tri_id of one call whose pieces (pv, pn) the oracle filler `o` has just rendered: base + parent of the piece that
    wrote each pixel last, -1 where the call wrote nothing ([h,w] int64)."""
    if len(parent) == 0:
        return np.full((o.h, o.w), -1, np.int64)
    ids = MIP.winner_ids(o.h, o.w, o.proj_mat.ravel(), pv, pn, o.z_buffer)
    return np.where(ids >= 0, base + parent[np.maximum(ids, 0)], -1)


def render(h, w, v, c, n, fov=90.0, z_near=0.1, view=None, filler=None, **render_kw):
    """Fresh frame of the [T,3,3] arrays clipped at z_near, optionally through the view transform `view` (16 floats):
    (oracle filler, tri_id).  `filler`: a fresh oracle filler to render into (e.g. a textured one, with its render_arrays
    keywords in `render_kw`); its z_near must match."""
    if view is not None:
        from cython3dmodelrenderer_b200 import views as VW
        v, n = VW.transform_arrays_host(view, v, n)
    pv, pc, pn, parent = clip(v, c, n, z_near)
    o = O.OracleFiller(h, w, fov=fov, z_near=z_near) if filler is None else filler
    o.render_arrays(pv, pc, pn, **render_kw)
    return o, clipped_ids(o, pv, pn, parent)
