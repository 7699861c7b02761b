"""CPU oracle of scenes in batched views (crb_render_scene_views, render_views(objects=...); DESIGN 2) -- an extension of this
project.

TEST INFRASTRUCTURE ONLY.  Composed of pinned pieces, nothing new but the choice of transform per triangle:

  1. camera_space(): for each object present in the view, views.transform_arrays_host with that object's transform applied to
     its triangles; the triangles stay in base-mesh order, hidden ones (pad neither +0 nor -0, NaN included) and those whose
     object lies outside [0, K) are dropped (dropping keeps the relative order of the others, which is all the tie rule reads),
     and `kept` lists the base-mesh index of every triangle that stays;
  2. the camera-space triangles are rendered by the pinned oracles exactly as one view of crb_render_views: oracle_render
     (ids_oracle.IdsOracleFiller, which also gives tri_id and bary), the texture oracles, ssaa_oracle, and clip_oracle for
     CRB_CLIP_NEAR;
  3. tri_id is mapped through `kept`, as clip_oracle.clipped_ids maps pieces to their parents.

tests/test_scene_oracle.py checks camera_space() against a scalar per-triangle restatement.
"""
import numpy as np

from oracle import clip_oracle as CL
from oracle import ids_oracle as ID
from oracle import oracle as O
from oracle import texture_mip_oracle as MIP

F32 = np.float32


def shown(tri_obj, views_v):
    """bool [T]: triangle t draws in the view whose transforms are views_v [K,16] -- tri_obj[t] in [0, K) and that object's
    pad is +0 or -0."""
    tri_obj = np.asarray(tri_obj, np.int64)
    views_v = np.asarray(views_v, F32).reshape(-1, 16)
    K = len(views_v)
    in_range = (tri_obj >= 0) & (tri_obj < K)
    visible = views_v[:, 15] == 0                       # NaN compares unequal: hidden
    return in_range & visible[np.clip(tri_obj, 0, K - 1)]


def camera_space(v, c, n, tri_obj, views_v):
    """One view of a scene: (cv, cc, cn, kept), the [P,3,3] camera-space arrays of the triangles that draw, in base-mesh
    order, and kept [P] int64, their base-mesh indices.  views_v: the view's [K,16] transforms."""
    v, c, n = (np.asarray(a, F32).reshape(-1, 3, 3) for a in (v, c, n))
    tri_obj = np.asarray(tri_obj, np.int64)
    views_v = np.asarray(views_v, F32).reshape(-1, 16)
    kept = np.flatnonzero(shown(tri_obj, views_v))
    cv, cn = v[kept].copy(), n[kept].copy()
    obj = tri_obj[kept]
    for k in np.unique(obj):
        sel = obj == k
        cv[sel], cn[sel] = _transform(views_v[k], v[kept[sel]], n[kept[sel]])
    return cv, np.ascontiguousarray(c[kept]), cn, kept


def _transform(view, v, n):
    from cython3dmodelrenderer_b200 import views as VW
    return VW.transform_arrays_host(view, v, n)


def _map(ids, kept):
    return np.where(ids >= 0, kept[np.maximum(ids, 0)] if len(kept) else 0, -1)


def render(h, w, v, c, n, tri_obj, views_v, fov=90.0, z_near=0.1, near_clip=False, filler=None, **render_kw):
    """Fresh frame of one view of a scene: (oracle filler, tri_id [h,w] int64, bary [h,w,3] float32 or None).  `filler`: a fresh
    oracle filler to render into (e.g. a textured one, with its render_arrays keywords in `render_kw`); bary is given for the
    default filler without near_clip only (a clipped piece's barycentrics are not its triangle's)."""
    cv, cc, cn, kept = camera_space(v, c, n, tri_obj, views_v)
    if near_clip:
        pv, pc, pn, parent = CL.clip(cv, cc, cn, z_near)
        o = O.OracleFiller(h, w, fov=fov, z_near=z_near) if filler is None else filler
        o.render_arrays(pv, pc, pn, **render_kw)
        return o, _map(CL.clipped_ids(o, pv, pn, parent), kept), None
    if filler is None:
        o = ID.IdsOracleFiller(h, w, fov=fov, z_near=z_near)
        o.render_arrays(cv, cc, cn)
        return o, _map(o.tri_id, kept), o.bary
    o = filler
    o.render_arrays(cv, cc, cn, **render_kw)
    ids = MIP.winner_ids(o.h, o.w, o.proj_mat.ravel(), cv, cn, o.z_buffer) if len(kept) else np.full((o.h, o.w), -1, np.int64)
    return o, _map(ids, kept), None


def render_resolved(h, w, s, v, c, n, tri_obj, views_v, fov=90.0, light=None, **tex):
    """uint8 [h, w, 3]: the supersampled image (ssaa_oracle) of one view of a scene."""
    from oracle import ssaa_oracle as SS
    cv, cc, cn, _ = camera_space(v, c, n, tri_obj, views_v)
    return SS.render_resolved(h, w, s, cv, cc, cn, fov=fov, light=light, **tex)
