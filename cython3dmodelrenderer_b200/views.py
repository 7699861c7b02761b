"""Camera views for batched rendering (config C5).

The reference has no camera stage: a new view is made by mutating the model on the host
(crender/cy/data_structures/model.py:238-256, `rotate` = vertices @ R.T followed by an O(T) Python normal
recomputation).  Here a view is 16 floats {R (9, row-major), p (3), q (3), pad} applied on the GPU inside the
setup and shading kernels:   v' = R (v - p) + q,   n' = R n,
each component evaluated as ((r0*d0 + r1*d1) + r2*d2) + q in float32 with one rounding per operation.
`transform_arrays_host` restates exactly that arithmetic in NumPy so the same camera-space arrays can be handed
to the reference / the oracle in parity tests (SURVEY.md section 8d, row C5).
"""
import numpy as np


def view_matrix(R=None, p=(0.0, 0.0, 0.0), q=None):
    """16 float32: R row-major, pivot p, translation q (defaults to p: rotate about p)."""
    M = np.zeros(16, dtype=np.float32)
    M[:9] = (np.eye(3) if R is None else np.asarray(R, dtype=np.float64)).astype(np.float32).ravel()
    M[9:12] = np.asarray(p, dtype=np.float32)
    M[12:15] = np.asarray(p if q is None else q, dtype=np.float32)
    return M


def rot_y(theta):
    """Rotation about y in the reference's convention (model.py:229-236,246-247: mat_rot_y[::2, ::2] = [[c,s],[-s,c]])."""
    c, s = np.cos(theta), np.sin(theta)
    return np.array([[c, 0.0, s], [0.0, 1.0, 0.0], [-s, 0.0, c]])


def orbit_views(n_total, first=0, count=None, center=(0.0, 0.0, 1.0), stride=1):
    """Views first, first+stride, ... (count of them) of an n_total-view orbit about the y axis through `center`
    (theta = 2*pi*k/n_total).  stride = world size, first = rank gives every rank an evenly spread sample of the orbit
    (view k -> GPU k mod N, SURVEY 8e): frames of different view angles cost differently, contiguous arcs would not balance."""
    count = (n_total - first + stride - 1) // stride if count is None else count
    out = np.zeros((count, 16), dtype=np.float32)
    for i in range(count):
        out[i] = view_matrix(rot_y(2.0 * np.pi * (first + i * stride) / n_total), p=center)
    return out


def transform_arrays_host(view, v, n):
    """NumPy float32 restatement of the GPU view transform: returns (v', n') for [T,3,3] float32 inputs."""
    M = np.asarray(view, dtype=np.float32).ravel()
    v = np.asarray(v, dtype=np.float32)
    n = np.asarray(n, dtype=np.float32)
    d = [v[..., k] - M[9 + k] for k in range(3)]
    vo = np.empty_like(v)
    no = np.empty_like(n)
    for r in range(3):
        vo[..., r] = ((M[3 * r] * d[0] + M[3 * r + 1] * d[1]) + M[3 * r + 2] * d[2]) + M[12 + r]
        no[..., r] = (M[3 * r] * n[..., 0] + M[3 * r + 1] * n[..., 1]) + M[3 * r + 2] * n[..., 2]
    return vo, no


def scene_views(camera, poses):
    """Per-object transforms of a scene (render_views(objects=...)): [V,K,16] float32, entry [v,k] = camera[v] after pose k.

    camera: [V,16] views, poses: [K,16] (the same poses in every view) or [V,K,16], both in the {R, p, q, pad} format.  A pose
    x -> Ro (x - po) + qo followed by the camera y -> Rc (y - pc) + qc is x -> Rc Ro (x - po) + (Rc (qo - pc) + qc), so the
    composition is R = Rc Ro, p = po, q = Rc (qo - pc) + qc, computed in float64 and rounded to float32 once.  The pose's pad is
    carried through: a pose with a non-zero pad hides its object in that view."""
    cam = np.asarray(camera, dtype=np.float64).reshape(-1, 16)
    V = cam.shape[0]
    pos = np.asarray(poses, dtype=np.float64)
    pos = np.broadcast_to(pos.reshape(1, -1, 16) if pos.ndim == 2 else pos, (V, pos.shape[-2], 16))
    Rc = cam[:, None, :9].reshape(V, 1, 3, 3)
    Ro = pos[..., :9].reshape(V, -1, 3, 3)
    out = np.empty(pos.shape, np.float64)
    out[..., :9] = (Rc @ Ro).reshape(V, -1, 9)
    out[..., 9:12] = pos[..., 9:12]
    out[..., 12:15] = (Rc @ (pos[..., 12:15] - cam[:, None, 9:12])[..., None])[..., 0] + cam[:, None, 12:15]
    out[..., 15] = pos[..., 15]
    return out.astype(np.float32)


def concat_meshes(meshes):
    """One base mesh of several objects: [(v, c, n), ...] of [T_k,3,3] float32 arrays -> (v, c, n, tri_obj), the arrays
    concatenated in the given order and tri_obj int32 [sum T_k], k for the triangles of mesh k."""
    if not meshes:
        raise ValueError("concat_meshes needs at least one mesh")
    v, c, n = (np.ascontiguousarray(np.concatenate([np.asarray(m[i], np.float32).reshape(-1, 3, 3) for m in meshes]))
               for i in range(3))
    tri_obj = np.concatenate([np.full(len(np.asarray(m[0]).reshape(-1, 9)), k, np.int32) for k, m in enumerate(meshes)])
    return v, c, n, tri_obj
