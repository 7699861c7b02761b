"""Synthetic workloads for the benchmark configs that have no asset in the reference tree (SURVEY.md section 8d).

uv_sphere: config C4 -- a UV sphere built directly as the three [T,3,3] float32 arrays render_model consumes (going through
the reference's Model.__init__ would run its O(T) Python normal loop, crender/cy/data_structures/model.py:174-188).
n_lat latitude bands, pole caps are single-triangle fans: T = 2 * n_lon * (n_lat - 1).  Vertex normals are the outward
unit radials, colours 127.5 * (n + 1) per channel.  NumPy only (works without a GPU)."""
import numpy as np


class ArrayModel:
    """Duck-typed model: render_model reads exactly these three attributes (pyx:94-96)."""

    def __init__(self, v, c, n):
        self._vertices_by_triangles = v
        self._colors_by_triangles = c
        self._normals_by_triangles = n


def uv_sphere(n_lon=3200, n_lat=1564, center=(0.0, 0.0, 1.5), radius=0.5):
    lon = (np.arange(n_lon + 1, dtype=np.float64) % n_lon) * (2.0 * np.pi / n_lon)
    lat = np.linspace(0.0, np.pi, n_lat + 1)          # 0 = north pole ... pi = south pole
    sl, cl = np.sin(lat)[:, None], np.cos(lat)[:, None]
    # unit normals of the (n_lat+1) x (n_lon+1) vertex grid
    g = np.stack([sl * np.cos(lon)[None, :], np.broadcast_to(cl, (n_lat + 1, n_lon + 1)), sl * np.sin(lon)[None, :]], axis=-1)
    g = g.astype(np.float32)
    a, b = g[:-1, :-1], g[:-1, 1:]     # upper ring: j, j+1
    c, d = g[1:, :-1], g[1:, 1:]       # lower ring: j, j+1
    tris = []
    tris.append(np.stack([a[0], c[0], d[0]], axis=1))                       # north cap: pole, ring1[j], ring1[j+1]
    if n_lat > 2:
        mid_a, mid_b, mid_c, mid_d = a[1:-1], b[1:-1], c[1:-1], d[1:-1]
        t1 = np.stack([mid_a, mid_c, mid_d], axis=2).reshape(-1, 3, 3)
        t2 = np.stack([mid_a, mid_d, mid_b], axis=2).reshape(-1, 3, 3)
        tris += [t1, t2]
    tris.append(np.stack([a[-1], c[-1], b[-1]], axis=1))                     # south cap: ring[j], pole, ring[j+1]
    n = np.ascontiguousarray(np.concatenate(tris, axis=0), dtype=np.float32)
    assert n.shape[0] == 2 * n_lon * (n_lat - 1)
    v = (n * np.float32(radius) + np.asarray(center, dtype=np.float32)).astype(np.float32)
    col = (np.float32(127.5) * (n + np.float32(1.0))).astype(np.float32)
    return ArrayModel(v, col, n)


def spherical_uvs(v, center=None):
    """Texture coordinates by triangle, float32 [T,3,2], from a spherical projection of the corners `v` ([T,3,3]) about
    `center` (default: the mean corner): u = 0.5 + atan2(z, x) / 2pi (longitude), v = 0.5 + asin(y / r) / pi (latitude).
    For uv_sphere these are its latitude-longitude coordinates.  For per-pixel texturing (`texture=` of the filler's
    render_arrays / render_views) of meshes that come without texture coordinates."""
    v = np.asarray(v, dtype=np.float64)
    c = v.reshape(-1, 3).mean(axis=0) if center is None else np.asarray(center, dtype=np.float64)
    d = v - c
    r = np.linalg.norm(d, axis=-1)
    u = 0.5 + np.arctan2(d[..., 2], d[..., 0]) / (2.0 * np.pi)
    w = 0.5 + np.arcsin(np.clip(d[..., 1] / np.where(r > 0, r, 1.0), -1.0, 1.0)) / np.pi
    return np.ascontiguousarray(np.stack([u, w], axis=-1), dtype=np.float32)
