"""Cost of scenes in batched views (crb_render_scene_views, render_views(objects=...)): step time, k_raster time and images/s of
three ways to render the same batch, alternated in one process.  Prints one JSON line (GPU name, power limit and max SM clock
read in the same run).

Workload: a room of generated quads (a floor and three walls) with the T-Rex, the bunny and the basketball in it
(tests/golden); each model turns about its own vertical axis at its own rate while the camera orbits the room.  1024^2, fov 45,
128 views per step, z / colour / normals out (bench.py's headline outputs).
  scene    (a) the scene call: one render_views(objects=...) of the 128 views, a transform per (view, object).
  static   (b) a lower bound: the same concatenated mesh with the camera transform alone (render_views without objects).  Its
           images differ (nothing turns); the difference to (a) isolates the front-end cost of per-triangle transforms.
  loop     (c) what a caller without scenes must do: per view, crb_transform_view per object into one camera-space buffer,
           then a single-view crb_render_views with views = NULL into that view's slab -- V x (K + 1) calls.  Its outputs must
           equal (a) bit for bit (checked, reported as `loop_equals_scene`).

Each round times every arm back to back (the order rotates between rounds); the report gives the median and the spread
(min, max) over the rounds.  `k_raster_ms` is the tile rasterizer's device time per step (crb_profile: CUDA events around each
launch), `step_ms` the whole step (CUDA events, synchronised).

    python tools/scene_bench.py [--rounds 7] [--steps 5] [--out profiles/scene_b200.json]
"""
import argparse
import ctypes
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from texture_bench import gpu_info, rounds_of, summary, timed  # noqa: E402

ARMS = ("scene", "static", "loop")
RES, FOV = 1024, 45.0
F32 = np.float32


def grid(nx, nz, size, rng):
    """2*nx*nz triangles in the plane y = 0 about the origin, normals +y, random colours"""
    xs, zs = np.linspace(-size / 2, size / 2, nx + 1), np.linspace(-size / 2, size / 2, nz + 1)
    tris = [t for i in range(nx) for j in range(nz) for t in
            (((xs[i], 0, zs[j]), (xs[i + 1], 0, zs[j + 1]), (xs[i + 1], 0, zs[j])),
             ((xs[i], 0, zs[j]), (xs[i], 0, zs[j + 1]), (xs[i + 1], 0, zs[j + 1])))]
    v = np.array(tris, F32)
    n = np.zeros_like(v)
    n[..., 1] = 1.0
    return v, (rng.random(v.shape) * 255).astype(F32), n


def room_and_models():
    """(meshes at their places in the room, centre of each): floor, three walls facing inwards, T-Rex, bunny, basketball"""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from conftest import load_indexed
    from cython3dmodelrenderer_b200 import views as VW
    rng = np.random.default_rng(0)
    rx = np.array([[1, 0, 0], [0, 0, -1], [0, 1, 0]], F32)                # +y normal -> +z: the wall at z = -2 faces in
    meshes, centres = [], []

    def place(v, c, n, R, t):
        R = np.asarray(R, F32)
        meshes.append(((v @ R.T + np.asarray(t, F32)).astype(F32), c, (n @ R.T).astype(F32)))
        centres.append(np.asarray(t, F32))
    place(*grid(32, 32, 4.0, rng), np.eye(3), (0.0, -0.4, 0.0))
    for ang, t in ((0.0, (0.0, 0.6, -2.0)), (np.pi / 2, (-2.0, 0.6, 0.0)), (-np.pi / 2, (2.0, 0.6, 0.0))):
        place(*grid(16, 8, 4.0, rng), VW.rot_y(ang) @ rx, t)
    for name, scale, t in (("trex", 1.0, (0.0, 0.2, 0.0)), ("bunny", 0.8, (0.9, 0.1, 0.5)), ("basketball", 0.4, (-0.9, 0.0, -0.4))):
        m = load_indexed(name)
        v = m._vertices_by_triangles
        ctr = (v.reshape(-1, 3).min(0) + v.reshape(-1, 3).max(0)) / 2
        place(((v - ctr) * F32(scale)).astype(F32), m._colors_by_triangles, m._normals_by_triangles, np.eye(3), t)
    return meshes, centres


RATES = (0.0, 0.0, 0.0, 0.0, 1.0, -2.0, 3.0)     # turns per orbit of each object about its own vertical axis (the room stands)


def batch(V, centres):
    """(camera [V,16], per-object transforms [V,K,16]): the camera orbits the room looking down; object k turns about its
    centre by RATES[k] turns per orbit"""
    from cython3dmodelrenderer_b200 import views as VW
    pitch = -0.4
    rx = np.array([[1, 0, 0], [0, np.cos(pitch), -np.sin(pitch)], [0, np.sin(pitch), np.cos(pitch)]])
    th = 2 * np.pi * np.arange(V) / V
    cams = np.stack([VW.view_matrix(rx @ VW.rot_y(t), p=(0.0, 0.0, 0.0), q=(0.0, 0.0, 3.2)) for t in th]).astype(F32)
    poses = np.stack([np.stack([VW.view_matrix(VW.rot_y(r * t), p=c, q=c) for r, c in zip(RATES, centres)]) for t in th])
    return cams, VW.scene_views(cams, poses)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--views", type=int, default=128)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("scene_bench needs a CUDA device")
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller, _lib, views as VW
    dev = torch.device("cuda", 0)
    result = {"tool": "tools/scene_bench.py", **gpu_info(torch), "rounds": args.rounds, "steps": args.steps, "arms": list(ARMS)}
    meshes, centres = room_and_models()
    v, c, n, tri_obj = VW.concat_meshes(meshes)
    V, K, T = args.views, len(meshes), len(v)
    cams, scene_views = batch(V, centres)
    dv, dc, dn, dobj = (torch.from_numpy(a).to(dev) for a in (v, c, n, tri_obj))
    dcams, dviews = torch.from_numpy(cams).to(dev), torch.from_numpy(scene_views).to(dev)
    runs = np.flatnonzero(np.diff(tri_obj)) + 1
    bounds = list(zip(np.concatenate([[0], runs]).tolist(), np.concatenate([runs, [T]]).tolist()))
    result.update({"res": RES, "fov": FOV, "views_per_step": V, "objects": K, "triangles": T,
                   "object_triangles": [b - a for a, b in bounds]})

    fills = {arm: AdvancedPixelBufferFiller(RES, RES, fov=FOV, device=0) for arm in ARMS}
    outs = {arm: tuple(torch.empty(s, dtype=torch.float32, device=dev) for s in ((V, RES, RES), (V, RES, RES, 3), (V, RES, RES, 3)))
            for arm in ARMS}
    cv, cn = torch.empty_like(dv), torch.empty_like(dn)
    L = fills["loop"]._L

    def scene_step(check=False):
        z, col, nor = outs["scene"]
        fills["scene"].render_views(dv, dc, dn, dviews, z_out=z, color_out=col, normals_out=nor, chunk=V, objects=dobj,
                                    check_status=check)

    def static_step(check=False):
        z, col, nor = outs["static"]
        fills["static"].render_views(dv, dc, dn, dcams, z_out=z, color_out=col, normals_out=nor, chunk=V, check_status=check)

    def loop_step(check=False):
        f = fills["loop"]
        z, col, nor = outs["loop"]
        H, st = f._handle, f._stream()
        for k in range(V):
            for a, b in bounds:
                _lib.check(L.crb_transform_view(H, dv[a:b].data_ptr(), dn[a:b].data_ptr(), b - a,
                                                dviews[k, int(tri_obj[a])].data_ptr(), cv[a:b].data_ptr(), cn[a:b].data_ptr(), st))
            _lib.check(L.crb_render_views(H, cv.data_ptr(), dc.data_ptr(), cn.data_ptr(), T, None, 1, z[k].data_ptr(),
                                          col[k].data_ptr(), nor[k].data_ptr(), None, 0, None, st))
        if check:
            need, cap = ctypes.c_int64(), ctypes.c_int64()
            _lib.check(L.crb_status(H, ctypes.byref(need), ctypes.byref(cap), st))

    steps = {"scene": scene_step, "static": static_step, "loop": loop_step}
    fills["loop"]._ensure_workspace(T, 1)
    for arm in ARMS:             # workspace and status checked once (the pair list fits), then warm-up
        steps[arm](check=True)
        for _ in range(2):
            steps[arm]()
    torch.cuda.synchronize()
    result["loop_equals_scene"] = all(torch.equal(a.view(torch.int32), b.view(torch.int32)) for a, b in zip(outs["scene"], outs["loop"]))
    result["covered_pixels"] = {arm: int((outs[arm][0] < 1e5).sum()) for arm in ARMS}

    def run(arm):
        step_ms, k_ms, _ = timed(torch, fills[arm], steps[arm], args.steps)
        return V / (step_ms / 1e3), step_ms, k_ms
    rows = rounds_of(list(ARMS), args.rounds, run)
    rep = {arm: {("images_per_s" if k == "fps" else k): summary(x) for k, x in rows[arm].items()} for arm in ARMS}
    med = {arm: {k: float(np.median(x)) for k, x in rows[arm].items()} for arm in ARMS}
    rep["scene"]["over_static_step"] = med["scene"]["step_ms"] / med["static"]["step_ms"]
    rep["scene"]["over_static_k_raster"] = med["scene"]["k_raster_ms"] / med["static"]["k_raster_ms"]
    rep["scene"]["speedup_over_loop"] = med["loop"]["step_ms"] / med["scene"]["step_ms"]
    result.update(rep)
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
