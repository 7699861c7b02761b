"""Cost of the id outputs (crb_bind_id_buffers, crb_render_views_ids): frames/s and k_raster time with them off, with the
triangle ids, and with the triangle ids and barycentrics, alternated in one process.  Prints one JSON line (GPU name, power
limit and max SM clock read in the same run).

  trex_1024_orbit  the headline workload of bench.py: T-Rex (tests/golden/trex_fit.npz) at 1024^2, batches of 128 orbit views
                   rendered by render_views into float32 z / colour / normals slabs, plus the int32 tri_id slab ("ids") and
                   the float32 [.,3] bary slab ("ids_bary").
  trex_256_orbit   the same at 256^2.
  sphere_8192      the 10 M-triangle synthetic.uv_sphere, one fresh frame at 8192^2 (render_arrays, device-resident inputs,
                   fused clear) into a filler built with triangle_ids / barycentrics.

Each round times every mode back to back (the order rotates between rounds); the report gives the median and the spread
(min, max) over the rounds, and each mode's medians over those of "off".  `k_raster_ms` is the tile rasterizer's device time
per step (crb_profile: CUDA events around each launch), `step_ms` the whole step (CUDA events).

    python tools/ids_bench.py [--rounds 5] [--steps 20] [--out profiles/ids_b200.json]
"""
import argparse
import gc
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from texture_bench import gpu_info, rounds_of, summary, timed  # noqa: E402

MODES = {"off": (False, False), "ids": (True, False), "ids_bary": (True, True)}


def report(rows):
    out = {mode: {k: summary(v) for k, v in rows[mode].items()} for mode in rows}
    for mode in rows:
        if mode != "off":
            out[mode]["over_off_k_raster"] = float(np.median(rows[mode]["k_raster_ms"]) / np.median(rows["off"]["k_raster_ms"]))
            out[mode]["over_off_fps"] = float(np.median(rows[mode]["fps"]) / np.median(rows["off"]["fps"]))
    return out


def trex_workload(torch, dev, AdvancedPixelBufferFiller, VW, m, args, RES, result):
    modes = list(MODES)
    T, V = int(m._vertices_by_triangles.shape[0]), args.views
    dv, dc, dn = (torch.from_numpy(a).to(dev) for a in (m._vertices_by_triangles, m._colors_by_triangles, m._normals_by_triangles))
    dviews = torch.from_numpy(VW.orbit_views(V, count=V)).to(dev)
    z = torch.empty((V, RES, RES), dtype=torch.float32, device=dev)
    col = torch.empty((V, RES, RES, 3), dtype=torch.float32, device=dev)
    nrm = torch.empty((V, RES, RES, 3), dtype=torch.float32, device=dev)
    tri = torch.empty((V, RES, RES), dtype=torch.int32, device=dev)
    bary = torch.empty((V, RES, RES, 3), dtype=torch.float32, device=dev)
    fill = {mode: AdvancedPixelBufferFiller(RES, RES, fov=45.0, device=0) for mode in modes}

    def trex_step(mode):
        f, (want_ids, want_bary) = fill[mode], MODES[mode]
        kw = {"triangle_id_out": tri if want_ids else None, "barycentrics_out": bary if want_bary else None}
        return lambda: f.render_views(dv, dc, dn, dviews, z_out=z, color_out=col, normals_out=nrm, chunk=V, check_status=False,
                                      **kw)
    for mode in modes:     # workspace, status check, warm-up
        f, (want_ids, want_bary) = fill[mode], MODES[mode]
        f.render_views(dv, dc, dn, dviews, z_out=z, color_out=col, normals_out=nrm, chunk=V,
                       triangle_id_out=tri if want_ids else None, barycentrics_out=bary if want_bary else None)
        for _ in range(3):
            trex_step(mode)()

    def trex_run(mode):
        step_ms, k_ms, _ = timed(torch, fill[mode], trex_step(mode), args.steps)
        return V / (step_ms / 1e3), step_ms, k_ms
    rows = rounds_of(modes, args.rounds, trex_run)
    result["workloads"][f"trex_{RES}_orbit"] = {"triangles": T, "views_per_step": V, "resolution": RES, "steps": args.steps,
                                                **report(rows)}
    del z, col, nrm, tri, bary, fill


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20, help="timed steps per mode and round (T-Rex); the sphere runs steps/4 + 1")
    ap.add_argument("--views", type=int, default=128)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("ids_bench needs a CUDA device")
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller, synthetic, views as VW
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from conftest import load_indexed
    dev = torch.device("cuda", 0)
    result = {"tool": "tools/ids_bench.py", **gpu_info(torch), "rounds": args.rounds, "modes": list(MODES), "workloads": {}}

    m = load_indexed("trex")
    for RES in (1024, 256):
        trex_workload(torch, dev, AdvancedPixelBufferFiller, VW, m, args, RES, result)
    gc.collect()
    torch.cuda.empty_cache()

    s = synthetic.uv_sphere(3200, 1564)
    T = int(s._vertices_by_triangles.shape[0])
    sv, sc, sn = (torch.from_numpy(a).to(dev) for a in (s._vertices_by_triangles, s._colors_by_triangles, s._normals_by_triangles))
    del s
    RES, ssteps = 8192, args.steps // 4 + 1
    fills = {mode: AdvancedPixelBufferFiller(RES, RES, fov=45.0, device=0, triangle_ids=MODES[mode][0],
                                             barycentrics=MODES[mode][1]) for mode in MODES}

    def sphere_step(mode):
        fs = fills[mode]

        def step():
            fs.clear()
            fs.render_arrays(sv, sc, sn, check_status=False)
        return step
    for mode, fs in fills.items():
        fs.clear()
        fs.render_arrays(sv, sc, sn)
        fs.get_z_buffer()         # status checked (the pair list fits)
        for _ in range(2):
            sphere_step(mode)()

    def sphere_run(mode):
        step_ms, k_ms, _ = timed(torch, fills[mode], sphere_step(mode), ssteps)
        return 1e3 / step_ms, step_ms, k_ms
    rows = rounds_of(list(MODES), args.rounds, sphere_run)
    result["workloads"]["sphere_8192"] = {"triangles": T, "resolution": RES, "steps": ssteps, **report(rows)}
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
