"""Cost of near-plane clipping (CRB_CLIP_NEAR, AdvancedPixelBufferFiller(near_clip=True)): step time and k_raster time with and
without the bit, alternated in one process.  Prints one JSON line (GPU name, power limit and max SM clock read in the same run).

Workloads (T-Rex, tests/golden/trex_fit.npz, 1024^2, fov 45, batches of 128 views, z / colour / normals out as bench.py's
headline):
  orbit    bench.py's headline orbit.  Nothing crosses z_near there, so the two arms must give identical outputs (checked, and
           reported as `outputs_identical`): the difference is the pure cost of the mode, a setup of 2T pieces and twice the
           chunks for k_fill.
  inside   cameras inside and passing through the model (look-at from points inside its bounding box, turning about y).
           Without the bit these frames are wrong (geometry behind the camera projects through, mirrored); the `off` arm
           is timed only as the reference point.

Each round times both arms back to back (the order alternates between rounds); the report gives the median and the spread
(min, max) over the rounds.  `k_raster_ms` is the tile rasterizer's device time per step (crb_profile: CUDA events around each
launch), `step_ms` the whole step (CUDA events, synchronised).

    python tools/clip_bench.py [--rounds 7] [--steps 10] [--out profiles/clip_b200.json]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from texture_bench import gpu_info, rounds_of, summary, timed  # noqa: E402

ARMS = ("off", "clip")
RES, FOV, Z_NEAR = 1024, 45.0, 0.1


def inside_views(V):
    """Cameras at points inside the T-Rex's bounding box, turning about y"""
    from cython3dmodelrenderer_b200 import views as VW
    out = []
    for k in range(V):
        th = 2 * np.pi * k / V
        p = (-0.4 + 0.3 * np.cos(th), 0.02, 1.1 + 0.3 * np.sin(th))
        out.append(VW.view_matrix(VW.rot_y(th), p=p, q=(0.0, 0.0, 0.0)))
    return np.stack(out).astype(np.float32)


def workload(torch, APBF, name, dv, dc, dn, views, args, result):
    dev = dv.device
    V = int(views.shape[0])
    fills = {arm: APBF(RES, RES, fov=FOV, z_near=Z_NEAR, device=0, near_clip=arm == "clip") for arm in ARMS}
    outs = {arm: tuple(torch.empty(s, dtype=torch.float32, device=dev) for s in ((V, RES, RES), (V, RES, RES, 3), (V, RES, RES, 3)))
            for arm in ARMS}

    def step_of(arm):
        z, c, n = outs[arm]
        return lambda: fills[arm].render_views(dv, dc, dn, views, z_out=z, color_out=c, normals_out=n, chunk=V,
                                               check_status=False)
    steps = {arm: step_of(arm) for arm in ARMS}
    for arm in ARMS:             # workspace and status checked once (the pair list fits), then warm-up
        z, c, n = outs[arm]
        fills[arm].render_views(dv, dc, dn, views, z_out=z, color_out=c, normals_out=n, chunk=V)
        for _ in range(2):
            steps[arm]()
    torch.cuda.synchronize()
    identical = all(torch.equal(a.view(torch.int32), b.view(torch.int32)) for a, b in zip(outs["off"], outs["clip"]))
    drawn = {arm: int((outs[arm][0] < 1e5).sum()) for arm in ARMS}

    def run(arm):
        step_ms, k_ms, _ = timed(torch, fills[arm], steps[arm], args.steps)
        return V / (step_ms / 1e3), step_ms, k_ms
    rows = rounds_of(list(ARMS), args.rounds, run)
    rep = {arm: {("images_per_s" if k == "fps" else k): summary(x) for k, x in rows[arm].items()} for arm in ARMS}
    rep["clip"]["over_off_step"] = float(np.median(rows["clip"]["step_ms"]) / np.median(rows["off"]["step_ms"]))
    rep["clip"]["over_off_k_raster"] = float(np.median(rows["clip"]["k_raster_ms"]) / np.median(rows["off"]["k_raster_ms"]))
    result["workloads"][name] = {"views_per_step": V, "res": RES, "z_near": Z_NEAR, "steps": args.steps,
                                 "outputs_identical": identical, "covered_pixels": drawn, **rep}
    del fills, outs, steps
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--views", type=int, default=128)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("clip_bench needs a CUDA device")
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller, views as VW
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from conftest import load_indexed
    dev = torch.device("cuda", 0)
    result = {"tool": "tools/clip_bench.py", **gpu_info(torch), "rounds": args.rounds, "arms": list(ARMS), "workloads": {}}
    m = load_indexed("trex")
    dv, dc, dn = (torch.from_numpy(a).to(dev) for a in (m._vertices_by_triangles, m._colors_by_triangles, m._normals_by_triangles))
    result["triangles"] = int(dv.shape[0])
    for name, views in (("orbit", VW.orbit_views(args.views, count=args.views)), ("inside", inside_views(args.views))):
        workload(torch, AdvancedPixelBufferFiller, name, dv, dc, dn, torch.from_numpy(views).to(dev), args, result)
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
