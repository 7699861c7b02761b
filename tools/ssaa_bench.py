"""Cost of supersampled images (CRB_SS2 / CRB_SS4, render_views(supersample=s)): images/s and k_raster time of three arms per
workload, alternated in one process.  Prints one JSON line (GPU name, power limit and max SM clock read in the same run).

Arms:
  fused      render_views(supersample=s, color_u8_out=...) at the sample resolution: the rasterizer resolves each s x s block
             and writes 3/s^2 bytes per sample;
  unfused    render_views(want=("color",)) at the sample resolution into float32 slabs (12 bytes per sample), then
             crb_color_u8_resolved per view (reads them back, writes 3/s^2);
  aliased    the 1x uint8 image at the output resolution (render_views(want=(), color_u8_out=...)): the floor.

Workloads:
  trex_512_ss2, trex_512_ss4, trex_1024_ss2   T-Rex (tests/golden/trex_fit.npz), batches of 128 orbit views, output 512^2 /
                                              512^2 / 1024^2 from 1024^2 / 2048^2 / 2048^2 samples
  sphere_4096_ss2                             the 10 M-triangle synthetic.uv_sphere, one view, 4096^2 from 8192^2 samples

Each round times every arm back to back (the order rotates between rounds); the report gives the median and the spread
(min, max) over the rounds.  `k_raster_ms` is the tile rasterizer's device time per step (crb_profile: CUDA events around each
launch), `step_ms` the whole step (CUDA events), `images_per_s` views per second of whole steps.

    python tools/ssaa_bench.py [--rounds 5] [--steps 10] [--out profiles/ssaa_b200.json]
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

ARMS = ("fused", "unfused", "aliased")
IDENTITY = np.array([[1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0, 0, 0, 0, 0]], np.float32)


def bytes_per_sample(s):
    """Algorithmic bytes each arm moves per sample for its image (inputs and binning aside)"""
    return {"fused": {"written": 3 / s ** 2, "read": 0.0},
            "unfused": {"written": 12 + 3 / s ** 2, "read": 12.0},
            "aliased": {"written": 3 / s ** 2, "read": 0.0, "note": "3 bytes per output pixel, no supersampling"}}


def workload(torch, dev, APBF, lib, name, v, c, n, views, out_res, s, args, result):
    V = int(views.shape[0])
    S = out_res * s
    fused = APBF(S, S, fov=45.0, device=0)
    unfused = APBF(S, S, fov=45.0, device=0)
    alias = APBF(out_res, out_res, fov=45.0, device=0)
    img = torch.empty((V, out_res, out_res, 3), dtype=torch.uint8, device=dev)
    col = unfused._color[None] if V == 1 else torch.empty((V, S, S, 3), dtype=torch.float32, device=dev)
    L, H = unfused._L, unfused._handle
    z, nrm = unfused._z.data_ptr(), unfused._normals.data_ptr()

    def resolve_all():
        st = unfused._stream()
        for k in range(V):
            if V > 1:        # the resolve reads the filler's bound colour buffer: bind view k's slab
                lib.check(L.crb_bind_buffers(H, z, col[k].data_ptr(), nrm))
            lib.check(L.crb_color_u8_resolved(H, s, img[k].data_ptr(), st))
        if V > 1:
            lib.check(L.crb_bind_buffers(H, z, unfused._color.data_ptr(), nrm))

    steps = {
        "fused": lambda: fused.render_views(v, c, n, views, color_u8_out=img, supersample=s, chunk=V, check_status=False),
        "unfused": lambda: (unfused.render_views(v, c, n, views, want=("color",), color_out=col, chunk=V, check_status=False),
                            resolve_all()),
        "aliased": lambda: alias.render_views(v, c, n, views, want=(), color_u8_out=img, chunk=V, check_status=False)}
    fills = {"fused": fused, "unfused": unfused, "aliased": alias}
    # workspaces and status checked once (the pair lists fit), then warm-up
    fused.render_views(v, c, n, views, color_u8_out=img, supersample=s, chunk=V)
    unfused.render_views(v, c, n, views, want=("color",), color_out=col, chunk=V)
    alias.render_views(v, c, n, views, want=(), color_u8_out=img, chunk=V)
    for arm in ARMS:
        for _ in range(2):
            steps[arm]()
    nsteps = args.steps if V > 1 else args.steps // 2 + 1

    def run(arm):
        step_ms, k_ms, _ = timed(torch, fills[arm], steps[arm], nsteps)
        return V / (step_ms / 1e3), step_ms, k_ms
    rows = rounds_of(list(ARMS), args.rounds, run)
    rep = {arm: {("images_per_s" if k == "fps" else k): summary(x) for k, x in rows[arm].items()} for arm in ARMS}
    for arm in ("unfused", "aliased"):
        rep[arm]["over_fused_step"] = float(np.median(rows[arm]["step_ms"]) / np.median(rows["fused"]["step_ms"]))
        rep[arm]["over_fused_k_raster"] = float(np.median(rows[arm]["k_raster_ms"]) / np.median(rows["fused"]["k_raster_ms"]))
    result["workloads"][name] = {"views_per_step": V, "output": out_res, "samples": S, "s": s, "steps": nsteps,
                                 "bytes_per_sample": bytes_per_sample(s), **rep}
    del fused, unfused, alias, img, col, fills, steps
    gc.collect()
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10, help="timed steps per arm and round (the sphere runs steps/2 + 1)")
    ap.add_argument("--views", type=int, default=128)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("ssaa_bench needs a CUDA device")
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller, _lib, synthetic, views as VW
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from conftest import load_indexed
    dev = torch.device("cuda", 0)
    result = {"tool": "tools/ssaa_bench.py", **gpu_info(torch), "rounds": args.rounds, "arms": list(ARMS), "workloads": {}}

    m = load_indexed("trex")
    dv, dc, dn = (torch.from_numpy(a).to(dev) for a in (m._vertices_by_triangles, m._colors_by_triangles, m._normals_by_triangles))
    dviews = torch.from_numpy(VW.orbit_views(args.views, count=args.views)).to(dev)
    for out_res, s in ((512, 2), (512, 4), (1024, 2)):
        workload(torch, dev, AdvancedPixelBufferFiller, _lib, f"trex_{out_res}_ss{s}", dv, dc, dn, dviews, out_res, s, args, result)

    sp = synthetic.uv_sphere(3200, 1564)
    sv, sc, sn = (torch.from_numpy(a).to(dev) for a in (sp._vertices_by_triangles, sp._colors_by_triangles, sp._normals_by_triangles))
    del sp
    workload(torch, dev, AdvancedPixelBufferFiller, _lib, "sphere_4096_ss2", sv, sc, sn, torch.from_numpy(IDENTITY).to(dev),
             4096, 2, args, result)
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
