"""Per-pixel texturing (CRB_TEXTURE) against per-vertex colours: frames/s and k_raster time of each shading mode on two
workloads, alternated, in one process.  Prints one JSON line (GPU name and power limit read in the same run).

Modes: "vertex" (per-vertex colours), and per-pixel texturing sampled "nearest" / "bilinear" (CRB_TEX_BILINEAR) / "trilinear"
(CRB_TEX_TRILINEAR, mip chain) from affine or, with the suffix "_persp", perspective-correct (CRB_TEX_PERSPECTIVE) coordinates
-- seven in all.

  trex_1024_orbit  the headline workload of bench.py: T-Rex (tests/golden/trex_fit.npz) at 1024^2, batches of 128 orbit views
                   rendered by render_views into float32 z / colour / normals slabs.  The fixture has no texture coordinates:
                   seeded spherical-projection ones (synthetic.spherical_uvs) and a seeded 709 x 709 texture.
  trex_256_orbit   the same at 256^2, where much of the texture is minified (the regime trilinear filtering is for).
  sphere_8192      the 10 M-triangle synthetic.uv_sphere, one frame at 8192^2 (render_arrays, device-resident inputs, fused
                   clear): its latitude-longitude coordinates and a seeded 4096 x 2048 texture.

Each round times every mode back to back (the order rotates between rounds); the report gives the median and the spread
(min, max) over the rounds, and each mode's medians over those of "vertex" and of "nearest".  `k_raster_ms` is the tile
rasterizer's device time per step (crb_profile: CUDA events around each launch), `step_ms` the whole step (CUDA events).
Also reported: `chain_build_ms`, the one-off crb_pack_texture_mips time (709^2 and 2048 x 4096; CUDA events, median of 20),
and `dropin_trilinear_ms`, the time per frame of the drop-in idiom (a new texture_filter="trilinear" filler and Renderer per
frame, render_model of the torus fixture at 1024^2, which rebuilds the chain every frame) against the same with "bilinear".

    python tools/texture_bench.py [--rounds 7] [--steps 20] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info(torch):
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["clocks_max_sm"] = [s.strip() for s in q.split(",")][:2]
    except Exception as e:      # (reported, not fatal: the numbers still stand with the card's name)
        info["power_limit"] = f"unavailable: {e}"
    return info


def timed(torch, f, step, steps):
    torch.cuda.synchronize()
    f.profile(True)
    f.profile_read()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    launches, k_ms = f.profile_read()
    f.profile(False)
    return e0.elapsed_time(e1) / steps, k_ms / steps, launches


def summary(xs):
    xs = sorted(xs)
    return {"median": float(np.median(xs)), "min": float(xs[0]), "max": float(xs[-1]), "n": len(xs)}


MODES = {"vertex": None, "nearest": ("nearest", False), "nearest_persp": ("nearest", True), "bilinear": ("bilinear", False),
         "bilinear_persp": ("bilinear", True), "trilinear": ("trilinear", False), "trilinear_persp": ("trilinear", True)}


def make_filler(AdvancedPixelBufferFiller, mode, res):
    if MODES[mode] is None:
        return AdvancedPixelBufferFiller(res, res, fov=45.0, device=0)
    filt, persp = MODES[mode]
    return AdvancedPixelBufferFiller(res, res, fov=45.0, device=0, texture_filter=filt, perspective_correct=persp)


def rounds_of(modes, rounds, run):
    """`rounds` rounds of every mode, the order rotated by one each round; returns mode -> {fps, step_ms, k_raster_ms} lists."""
    rows = {mode: {"fps": [], "step_ms": [], "k_raster_ms": []} for mode in modes}
    for r in range(rounds):
        k = r % len(modes)
        for mode in modes[k:] + modes[:k]:
            fps, step_ms, k_ms = run(mode)
            rows[mode]["fps"].append(fps)
            rows[mode]["step_ms"].append(step_ms)
            rows[mode]["k_raster_ms"].append(k_ms)
    return rows


def report(rows):
    out = {mode: {k: summary(v) for k, v in rows[mode].items()} for mode in rows}
    for base in ("vertex", "nearest"):
        for mode in rows:
            if mode != base:
                out[mode][f"over_{base}_k_raster"] = float(np.median(rows[mode]["k_raster_ms"]) / np.median(rows[base]["k_raster_ms"]))
                out[mode][f"over_{base}_fps"] = float(np.median(rows[mode]["fps"]) / np.median(rows[base]["fps"]))
    return out


def trex_workload(torch, dev, AdvancedPixelBufferFiller, VW, m, uv, tex, args, modes, RES, result):
    T, V = int(m._vertices_by_triangles.shape[0]), args.views
    dv, dc, dn = (torch.from_numpy(a).to(dev) for a in (m._vertices_by_triangles, m._colors_by_triangles, m._normals_by_triangles))
    duv = torch.nn.functional.pad(torch.from_numpy(uv).to(dev), (0, 1)).contiguous()
    dviews = torch.from_numpy(VW.orbit_views(V, count=V)).to(dev)
    z = torch.empty((V, RES, RES), dtype=torch.float32, device=dev)
    col = torch.empty((V, RES, RES, 3), dtype=torch.float32, device=dev)
    nrm = torch.empty((V, RES, RES, 3), dtype=torch.float32, device=dev)
    fill = {mode: make_filler(AdvancedPixelBufferFiller, mode, RES) for mode in modes}

    def trex_step(mode):
        f = fill[mode]
        kw = {"texture": tex} if MODES[mode] else {}
        c = duv if MODES[mode] else dc
        return lambda: f.render_views(dv, c, dn, dviews, z_out=z, color_out=col, normals_out=nrm, chunk=V, check_status=False,
                                      **kw)
    for mode in fill:     # workspace, status check, texture upload, warm-up
        fill[mode].render_views(dv, duv if MODES[mode] else dc, dn, dviews, z_out=z, color_out=col, normals_out=nrm, chunk=V,
                                **({"texture": tex} if MODES[mode] else {}))
        for _ in range(3):
            trex_step(mode)()

    def trex_run(mode):
        step_ms, k_ms, _ = timed(torch, fill[mode], trex_step(mode), args.steps)
        return V / (step_ms / 1e3), step_ms, k_ms
    rows = rounds_of(modes, args.rounds, trex_run)
    result["workloads"][f"trex_{RES}_orbit"] = {
        "triangles": T, "views_per_step": V, "resolution": RES, "texture": [709, 709], "steps": args.steps, **report(rows)}
    del z, col, nrm, fill


def chain_build(torch, dev):
    """One-off crb_pack_texture_mips time (ms, median of 20 after 3 warm-ups) for a 709^2 and a 2048 x 4096 texture."""
    import ctypes
    from cython3dmodelrenderer_b200 import _lib
    L = _lib.load_library()
    out = {}
    for th, tw in ((709, 709), (2048, 4096)):
        bgr = torch.from_numpy(np.random.default_rng(th).integers(0, 256, (th, tw, 3), dtype=np.uint8)).to(dev)
        texels = ctypes.c_int64()
        _lib.check(L.crb_mip_layout(th, tw, None, ctypes.byref(texels)))
        chain = torch.empty((texels.value,), dtype=torch.int32, device=dev)
        st = torch.cuda.current_stream().cuda_stream
        ts = []
        for i in range(23):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            _lib.check(L.crb_pack_texture_mips(bgr.data_ptr(), th, tw, chain.data_ptr(), st))
            e1.record()
            torch.cuda.synchronize()
            if i >= 3:
                ts.append(e0.elapsed_time(e1))
        out[f"{th}x{tw}"] = summary(ts)
    return out


def dropin(torch, rounds):
    """Time per frame (ms, host clock around frames that end in a download) of the drop-in idiom with a new filler per frame."""
    import time
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller, NoIllumination, Renderer
    from cython3dmodelrenderer_b200.model import Model
    cwd = os.getcwd()
    os.chdir(os.path.join(ROOT, "tests", "golden", "obj"))
    try:
        model = Model.read_model("torus.obj")
    finally:
        os.chdir(cwd)
    rows = {"bilinear": [], "trilinear": []}
    for r in range(rounds + 1):
        for filt in rows:
            t0 = time.perf_counter()
            for _ in range(10):
                f = AdvancedPixelBufferFiller(1024, 1024, fov=45, texturing="pixel", texture_filter=filt)
                Renderer(f, NoIllumination(), None, 1024, 1024).render(model)
            torch.cuda.synchronize()
            if r:
                rows[filt].append((time.perf_counter() - t0) / 10 * 1e3)
    return {filt: summary(v) for filt, v in rows.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=20, help="timed steps per mode and round (headline); the sphere runs steps/4 + 1")
    ap.add_argument("--views", type=int, default=128)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    modes = list(MODES)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("texture_bench needs a CUDA device")
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller, synthetic, views as VW
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from conftest import load_indexed
    dev = torch.device("cuda", 0)
    result = {"tool": "tools/texture_bench.py", **gpu_info(torch), "rounds": args.rounds, "modes": modes, "workloads": {}}

    # ---- headline: T-Rex 1024^2 (and 256^2), 128 orbit views per step
    m = load_indexed("trex")
    T = int(m._vertices_by_triangles.shape[0])
    uv = synthetic.spherical_uvs(m._vertices_by_triangles)
    tex = np.random.default_rng(709).integers(0, 256, (709, 709, 3), dtype=np.uint8)
    for RES in (1024, 256):
        trex_workload(torch, dev, AdvancedPixelBufferFiller, VW, m, uv, tex, args, modes, RES, result)
    torch.cuda.empty_cache()
    result["chain_build_ms"] = chain_build(torch, dev)
    result["dropin_trilinear_ms"] = dropin(torch, args.rounds)

    # ---- 10 M-triangle sphere at 8192^2, one frame per step
    s = synthetic.uv_sphere(3200, 1564)
    T = int(s._vertices_by_triangles.shape[0])
    suv = synthetic.spherical_uvs(s._vertices_by_triangles, center=(0.0, 0.0, 1.5))
    stex = np.random.default_rng(4096).integers(0, 256, (2048, 4096, 3), dtype=np.uint8)
    sv, sc, sn = (torch.from_numpy(a).to(dev) for a in (s._vertices_by_triangles, s._colors_by_triangles, s._normals_by_triangles))
    suvd = torch.nn.functional.pad(torch.from_numpy(suv).to(dev), (0, 1)).contiguous()
    del s, suv
    RES = 8192
    fills = {mode: make_filler(AdvancedPixelBufferFiller, mode, RES) for mode in modes}

    def sphere_step(mode):
        fs = fills[mode]

        def step():
            fs.clear()
            if MODES[mode]:
                fs.render_arrays(sv, suvd, sn, check_status=False, texture=stex)
            else:
                fs.render_arrays(sv, sc, sn, check_status=False)
        return step
    for mode in modes:
        fs = fills[mode]
        fs.clear()
        fs.render_arrays(sv, suvd if MODES[mode] else sc, sn, **({"texture": stex} if MODES[mode] else {}))
        fs.get_z_buffer()         # status checked (the pair list fits)
        for _ in range(2):
            sphere_step(mode)()
    ssteps = args.steps // 4 + 1

    def sphere_run(mode):
        step_ms, k_ms, _ = timed(torch, fills[mode], sphere_step(mode), ssteps)
        return 1e3 / step_ms, step_ms, k_ms
    srows = rounds_of(modes, args.rounds, sphere_run)
    result["workloads"]["sphere_8192"] = {
        "triangles": T, "resolution": RES, "texture": [2048, 4096], "steps": ssteps, **report(srows)}
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
