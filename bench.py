#!/usr/bin/env python
"""bench.py -- T-Rex 1024^2 frames/s (BASELINE.json metric) on N B200s, beside the reference's CPU path.

Workload (config.workload = "trex_1024_orbit"): every rank renders V (default 128) views per step of an N*V-view
orbit of T-Rex (README fit_model flow, 13 814 triangles) at 1024x1024, fov 45, no illumination -- each view with
fresh-filler buffers, all three float32 buffers (z, colour, normals: 28 B/pixel) written to its own slab in HBM.
At N=8 one step is exactly BASELINE.json's config C5 (1024-view orbit, view-sharded); views are independent, so there is
no data-path collective ("scaling": "weak").  `value` = frames/s with mesh + view matrices resident in HBM; `e2e` =
frames/s through the host-buffer C-ABI call (crb_render_host: H2D of the three [T,3,3] arrays, render, D2H of all three
buffers, per frame).  `--impl reference` times the reference's own Cython/OpenMP Version C (oracle/_ref, else the C
oracle port) on the host cores on a bounded sample of the same orbit.

One JSON line on stdout (rank 0).  See DESIGN.md section "Measurement" for the definitions of every key.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

RES = 1024
FOV = 45.0
METRIC = "T-Rex 1024^2 frames/s"


def load_trex():
    from conftest import load_indexed
    return load_indexed("trex")


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


class ClockSampler:
    """SM clock + throttle reasons sampled every few ms while the timed region runs: NVML in a thread (no process to
    spawn, so even a 20 ms region gets several samples); `nvidia-smi -lms` as the fallback."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index, period_s=0.004):
        self.index, self.rows, self.proc, self.period = index, [], None, period_s
        self.nvml, self.stop_flag, self.how, self.err = None, False, None, None

    def _nvml_setup(self):
        """Everything that can be done before the load starts: handle, constants, the one-sample closure."""
        n, hnd = self.nvml
        R = {"hw_slowdown": getattr(n, "nvmlClocksEventReasonHwSlowdown", getattr(n, "nvmlClocksThrottleReasonHwSlowdown", 0x8)),
             "hw_thermal_slowdown": getattr(n, "nvmlClocksEventReasonHwThermalSlowdown", getattr(n, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40)),
             "sw_thermal_slowdown": getattr(n, "nvmlClocksEventReasonSwThermalSlowdown", getattr(n, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20)),
             "sw_power_cap": getattr(n, "nvmlClocksEventReasonSwPowerCap", getattr(n, "nvmlClocksThrottleReasonSwPowerCap", 0x4))}
        get_reasons = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
        mx = n.nvmlDeviceGetMaxClockInfo(hnd, n.NVML_CLOCK_SM)

        def one():
            try:
                sm = n.nvmlDeviceGetClockInfo(hnd, n.NVML_CLOCK_SM)
                bits = get_reasons(hnd)
                self.rows.append((float(sm), float(mx), [k for k, b in R.items() if bits & b]))
            except Exception as ex:
                self.err = repr(ex)[:120]
        self.one = one

    def _nvml_loop(self):
        while not self.stop_flag:
            self.one()
            time.sleep(self.period)

    def __enter__(self):
        try:
            import pynvml as n
            n.nvmlInit()
            idx = self.index
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:
                idx = int(vis.split(",")[self.index])
            self.nvml = (n, n.nvmlDeviceGetHandleByIndex(idx))
            self.how = "nvml"
            self._nvml_setup()
            self.t = threading.Thread(target=self._nvml_loop, daemon=True)
            self.t.start()
            return self
        except Exception as ex:
            self.err = repr(ex)[:120]
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.how = "nvidia-smi -lms 20"
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def sample_now(self, n=3):
        """Synchronous samples from the calling thread -- called right after the timed steps have been queued, while the
        GPU is still working through them (a short region may end before the sampling thread is scheduled once)."""
        one = getattr(self, "one", None)
        for _ in range(n):
            if one:
                one()

    def _read(self):
        for line in self.proc.stdout:
            r = [x.strip() for x in line.split(",")]
            try:
                self.rows.append((float(r[0]), float(r[1]),
                                  [name for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7])
                                   if v.lower().startswith("active")]))
            except Exception:
                pass

    def __exit__(self, *a):
        if self.nvml:
            self.stop_flag = True
            self.t.join(timeout=1)
        elif self.proc:
            time.sleep(0.05)
            self.proc.terminate()
            self.t.join(timeout=2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"], "how": self.how, "error": self.err}
        reasons = sorted({r for row in self.rows for r in row[2]})
        return {"sm_mhz": statistics.median(r[0] for r in self.rows), "sm_max_mhz": max(r[1] for r in self.rows),
                "reasons": reasons, "samples": len(self.rows), "how": self.how}


# --------------------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's own Version C on the host cores
# --------------------------------------------------------------------------------------------------------------------
def cpu_reference_runner(n_threads=None, res=None, fov=FOV):
    """Returns (kind, cores, render(v, c, n) -> seconds).  A fresh filler per frame (Version C has no buffer reset),
    constructor and lock-grid initialisation outside the timed part, stdout silenced (the reference printf()s)."""
    from conftest import TriModel
    from oracle import build_ref
    res = RES if res is None else int(res)
    cores = n_threads or os.cpu_count() or 1
    if build_ref.built():
        sys.path.insert(0, os.path.join(ROOT, "oracle", "_ref"))
        devnull = os.open(os.devnull, os.O_WRONLY)
        saved = os.dup(1)
        os.dup2(devnull, 1)
        try:
            from crender.cy.pixel_buffer_filler import AdvancedPixelBufferFiller as Ref
        finally:
            os.dup2(saved, 1)

        def render(v, c, n):
            f = Ref(res, res, fov=fov, n_threads=cores)
            f.get_z_buffer()[...] += 0  # pre-touch all three buffers (np.zeros pages are mapped lazily)
            f.get_color_buffer()[...] = 0
            f.get_normals_buffer()[...] = 0
            m = TriModel(v, c, n)
            sys.stdout.flush()
            os.dup2(devnull, 1)
            try:
                t0 = time.perf_counter()
                f.render_model(m)
                dt = time.perf_counter() - t0
            finally:
                os.dup2(saved, 1)
            return dt
        return "reference", cores, render
    from oracle import oracle as O

    def render(v, c, n):
        f = O.OracleFiller(res, res, fov=fov, n_threads=cores)
        t0 = time.perf_counter()
        f.render_arrays(v, c, n)
        return time.perf_counter() - t0
    return "port", cores, render


def best_cpu_threads(arrays, colors):
    """The reference's OpenMP path does not scale monotonically (dynamic schedule + per-pixel locks): it gets its best
    thread count among {8, 16, 32, nproc/2, nproc} (median of 8 frames each after a warm-up) instead of blindly nproc."""
    nproc = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, nproc // 2, nproc) if 1 <= c <= nproc} or {1})
    best = None
    for c in cands:
        _, _, render = cpu_reference_runner(c)
        ts = []
        for i in range(9):
            v, n = arrays[i % len(arrays)]
            ts.append(render(v, colors, n))
        med = statistics.median(ts[1:])
        if best is None or med < best[0]:
            best = (med, c)
    return best[1]


def headline_config(T, V, n_total, chunk):
    """`config` of the headline line -- one function, because both arms must print the same dict."""
    return {"workload": "trex_1024_orbit", "res": RES, "fov": FOV, "triangles": int(T), "views_per_gpu_per_step": int(V),
            "orbit_views_total": int(n_total), "view_to_rank": "k mod N", "views_per_launch": int(chunk), "illumination": False,
            "buffers": "z+color+normals f32, fresh per view", "l2": "outputs %.2f GB/step per GPU >> 126 MB L2; "
            "the 1.5 MB mesh is re-read per view by design" % (V * 28 * RES * RES / 1e9)}


DUMP_SAMPLE_PIXELS = 1 << 19


def dump_outputs(out_dir, z, col, nrm):
    """--dump-outputs: the buffers the timed render_views steps left for their caller (z [V,H,W], colour and normals
    [V,H,W,3], float32) as .npy files, so that two builds can be compared output for output.  The whole batch is 3.7 GB at
    V = 128, so what is written is view 0 in full (<name>_view0.npy, 29 MB) and the same pixels of every view at
    DUMP_SAMPLE_PIXELS flat indices into [V,H,W] drawn without replacement by numpy's default_rng(0), in ascending order
    (<name>_sample.npy, 15 MB).  Only rank 0 writes, and rank 0 renders orbit views 0, N, 2N, ... of the N * V-view orbit
    (N = ranks, V = --views): dumps compare output for output when they were taken with the same N and V."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    n = z.numel()
    idx = np.sort(np.random.default_rng(0).choice(n, size=min(DUMP_SAMPLE_PIXELS, n), replace=False))
    didx = torch.from_numpy(idx).to(z.device)
    for name, t in (("z", z), ("color", col), ("normals", nrm)):
        np.save(os.path.join(out_dir, f"{name}_view0.npy"), t[0].cpu().numpy())
        np.save(os.path.join(out_dir, f"{name}_sample.npy"), t.reshape(n, -1)[didx].squeeze(-1).cpu().numpy())


def sample_view_indices(n_total, count=8):
    """Views k * n_total / count: an evenly spread sample of the orbit (frames of different view angles cost differently)."""
    return [(k * n_total) // count for k in range(count)]


def orbit_sample_arrays(model, n_total, count=8):
    from cython3dmodelrenderer_b200 import views as VW
    out = []
    for k in sample_view_indices(n_total, count):
        view = VW.orbit_views(n_total, first=k, count=1)[0]
        out.append(VW.transform_arrays_host(view, model._vertices_by_triangles, model._normals_by_triangles))
    return out


def cpu_frames(model, n_total, frames, warm=2):
    """Host Version C on `frames` frames cycling through 8 evenly spread views of the n_total-view orbit."""
    arrays = orbit_sample_arrays(model, n_total, 8)
    kind, cores, render = cpu_reference_runner(best_cpu_threads(arrays, model._colors_by_triangles))
    times = []
    for i in range(warm + frames):
        v, n = arrays[i % len(arrays)]
        dt = render(v, model._colors_by_triangles, n)
        if i >= warm:
            times.append(dt)
    return kind, cores, times


def reference_renderer_flow_ms(model, cores, frames=5, res=None):
    """The whole run.py:20-25 flow of the reference on the host: its Renderer, GuroIllumination([0, 0, 1]) (NumPy over the whole
    frame) and Version C filler, a new filler per frame; median milliseconds per frame.  None without oracle/_ref."""
    from conftest import TriModel
    from oracle import build_ref
    if not build_ref.built():
        return None
    sys.path.insert(0, os.path.join(ROOT, "oracle", "_ref"))
    devnull = os.open(os.devnull, os.O_WRONLY)
    saved = os.dup(1)
    sys.stdout.flush()
    os.dup2(devnull, 1)          # (the reference printf()s per OpenMP thread)
    try:
        from crender.cy import Renderer
        from crender.cy.illumination import GuroIllumination
        from crender.cy.pixel_buffer_filler import AdvancedPixelBufferFiller as Ref
        m = TriModel(model._vertices_by_triangles, model._colors_by_triangles, model._normals_by_triangles)
        ts = []
        for _ in range(frames + 1):
            t0 = time.perf_counter()
            Renderer(Ref(res or RES, res or RES, fov=FOV, n_threads=cores), GuroIllumination([0, 0, 1]), None, res or RES, res or RES).render(m)
            ts.append(time.perf_counter() - t0)
    finally:
        os.dup2(saved, 1)
        os.close(devnull)
        os.close(saved)
    return 1000.0 * statistics.median(ts[1:])


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    model = load_trex()
    T = model._vertices_by_triangles.shape[0]
    n_total = args.gpus * args.views
    arrays = orbit_sample_arrays(model, n_total, 8)           # views k * n_total / 8: the whole orbit, not one pose
    kind, cores, render = cpu_reference_runner(best_cpu_threads(arrays, model._colors_by_triangles))
    sample = 16  # frames per step: a bounded sample of the orbit (each of the 8 views twice)
    step_s = []
    for s in range(args.warmup + args.steps):
        t = 0.0
        for i in range(sample):
            v, n = arrays[i % 8]
            t += render(v, model._colors_by_triangles, n)
        if s >= args.warmup:
            step_s.append(t)
    total = sum(step_s)
    fps = sample * args.steps / total
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 * total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic orbit of the T-Rex fixture (tests/golden/trex_fit.npz)",
        # the same config as the GPU arm's line (the driver compares the two dicts); what this arm sampled of it is said beside it
        "config": headline_config(int(T), args.views, n_total, args.chunk),
        "reference_sample": {"frames_per_step": sample, "views": sample_view_indices(n_total, 8)},
        "gtri_per_s": fps * T / 1e9,
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "host_cores": os.cpu_count(), "kind": kind,
                         "sample": f"{sample} frames per step x {args.steps} steps cycling through 8 evenly spread views "
                                   f"(k * {n_total} / 8) of the orbit, render_model only, fresh filler per frame, n_threads={cores} "
                                   f"(the fastest of 8/16/32/nproc/2/nproc on this host, nproc={os.cpu_count()})"},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# --------------------------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------------------------
def run_gpu_arm(args):
    import torch
    import torch.distributed as dist
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller, _lib
    from cython3dmodelrenderer_b200 import views as VW

    world, rank, local, dev = init_dist()

    model = load_trex()
    T = int(model._vertices_by_triangles.shape[0])
    V = args.views
    n_total = world * V
    views_np = VW.orbit_views(n_total, first=rank, count=V, stride=world)      # view k -> rank k mod N: equal work per rank
    f = AdvancedPixelBufferFiller(RES, RES, fov=FOV, device=local)
    dv, dc, dn = (torch.from_numpy(a).to(dev) for a in
                  (model._vertices_by_triangles, model._colors_by_triangles, model._normals_by_triangles))
    dviews = torch.from_numpy(views_np).to(dev)
    z = torch.empty((V, RES, RES), dtype=torch.float32, device=dev)
    col = torch.empty((V, RES, RES, 3), dtype=torch.float32, device=dev)
    nrm = torch.empty((V, RES, RES, 3), dtype=torch.float32, device=dev)

    def step():
        # back-to-back batches: the join with the internal rasterizer stream is deferred (f.join() below), so the next
        # step's setup / binning kernels run beside this step's rasterizer
        f.render_views(dv, dc, dn, dviews, z_out=z, color_out=col, normals_out=nrm, chunk=args.chunk, check_status=False,
                       defer_join=True)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    f.render_views(dv, dc, dn, dviews, z_out=z, color_out=col, normals_out=nrm, chunk=args.chunk)  # sizes workspace, checks status
    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    launches0 = f.launch_count
    f.profile(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clocks:
        barrier()
        e0.record()
        for _ in range(args.steps):
            step()
        f.join()
        e1.record()
        clocks.sample_now()      # the GPU is still inside the timed steps here (launches are asynchronous)
        barrier()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, z, col, nrm)
    k_launches, k_ms = f.profile_read()
    f.profile(False)
    launches = f.launch_count - launches0
    need, cap = ctypes.c_int64(), ctypes.c_int64()
    _lib.check(f._L.crb_status(f._handle, ctypes.byref(need), ctypes.byref(cap), f._stream()))
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    frames = world * V * args.steps
    fps = frames / (ms / 1000.0)
    if rank == 0:      # what the watchdog prints should a later leg (deliveries, secondary configs) hang: the headline, measured above
        _PARTIAL.update({
            "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic orbit of the T-Rex fixture (tests/golden/trex_fit.npz = README fit_model flow)",
            "config": headline_config(T, V, n_total, args.chunk), "gtri_per_s": fps * T / 1e9, "clocks": clocks.summary(),
            "gpu_launches": launches})

    # the rasterizer timed alone: the same steps without the front end of the next launch running beside it
    _lib.check(f._L.crb_set_option(f._handle, _lib.CRB_OPT_CHUNK_PIPELINE, 0))
    for _ in range(2):
        step()
    torch.cuda.synchronize()
    f.profile(True)
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    for _ in range(5):
        step()
    s1.record()
    torch.cuda.synchronize()
    a_launches, a_ms = f.profile_read()
    a_step_ms = s0.elapsed_time(s1)
    f.profile(False)
    _lib.check(f._L.crb_set_option(f._handle, _lib.CRB_OPT_CHUNK_PIPELINE, 1))

    # ---- delivery of the view-sharded result over NVLink (SURVEY 8e; reported beside `value`, which is the rendering rate) ----
    gather = None
    if world > 1 and args.gather != "none":
        from cython3dmodelrenderer_b200 import sharding
        NVLINK_IN = 900.0e9        # NVLink 5 / NVSwitch: bytes per second into one GPU (nominal, per direction)
        gchunk = min(args.chunk, 32)
        u8 = torch.empty((V, RES, RES, 3), dtype=torch.uint8, device=dev)

        def produce_u8(first, count):
            f.render_views(dv, dc, dn, dviews[first:first + count], want=(), color_u8_out=u8[first:first + count], chunk=count,
                           check_status=False)
            return u8[first:first + count]

        def produce_z(first, count):
            f.render_views(dv, dc, dn, dviews[first:first + count], want=("z",), z_out=z[first:first + count], chunk=count,
                           check_status=False)
            return z[first:first + count]

        def timed(fn, reps=3):
            fn()
            barrier()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            for _ in range(reps):
                fn()
            g1.record()
            barrier()
            t_ = torch.tensor([g0.elapsed_time(g1) / reps], dtype=torch.float64, device=dev)
            dist.all_reduce(t_, op=dist.ReduceOp.MAX)
            return float(t_.item())

        def render_only(produce):
            for first in range(0, V, gchunk):
                produce(first, min(gchunk, V - first))

        gather = {"note": "`value` is the rendering rate with every rank's views left in its own HBM; the entries below add the "
                          "delivery.  One GPU takes 900 GB/s from NVLink while eight produce 2-3 TB/s of frames, so everything "
                          "gathered into ONE rank is bound by that rank's ingress (ingress_bound_frames_per_s); the row exchange "
                          "(all-to-all: every rank ends with its row band of ALL views) spreads the ingress over the ranks and "
                          "scales", "chunk_views": gchunk}
        want_modes = ("u8", "z", "exchange_nccl", "u8_peer", "exchange") if args.gather in ("auto", "all") else (args.gather,)

        def fused(mode):
            """Delivery fused into the rasterizer (sharding.RowExchange / crb_set_u8_exchange): k_raster stores the uint8 image
            row band by row band into the receiving ranks' memory over NVLink -- one launch of all V views, no NCCL call."""
            xch = sharding.RowExchange(V, RES, RES, local_device=local, gather_to=0 if mode == "u8_peer" else None)
            try:
                def both_fn():
                    f.render_views(dv, dc, dn, dviews, want=(), chunk=args.chunk, check_status=False, u8_exchange=xch.plan(0))

                def only_fn():
                    f.render_views(dv, dc, dn, dviews, want=(), color_u8_out=u8, chunk=args.chunk, check_status=False)
                both = timed(both_fn)
                only = timed(only_fn)
                t = xch.tensor()
                # lit pixels of view 0 of the LAST rank as far as this rank received it (all of it on the gather destination, this
                # rank's row band after the exchange -- summed over the ranks below)
                check_px = int((t[world - 1, 0].sum(dim=-1) > 0).sum().item()) if t is not None else 0
                if mode == "exchange":
                    cp = torch.tensor([check_px], dtype=torch.int64, device=dev)
                    dist.all_reduce(cp)
                    check_px = int(cp.item())
                same = None
                if t is not None:      # the delivered bytes are the ones a local render of the same views holds
                    band = u8[0, :xch.hb] if mode == "exchange" and rank == 0 else (u8[0] if rank == 0 else None)
                    same = bool(torch.equal(t[rank, 0], band)) if band is not None else None
                return both, only, check_px, same
            finally:
                xch.close()

        for mode in want_modes:
            if mode in ("exchange", "u8_peer"):
                bpf = 3 * RES * RES
                try:
                    both, only, check_px, same = fused(mode)
                    if mode == "exchange":
                        bound = NVLINK_IN * world * world / (bpf * max(world - 1, 1))
                        what = ("row exchange of the uint8 images fused into the rasterizer: k_raster stores each image row band straight into "
                                "the memory of the rank that owns the band (peer memory over NVLink / NVSwitch, crb_set_u8_exchange); rank r "
                                "ends with rows [r*H/N, (r+1)*H/N) of all N*V views; no NCCL call, no staging copy")
                    else:
                        bound = NVLINK_IN / bpf * world / max(world - 1, 1)
                        what = ("the uint8 images of all views written by every rank's k_raster straight into rank 0's memory (peer stores "
                                "over NVLink, crb_set_u8_exchange with one band): a gather without a collective")
                    delivered = n_total / (both / 1000.0)
                    gather[mode] = {"what": what, "bytes_per_frame": bpf, "ms_render_only": only, "ms_render_and_delivery": both,
                                    "frames_per_s_render_only": n_total / (only / 1000.0), "frames_per_s_delivered": delivered,
                                    "ingress_bound_frames_per_s": bound, "frac_of_ingress_bound": delivered / bound,
                                    "delivery_efficiency": only / both,
                                    "check_pixels": check_px, "delivered_equals_local_render": same}
                except Exception as ex:
                    gather[mode] = {"error": repr(ex)[:300]}
                continue
            if mode == "u8":
                produce, bpf, what = produce_u8, 3 * RES * RES, "run.py:26's uint8 images of all views gathered to rank 0 (NCCL gather per chunk, travelling while the next chunk is rendered)"
            elif mode == "z":
                produce, bpf, what = produce_z, 4 * RES * RES, "the float32 z buffers of all views gathered to rank 0 (NCCL gather per chunk beside the rendering)"
            elif mode == "exchange_nccl":
                produce, bpf, what = produce_u8, 3 * RES * RES, ("row exchange of the uint8 images the library way (NCCL all-to-all per chunk beside the rendering; kept as the baseline of the fused exchange): rank r ends "
                                                                "with rows [r*H/N, (r+1)*H/N) of all N*V views -- the delivery layout whose ingress is spread over the ranks")
            else:
                continue
            try:
                if mode == "exchange_nccl":
                    res_buf = sharding.exchange_rows_overlapped(produce, V, gchunk)
                    both = timed(lambda: sharding.exchange_rows_overlapped(produce, V, gchunk, out=res_buf))
                    bound = NVLINK_IN * world * world / (bpf * max(world - 1, 1))   # a rank receives its 1/N row band of the (N-1)/N frames other ranks render
                    check_px = int((res_buf[world - 1, 0].sum(dim=-1) > 0).sum().item())
                else:
                    res_buf = sharding.gather_views_overlapped(produce, V, gchunk, dst=0)
                    both = timed(lambda: sharding.gather_views_overlapped(produce, V, gchunk, dst=0, out=res_buf))
                    bound = NVLINK_IN / bpf * world / max(world - 1, 1)     # rank 0 receives the frames of the other N-1 ranks
                    check_px = int((res_buf[world - 1, 0].reshape(RES * RES, -1).abs().sum(dim=-1) > 0).sum().item()) if rank == 0 else None
                only = timed(lambda: render_only(produce))
                delivered = n_total / (both / 1000.0)
                gather[mode] = {"what": what, "bytes_per_frame": bpf, "ms_render_only": only, "ms_render_and_delivery": both,
                                "frames_per_s_render_only": n_total / (only / 1000.0), "frames_per_s_delivered": delivered,
                                "ingress_bound_frames_per_s": bound, "frac_of_ingress_bound": delivered / bound,
                                "delivery_efficiency": only / both, "check_pixels": check_px}
                del res_buf
            except Exception as ex:     # a delivery variant must never take the headline line down
                gather[mode] = {"error": repr(ex)[:300]}
        del u8

    # sanity: the timed output is a real frame (covered pixel count of view 0 of rank 0 is the reference's 252 539)
    covered0 = int((z[0] < 1e5).sum().item())

    # ---- roofline of the dominant kernel (tile rasterizer + deferred shading) -----------------------------------
    peak, peak_src = peaks()
    alg_bytes_frame = 108 * T + 28 * RES * RES          # SURVEY 8d: read 3x[T,3,3] once, write 28 B/pixel once
    views_per_launch = V * args.steps / max(k_launches, 1)
    k_avg_ms = k_ms / max(k_launches, 1)
    achieved = alg_bytes_frame * views_per_launch / (k_avg_ms / 1000.0) / 1e9 if k_avg_ms > 0 else None
    roofline = {"bound": "hbm", "kernel": "k_raster (tile rasterizer + deferred shading; every fourth CTA issues the fused clear as TMA boxes)",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": (achieved / peak) if achieved else None,
                "traffic": None, "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes_frame * views_per_launch,
                "avg_launch_ms": k_avg_ms, "launches_timed": k_launches,
                "share_of_step": a_ms / a_step_ms if a_step_ms else None,       # serial launches: comparable with the ncu launch list
                "share_of_step_timed_region": k_ms / ms if ms else None,       # overlapped: k_raster spans almost the whole step
                "whole_step_achieved_gbs": alg_bytes_frame * V * args.steps / (e0.elapsed_time(e1) / 1000.0) / 1e9,
                "whole_step_frac": alg_bytes_frame * V * args.steps / (e0.elapsed_time(e1) / 1000.0) / 1e9 / peak,
                "note": "in the timed region the setup/binning kernels of the next launch run beside k_raster (second stream), which "
                        "lengthens each k_raster launch; frac_kernel_alone is k_raster with that overlap switched off",
                "frac_kernel_alone": (alg_bytes_frame * views_per_launch / (a_ms / max(a_launches, 1) / 1000.0) / 1e9 / peak) if a_ms > 0 else None,
                "avg_launch_ms_alone": a_ms / max(a_launches, 1)}
    for name in ("r02_k_raster_traffic.json", "r01_k_raster_traffic.json"):    # from the ncu --set full capture of the same launch
        prof = os.path.join(ROOT, "profiles", name)
        if os.path.exists(prof):
            try:
                roofline["traffic"] = json.load(open(prof)).get("dram_bytes_per_launch")
                roofline["traffic_source"] = "profiles/" + name
                break
            except Exception:
                pass

    # ---- e2e: host buffers through the C ABI, H2D + render + D2H of all three buffers per frame -------------------
    e2e_frames = args.e2e_frames
    host_in = []
    NIN = 5     # distinct host inputs, coprime with the pipeline depth: every slot keeps seeing different views
    for k in range(NIN):
        vk, nk = VW.transform_arrays_host(views_np[k % V], model._vertices_by_triangles, model._normals_by_triangles)
        st = torch.empty((3, T, 3, 3), dtype=torch.float32).pin_memory()
        st[0].copy_(torch.from_numpy(vk)); st[1].copy_(torch.from_numpy(model._colors_by_triangles)); st[2].copy_(torch.from_numpy(nk))
        host_in.append(st)
    hz = torch.empty((RES, RES), dtype=torch.float32).pin_memory()
    hc = torch.empty((RES, RES, 3), dtype=torch.float32).pin_memory()
    hn = torch.empty((RES, RES, 3), dtype=torch.float32).pin_memory()
    f._ensure_workspace(T)
    L, h = f._L, f._handle

    def e2e_frame(i):
        st = host_in[i % NIN]
        _lib.check(L.crb_render_host(h, st[0].data_ptr(), st[1].data_ptr(), st[2].data_ptr(), T, _lib.CRB_CLEAR_FIRST,
                                     _lib.CRB_BUF_ALL, hz.data_ptr(), hc.data_ptr(), hn.data_ptr(), f._stream()))
    for i in range(3):
        e2e_frame(i)
    barrier()
    t0 = time.perf_counter()
    for i in range(e2e_frames):
        e2e_frame(i)
    torch.cuda.synchronize()
    sync_s = time.perf_counter() - t0
    sync_cov = int((hz < 1e5).sum().item())

    # pipelined: `depth` fillers round-robin (own stream, device buffers, pinned outputs); frame k+1's upload + render
    # overlap frame k's download.  Same call (crb_render_host, CRB_NO_SYNC), same bytes per frame, every frame's three
    # buffers land in host memory before its slot is reused.
    from cython3dmodelrenderer_b200.pipeline import HostFramePipeline

    def run_pipeline(sparse, want=("z", "color", "normals")):
        pipe = HostFramePipeline(RES, RES, fov=FOV, depth=args.e2e_depth, device=local, sparse=sparse, want=want)
        for i in range(2 * args.e2e_depth):
            pipe.submit(*host_in[i % NIN])
        pipe.drain()
        if sparse:
            pipe.readback_tiles()
        l0 = pipe.launch_count
        barrier()
        t0 = time.perf_counter()
        last = 0
        for i in range(e2e_frames):
            last = pipe.submit(*host_in[i % NIN])
        pipe.drain()
        dt = time.perf_counter() - t0
        res = pipe.result(last)
        cov = int((res["z"] < 1e5).sum()) if "z" in res else int((res["color"].sum(axis=-1) > 0).sum())
        tiles = pipe.readback_tiles() if sparse else None
        return dt, cov, pipe.launch_count - l0, tiles

    # run.py's product: the flipped uint8 image (N3), 3 bytes per pixel over PCIe, nothing else produced
    from cython3dmodelrenderer_b200.pipeline import HostImagePipeline

    def run_image_pipeline():
        pipe = HostImagePipeline(RES, RES, fov=FOV, depth=args.e2e_depth, device=local)
        for i in range(2 * args.e2e_depth):
            pipe.submit(host_in[i % NIN])
        pipe.drain()
        barrier()
        t0 = time.perf_counter()
        last = 0
        for i in range(e2e_frames):
            last = pipe.submit(host_in[i % NIN])
        pipe.drain()
        dt = time.perf_counter() - t0
        img = pipe.result(last)
        return dt, int((img.sum(axis=-1) > 0).sum())

    img_s, img_cov = run_image_pipeline()
    dense_s, dense_cov, dense_launches, _ = run_pipeline(False)
    e2e_s, e2e_cov, e2e_launches, tiles_copied = run_pipeline(True)
    col_s, col_cov, _, col_tiles = run_pipeline(True, want=("color",))
    if world > 1:
        t = torch.tensor([e2e_s, sync_s, dense_s, col_s, img_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s, sync_s, dense_s, col_s, img_s = (float(x) for x in t.tolist())
    d2h_sparse = tiles_copied * 32 * 32 * 28 / e2e_frames
    e2e = {"value": world * e2e_frames / e2e_s, "unit": "frames/s", "h2d_bytes_per_step": 108 * T,
           "d2h_bytes_per_step": d2h_sparse, "frames_timed": e2e_frames, "pipeline_depth": args.e2e_depth,
           "gpu_launches": e2e_launches,
           "api": "HostFramePipeline.submit -> crb_render_host(CRB_NO_SYNC | CRB_DL_SPARSE): pinned host [T,3,3] arrays in; z+colour+"
                  "normals (f32, 28 B/pixel) complete in pinned host memory after every frame; only tiles that are busy in the frame "
                  "or were busy in the frame the host arrays showed before cross PCIe (bit-identical to a full download); wall "
                  "clock over all frames incl. the final drain",
           "dense_value": world * e2e_frames / dense_s, "dense_d2h_bytes_per_step": 28 * RES * RES,
           "dense_api": "same pipeline with sparse=False: cudaMemcpy of all three buffers (29.4 MB) every frame",
           "image_u8_value": world * e2e_frames / img_s, "image_u8_d2h_bytes_per_step": 3 * RES * RES,
           "image_u8_api": "HostImagePipeline.submit: pinned [3,T,3,3] block in, run.py:26's flipped uint8 image (3 B/pixel) in pinned "
                           "host memory out; the rasterizer writes the uint8 image itself, no float32 buffer is produced",
           "color_only_value": world * e2e_frames / col_s, "color_only_d2h_bytes_per_step": col_tiles * 32 * 32 * 12 / e2e_frames,
           "color_only_api": "the same pipeline fetching only the colour buffer (want=('color',)): what Renderer.render returns "
                             "and run.py consumes (renderer.py:49); z and normals stay on the device, as they do for a drop-in "
                             "caller that never calls get_z_buffer()/get_normals_buffer()", "color_only_lit_pixels": col_cov,
           "synchronous_value": world * e2e_frames / sync_s,
           "synchronous_api": "crb_render_host, one frame per call, full download, stream-synchronised before returning",
           "pcie_floor_note": "a full 29.4 MB download per frame bounds the dense variants at ~1.9 k frames/s on a 55 GB/s link"}

    # ---- single frame through a CUDA graph (config C1: one render_model per frame, fresh buffers) -----------------
    single = None
    try:
        g = torch.cuda.CUDAGraph()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(3):
                _lib.check(L.crb_render(h, dv.data_ptr(), dc.data_ptr(), dn.data_ptr(), T, _lib.CRB_CLEAR_FIRST, f._stream()))
            torch.cuda.synchronize()
            with torch.cuda.graph(g, stream=s):
                _lib.check(L.crb_render(h, dv.data_ptr(), dc.data_ptr(), dn.data_ptr(), T, _lib.CRB_CLEAR_FIRST, f._stream()))
            for _ in range(5):
                g.replay()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 500
            a.record()
            for _ in range(reps):
                g.replay()
            b.record()
            torch.cuda.synchronize()
            us = a.elapsed_time(b) * 1000.0 / reps
        torch.cuda.current_stream().wait_stream(s)
        single = {"us_per_frame": us, "frames_per_s": 1e6 / us, "how": "crb_render(CLEAR_FIRST) captured in a CUDA graph, "
                  f"{reps} replays, device-resident inputs, L2-resident buffers (29 MB frame < 126 MB L2)"}
    except Exception as ex:  # graph capture is an extra, never fatal
        single = {"error": str(ex)[:200]}

    # ---- the literal reference usage (run.py:20-26 idiom): host model in, host NumPy buffers out, synchronous ------------
    drop_in = None
    if rank == 0:
        from conftest import TriModel
        vk, nk = VW.transform_arrays_host(views_np[0], model._vertices_by_triangles, model._normals_by_triangles)
        mk = TriModel(vk, model._colors_by_triangles, nk)

        def per_frame(fn, nrep=20):
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            t0_ = time.perf_counter()
            for _ in range(nrep):
                fn()
            torch.cuda.synchronize()
            return (time.perf_counter() - t0_) / nrep * 1e3

        def new_filler():
            ff = AdvancedPixelBufferFiller(RES, RES, fov=FOV, n_threads=8, device=local)
            ff.render_model(mk)
            return ff.get_color_buffer(), ff.get_normals_buffer(), ff.get_z_buffer()
        fr = AdvancedPixelBufferFiller(RES, RES, fov=FOV, device=local)

        def reused():
            fr.clear()
            fr.render_model(mk)
            return fr.get_color_buffer(), fr.get_normals_buffer(), fr.get_z_buffer()
        def new_filler_color_only():
            ff = AdvancedPixelBufferFiller(RES, RES, fov=FOV, n_threads=8, device=local)
            ff.render_model(mk)
            return ff.get_color_buffer()
        def renderer_flow():     # run.py:20-25 with this package's Renderer + GuroIllumination: the light on the device buffers
            from cython3dmodelrenderer_b200 import GuroIllumination, Renderer
            ff = AdvancedPixelBufferFiller(RES, RES, fov=FOV, n_threads=8, device=local)
            return Renderer(ff, GuroIllumination([0, 0, 1]), None, RES, RES).render(mk)
        try:
            renderer_ms = per_frame(renderer_flow)
        except Exception as ex:      # (must never take the headline line down)
            renderer_ms = repr(ex)[:200]
        drop_in = {"new_filler_per_frame_ms": per_frame(new_filler), "one_filler_clear_render_get3_ms": per_frame(reused),
                   "new_filler_color_only_ms": per_frame(new_filler_color_only),
                   "renderer_guro_new_filler_ms": renderer_ms,
                   "renderer_guro_what": "Renderer(filler, GuroIllumination([0, 0, 1]), ...).render(model) of this package, a new filler "
                                         "per frame: rasterizer + crb_guro on the device, the lit colour buffer (12.6 MB) downloaded; "
                                         "cpu_baseline.renderer_guro_ms is the reference's own three classes on the host",
                   "pcie_floor_ms": {"three_buffers": 28 * RES * RES / 55e6, "color_only": 12 * RES * RES / 55e6,
                                     "note": "dense float32 download at the ~55 GB/s this link sustains"},
                   "what": "AdvancedPixelBufferFiller(...).render_model(model) + the three get_*_buffer() calls on host NumPy data, "
                           "synchronous, full 29.4 MB download (the unmodified run.py flow with the import swapped)"}
        del fr

    cpu, cpu_threads = None, None
    if rank == 0 and world == 1 and not args.no_cpu:
        kind, cores, times = cpu_frames(model, n_total, frames=args.cpu_frames)
        cpu = {"value": len(times) / sum(times), "unit": "frames/s", "cores": cores, "host_cores": os.cpu_count(), "kind": kind,
               "sample": f"{len(times)} frames cycling through 8 evenly spread views (k * {n_total} / 8) of the orbit after 2 warm-ups, "
                         f"render_model only, fresh filler per frame, n_threads={cores} (the fastest of 8/16/32/nproc/2/nproc on this "
                         f"host, nproc={os.cpu_count()})", "median_ms": 1000 * statistics.median(times)}
        cpu_threads = cores
        try:
            cpu["renderer_guro_ms"] = reference_renderer_flow_ms(model, cores)
        except Exception as ex:
            cpu["renderer_guro_ms"] = repr(ex)[:200]

    # ---- the other BASELINE.json configs, measured in the same run (C2, C3: one GPU; C4: row bands over the N ranks) ----------
    secondary = None
    if not args.no_secondary:
        del z, col, nrm, f
        torch.cuda.empty_cache()
        secondary = {}
        for wl in (("bunny_4096_guro", "basketball_2048", "sphere_8192_bands") if world == 1 else ("sphere_8192_bands",)):
            try:
                if world > 1:
                    # the frame twice: bands left where they are rendered, and the complete frame on rank 0 (PeerFrame)
                    for mode in ("none", "peer", "u8_peer"):
                        a2 = argparse.Namespace(**vars(args)); a2.gather = mode
                        ln = measure_workload(a2, wl, world, rank, local, dev, cpu_threads, with_cpu=False)
                        if rank == 0:
                            secondary[wl + {"none": "", "peer": "_complete_on_rank0", "u8_peer": "_u8_image_complete_on_rank0"}[mode]] = ln
                else:
                    secondary[wl] = measure_workload(args, wl, world, rank, local, dev, cpu_threads)
                    if wl == "sphere_8192_bands":      # the single-GPU rate of the image-only frame, the base of the N-GPU u8 lines
                        a2 = argparse.Namespace(**vars(args)); a2.gather = "u8_local"
                        secondary[wl + "_u8_image"] = measure_workload(a2, wl, world, rank, local, dev, cpu_threads, with_cpu=False)
            except Exception as ex:
                secondary[wl] = {"error": repr(ex)[:300]}
            torch.cuda.empty_cache()

    if rank == 0:
        line = {
            "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic orbit of the T-Rex fixture (tests/golden/trex_fit.npz = README fit_model flow)",
            "config": headline_config(T, V, n_total, args.chunk),
            "gtri_per_s": fps * T / 1e9, "clocks": clocks.summary(), "e2e": e2e, "gpu_launches": launches,
            "roofline": roofline, "cpu_baseline": cpu, "single_frame": single, "drop_in": drop_in, "gather": gather, "secondary": secondary,
            "checks": {"covered_pixels_view0": covered0, "e2e_covered_pixels": e2e_cov, "e2e_image_u8_lit_pixels": img_cov, "e2e_dense_covered_pixels": dense_cov, "e2e_sync_covered_pixels": sync_cov, "pairs_last_launch": int(need.value),
                       "pair_capacity": int(cap.value)},
        }
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# --------------------------------------------------------------------------------------------------------------------
# secondary workloads (not the headline line): BASELINE.json configs C2, C3 and C4
# --------------------------------------------------------------------------------------------------------------------
def init_dist():
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    bind_rank_to_cpus(local, int(os.environ.get("LOCAL_WORLD_SIZE", str(world))))
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    return world, rank, local, torch.device("cuda", local)


def bind_rank_to_cpus(local, local_world):
    """One process per GPU: each rank gets its own slice of the CPUs nearest its GPU (`nvidia-smi topo -m`, column "CPU
    Affinity"; all allowed CPUs if that cannot be read), BEFORE any pinned buffer is allocated -- page-locked memory is placed on
    the NUMA node of the thread that touches it first, and eight ranks submitting from the same few cores serialise."""
    if local_world <= 1 or not hasattr(os, "sched_setaffinity"):
        return None
    try:
        allowed = sorted(os.sched_getaffinity(0))
        near = None
        try:
            txt = subprocess.run(["nvidia-smi", "topo", "-m"], capture_output=True, text=True, timeout=20).stdout
            for ln in txt.splitlines():
                cells = ln.split("\t") if "\t" in ln else ln.split()
                if cells and cells[0].strip() == f"GPU{local}":
                    for cell in cells[1:]:
                        cell = cell.strip()
                        if cell and all(ch.isdigit() or ch in ",-" for ch in cell) and any(ch.isdigit() for ch in cell) and ("-" in cell or "," in cell):
                            cpus = set()
                            for part in cell.split(","):
                                lo, _, hi = part.partition("-")
                                cpus.update(range(int(lo), int(hi or lo) + 1))
                            near = sorted(cpus & set(allowed))
                            break
        except Exception:
            near = None
        pool = near or allowed
        # ranks whose GPUs share the same CPU set split it evenly
        per = max(1, len(pool) // local_world)
        mine = pool[(local * per) % len(pool):][:per] or pool
        os.sched_setaffinity(0, mine)
        return mine
    except Exception:
        return None


WORKLOADS = {
    # name: (BASELINE.json config, fixture / generator, resolution, fused Guro light, CPU frames in the cpu_baseline sample)
    "bunny_4096_guro": ("C2", "bunny", 4096, True, 3),
    "basketball_2048": ("C3", "basketball", 2048, False, 5),
    "sphere_8192_bands": ("C4", "sphere", 8192, False, 1),
}


def measure_workload(args, workload, world, rank, local, dev, cpu_threads=None, with_cpu=True):
    """One frame per step of a secondary config: bunny_4096_guro (C2: bunny + igor texture, 4096^2, fused clear + render + Guro
    pass), basketball_2048 (C3 substitute: the quad-faced, textured basketball at 2048^2) -- one GPU each (replicas only) -- and
    sphere_8192_bands (C4: 10 M-triangle UV sphere at 8192^2, screen-row bands over the N ranks, the complete frame either
    staying where it is rendered, all-gathered by NCCL or written straight into rank 0's memory over NVLink).  Returns, on
    rank 0, a dict shaped like the headline line (value, roofline of k_raster, cpu_baseline and e2e at N = 1)."""
    import torch
    import torch.distributed as dist
    from conftest import TriModel, load_indexed
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller, sharding, synthetic
    from cython3dmodelrenderer_b200 import views as VW

    cfg, source, res0, guro, cpu_n = WORKLOADS[workload]
    banded = source == "sphere"
    if banded:
        res = args.res or res0
        scale = res / 8192.0
        model = synthetic.uv_sphere(max(8, int(3200 * scale)), max(3, int(1564 * scale)))
        band = sharding.band_shard(res, rank, world)
        bands = [sharding.band_shard(res, r, world) for r in range(world)]
    else:
        res, model, band, bands = res0, load_indexed(source), None, None
        if rank != 0:
            return None              # replicas only: nothing to shard, rank 0 measures
    T = int(model._vertices_by_triangles.shape[0])
    dv, dc, dn = (torch.from_numpy(a).to(dev) for a in
                  (model._vertices_by_triangles, model._colors_by_triangles, model._normals_by_triangles))
    if banded and world > 1 and args.bands == "balanced":
        # cut the frame where the estimated cost (triangles per 32-row strip) balances, not into equal row counts: the
        # sphere's poles hold far more triangles per row than its equator.  Rank 0 decides, everybody follows.
        costs = [float(x) for x in sharding.tile_row_costs(dv, dn, res, res, FOV)] if rank == 0 else None
        box = [sharding.balanced_bands(costs, world, res) if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        bands = box[0]
        # ... and the estimate is corrected by what the bands really cost: three rounds of (render a few frames, compare the
        # ranks' times, cut again) -- load balancing before the timed region, like the choice of the bands itself
        # (the cut that measured best is kept: a re-cut can also land on the wrong side of a threshold, e.g. of the band pre-pass)
        tried = []
        for rnd in range(4):
            fcal = AdvancedPixelBufferFiller(res, res, fov=FOV, device=local, band=bands[rank])
            for _w in range(2):
                fcal.clear(); fcal.render_arrays(dv, dc, dn)
            torch.cuda.synchronize(); dist.barrier()
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record()
            for _w in range(4):
                fcal.clear(); fcal.render_arrays(dv, dc, dn, check_status=False)
            c1.record(); torch.cuda.synchronize()
            mine = torch.tensor([c0.elapsed_time(c1) / 4], dtype=torch.float64, device=dev)
            every = [torch.zeros_like(mine) for _r in range(world)]
            dist.all_gather(every, mine)
            del fcal
            if rank == 0:
                times = [float(t.item()) for t in every]
                tried.append((max(times), bands))
                if rnd < 3:
                    new_bands, costs = sharding.rebalance_bands(costs, bands, times, world, res)
                else:
                    new_bands = min(tried, key=lambda tb: tb[0])[1]
                box = [new_bands]
            dist.broadcast_object_list(box, src=0)
            bands = box[0]
        band = bands[rank]
    gather_mode = args.gather if banded and (world > 1 or args.gather == "u8_local") else "none"
    if gather_mode == "auto":
        gather_mode = "peer"
    frame = image = None
    if banded and world > 1 and gather_mode == "u8_peer":
        # run.py's product (the flipped uint8 image) complete on rank 0: every rank's rasterizer stores its band's image rows
        # straight into rank 0's memory (sharding.PeerImage); no float32 buffer is produced
        image = sharding.PeerImage(res, res, dst=0, local_device=local)
        f = AdvancedPixelBufferFiller(res, res, fov=FOV, device=local, band=band)
    elif banded and world > 1 and gather_mode == "peer":
        frame = sharding.PeerFrame(res, res, dst=0, local_device=local)
        f = AdvancedPixelBufferFiller(res, res, fov=FOV, device=local, band=band, out_ptrs=frame.band_pointers(band[0]))
    else:
        f = AdvancedPixelBufferFiller(res, res, fov=FOV, device=local, band=band if (banded and world > 1) else None)
    ident = torch.from_numpy(VW.view_matrix()[None, :]).to(dev)     # identity rotation, zero pivot / translation
    zb, cb, nb_ = f.device_buffers()

    u8_local = torch.empty((1, res, res, 3), dtype=torch.uint8, device=dev) if (gather_mode == "u8_local") else None

    def step():
        if image is not None:
            f.render_views(dv, dc, dn, ident, want=(), chunk=1, check_status=False, u8_exchange=image.plan(band))
        elif u8_local is not None:
            f.render_views(dv, dc, dn, ident, want=(), color_u8_out=u8_local, chunk=1, check_status=False)
        elif guro:
            # one frame = fused clear + raster + shading with the Guro light applied in the shading pass (CRB_GURO),
            # written straight into the filler's own buffers (identity view: x*1 + 0 terms are exact)
            f.render_views(dv, dc, dn, ident, z_out=zb[None], color_out=cb[None], normals_out=nb_[None], guro_light=[0, 0, 1],
                           chunk=1, check_status=False)
        else:
            f.clear()
            f.render_arrays(dv, dc, dn, check_status=False)

    def barrier():
        torch.cuda.synchronize()
        if world > 1 and banded:
            dist.barrier()
        torch.cuda.synchronize()

    f.clear(); f.render_arrays(dv, dc, dn); f.device_buffers()       # sizes the workspace, checks the pair list
    steps = args.steps
    for _ in range(3):
        step()
    barrier()
    launches0 = f.launch_count
    f.profile(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clocks:
        barrier()
        e0.record()
        for _ in range(steps):
            step()
        if frame is not None:
            pass        # (the stores into rank 0's frame are complete when this rank's stream has drained: barrier below)
        e1.record()
        clocks.sample_now()
        barrier()
    ms_own = e0.elapsed_time(e1)
    ms = ms_own
    k_launches, k_ms = f.profile_read()
    f.profile(False)
    launches = f.launch_count - launches0
    gather = None
    if banded and world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        if image is not None:
            gather = {"mode": "u8_peer", "ms": 0.0, "bytes": 3 * res * res,
                      "what": "none needed: every rank's rasterizer stores its band of run.py's flipped uint8 image straight into rank "
                              "0's memory over NVLink (sharding.PeerImage, crb_set_u8_exchange); `value` is complete images per second on "
                              "rank 0; no float32 buffer is produced",
                      "lit_pixels": int((image.tensor().sum(dim=-1) > 0).sum().item()) if rank == 0 else None}
        elif frame is not None:
            full_z = frame.tensors()[0]
            gather = {"mode": "peer", "ms": 0.0, "bytes": 28 * res * res,
                      "what": "none needed: every rank's rasterizer stores its band straight into rank 0's frame over NVLink "
                              "(sharding.PeerFrame); `value` is complete frames per second on rank 0",
                      "covered_pixels": int((full_z < 1e5).sum().item()) if rank == 0 else None}
        elif gather_mode in ("bands", "all"):     # final NCCL all-gather of the row bands (north_star: "a final NCCL gather over NVLink")
            z, c, n = f.device_buffers()
            for b_ in (z, c, n):                     # first use of the communicator / buffers is not what is being timed
                sharding.gather_bands(b_, res, bands=bands)
            barrier()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            full = [sharding.gather_bands(b_, res, bands=bands) for b_ in (z, c, n)]
            g1.record()
            barrier()
            gms = torch.tensor([g0.elapsed_time(g1)], dtype=torch.float64, device=dev)
            dist.all_reduce(gms, op=dist.ReduceOp.MAX)
            gather = {"mode": "nccl_all_gather", "ms": float(gms.item()), "bytes": 28 * res * res,
                      "what": "all_gather_into_tensor of the z + colour + normal row bands after the frame (every rank ends with the whole frame)",
                      "frames_per_s_including_gather": 1000.0 / (ms / steps + float(gms.item())),
                      "covered_pixels": int((full[0] < 1e5).sum().item())}
            del full
    z = f.device_buffers()[0]
    if image is not None or u8_local is not None:        # (the timed steps produced no float32 buffer: draw one frame for the check)
        f.clear(); f.render_arrays(dv, dc, dn)
        z = f.device_buffers()[0]
    cov = torch.tensor([int((z < 1e5).sum().item())], dtype=torch.int64, device=dev)   # (PeerFrame: read over NVLink)
    if banded and world > 1:
        dist.all_reduce(cov)
    fps = steps / (ms / 1000.0)
    peak, peak_src = peaks()
    rows = res if not (banded and world > 1) else band[1] - band[0]
    bpp = 3 if (image is not None or u8_local is not None) else 28       # image-only frames write 3 bytes per pixel
    alg = 108 * T + bpp * rows * res      # per GPU: every rank reads all triangles, writes its own rows
    k_avg = k_ms / max(k_launches, 1)

    cpu = e2e = None
    if rank == 0 and world == 1 and with_cpu and not args.no_cpu:
        # host Version C on the same frame (the reference build where it exists): fresh filler per frame, render_model only --
        # plus, for C2, the reference's own GuroIllumination pass over the result (renderer.py:48)
        kind, cores, render = cpu_reference_runner(cpu_threads, res=res, fov=FOV)
        times = [render(model._vertices_by_triangles, model._colors_by_triangles, model._normals_by_triangles) for _ in range(cpu_n)]
        cpu = {"value": len(times) / sum(times), "unit": "frames/s", "cores": cores, "host_cores": os.cpu_count(), "kind": kind,
               "sample": f"{len(times)} frame(s), render_model only, fresh pre-touched filler per frame, n_threads={cores}",
               "median_ms": 1000 * statistics.median(times)}
        # e2e: the drop-in idiom on host arrays -- a new filler, render_model, the three get_*_buffer (dense download)
        m_host = TriModel(model._vertices_by_triangles, model._colors_by_triangles, model._normals_by_triangles)

        def drop_in_frame():
            ff = AdvancedPixelBufferFiller(res, res, fov=FOV, n_threads=8, device=local)
            ff.render_model(m_host)
            if guro:
                ff.illuminate_guro(np.float32([0, 0, -1]))
            return ff.get_color_buffer(), ff.get_normals_buffer(), ff.get_z_buffer()
        nrep = 3 if res >= 8192 else 8
        t_first = time.perf_counter()
        out = drop_in_frame()                   # the first frames of a process page-lock their host mirrors (cudaHostAlloc,
        first_ms = (time.perf_counter() - t_first) * 1e3      # ~0.55 ms per MB, reported as first_frame_ms); a render loop then
        for _ in range(2):                      # alternates between two cached sets: steady state from the third frame on
            out = drop_in_frame()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(nrep):
            out = drop_in_frame()
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / nrep
        e2e = {"value": 1.0 / dt, "unit": "frames/s", "h2d_bytes_per_step": 108 * T, "d2h_bytes_per_step": 28 * res * res,
               "api": "AdvancedPixelBufferFiller(...).render_model(model) + get_color/normals/z_buffer() on host NumPy arrays, a new "
                      "filler per frame, synchronous" + (" (+ illuminate_guro before the reads)" if guro else "") +
                      "; steady state of a render loop (frames 4.. of the process)", "first_frame_ms": first_ms, "frames_timed": nrep,
               "covered_pixels": int((out[2] < 1e5).sum())}
        del out
        if guro:      # the reference's render() flow (renderer.py:47-49) with this package's Renderer + GuroIllumination: lit colour only
            try:
                from cython3dmodelrenderer_b200 import GuroIllumination, Renderer

                def renderer_frame():
                    ff = AdvancedPixelBufferFiller(res, res, fov=FOV, n_threads=8, device=local)
                    return Renderer(ff, GuroIllumination([0, 0, 1]), None, res, res).render(m_host)
                for _ in range(3):
                    renderer_frame()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(nrep):
                    renderer_frame()
                torch.cuda.synchronize()
                e2e["renderer_guro_value"] = nrep / (time.perf_counter() - t0)
                e2e["renderer_guro_d2h_bytes_per_step"] = 12 * res * res
                cpu["renderer_guro_ms"] = reference_renderer_flow_ms(model, cores, frames=2, res=res)
            except Exception as ex:
                e2e["renderer_guro_value"] = repr(ex)[:200]

    line = None
    if rank == 0:
        line = {
            "metric": f"{workload} frames/s", "value": fps, "unit": "frames/s", "n_gpus": world if banded else 1, "steps": steps,
            "warmup": 3, "ms_per_step": ms / steps, "higher_is_better": True,
            "scaling": "strong" if (banded and world > 1) else "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic UV sphere (SURVEY 8d C4)" if banded else f"{source} fixture + igor texture (tests/golden/{source}_fit.npz)",
            "config": {"workload": workload, "baseline_config": cfg, "res": res, "fov": FOV, "triangles": T, "illumination": bool(guro),
                       "sharding": (f"screen-row bands, tile aligned, {args.bands}: {bands}") if (banded and world > 1) else "none (replicas only)",
                       "l2": "frame buffers %.2f GB per GPU vs 126 MB L2" % (28 * rows * res / 1e9)},
            "gtri_per_s": fps * T / 1e9, "clocks": clocks.summary(), "gpu_launches": launches,
            "roofline": {"bound": "hbm", "kernel": "k_raster", "achieved": alg / (k_avg / 1000.0) / 1e9 if k_avg else None,
                         "peak": peak, "unit": "GB/s",
                         # (a band-sharded rank rasterizes only the triangles its pre-pass listed: 108 T bytes per rank would
                         # overstate what rank 0's small pole band reads, so the fraction is given for whole frames only)
                         "frac": (alg / (k_avg / 1000.0) / 1e9 / peak) if (k_avg and not (banded and world > 1)) else None,
                         "band_note": ("rank 0's k_raster on its own band; `achieved` counts 108 B for every triangle of the frame "
                                       "although the band pre-pass hands k_raster only the chunks that reach the band") if (banded and world > 1) else None,
                         "traffic": None, "peak_source": peak_src, "avg_launch_ms": k_avg,
                         "algorithmic_bytes_per_launch": alg, "share_of_step": k_ms / ms_own if ms_own else None},
            "cpu_baseline": cpu, "e2e": e2e, "gather": gather, "checks": {"covered_pixels": int(cov.item())},
        }
    del f
    if frame is not None:
        frame.close()
    if image is not None:
        image.close()
    return line


def run_extra_workload(args):
    import torch.distributed as dist
    world, rank, local, dev = init_dist()
    line = measure_workload(args, args.workload, world, rank, local, dev)
    if rank == 0 and line is not None:
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


_REAL_STDOUT = None
_T_START = time.time()
_PARTIAL = {}          # rank 0: the headline fields, as soon as they are measured (see start_watchdog)
_EMITTED = False


def start_watchdog(budget_s):
    """Last resort, never reached by a healthy run (the default run takes a minute or two): the legs after the headline exchange
    data between ranks (NCCL, peer mappings), and a rank that fails inside one leaves the others waiting in a collective until the
    driver's limit kills the job with nothing printed.  After `budget_s` seconds of process time every rank leaves; rank 0 first
    prints the headline it has already measured, marked "truncated"."""
    def fire():
        if not _EMITTED and int(os.environ.get("RANK", "0")) == 0 and _PARTIAL:
            line = dict(_PARTIAL)
            line["truncated"] = f"watchdog: a leg after the headline did not finish within {budget_s:.0f} s of process time"
            emit(line)
        os._exit(0 if (_EMITTED or int(os.environ.get("RANK", "0")) != 0) else 3)
    t = threading.Timer(budget_s, fire)
    t.daemon = True
    t.start()
    return t


def emit(line):
    """The JSON line goes to the process's original stdout; everything else (NCCL banners, library chatter) was sent to
    stderr by main()."""
    global _EMITTED
    line.setdefault("wall_s", round(time.time() - _T_START, 1))    # process start -> this line (imports, fixtures, every leg)
    _EMITTED = True
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)          # anything a library prints on fd 1 (e.g. "NCCL version ...") must not precede the JSON line
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--views", type=int, default=128, help="views per GPU per step")
    ap.add_argument("--chunk", type=int, default=128, help="views per kernel launch (larger launches amortise the kernel tail: 32 -> 93 k, 128 -> 98 k frames/s)")
    ap.add_argument("--e2e-frames", type=int, default=200)
    ap.add_argument("--e2e-depth", type=int, default=6, help="fillers in flight in the pipelined e2e measurement (4: 5 700, 6: 6 275, 8: 6 140, 12: 6 140 frames/s)")
    ap.add_argument("--cpu-frames", type=int, default=60)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--workload", default="trex_1024_orbit",
                    choices=["trex_1024_orbit", "bunny_4096_guro", "basketball_2048", "sphere_8192_bands"])
    ap.add_argument("--bands", default="balanced", choices=["balanced", "uniform"],
                    help="sphere_8192_bands only: rows per rank equal (uniform) or cut where the estimated cost balances")
    ap.add_argument("--res", type=int, default=0, help="sphere_8192_bands only: override the resolution (scaled sphere)")
    ap.add_argument("--no-secondary", action="store_true", help="skip the C2 / C3 / C4 lines measured after the headline")
    ap.add_argument("--gather", default="auto", choices=["auto", "none", "bands", "u8", "z", "exchange", "exchange_nccl", "u8_peer", "u8_local", "all", "peer"],
                    help="also time the final NCCL gather (reported beside, never inside, the headline value); "
                         "peer (sphere_8192_bands only): no gather at all -- every rank's filler renders its band straight into "
                         "rank 0's frame over NVLink (sharding.PeerFrame), and the value is frames/s complete on rank 0")
    ap.add_argument("--budget-s", type=float, default=float(os.environ.get("CRB_BENCH_BUDGET_S", "720")),
                    help="watchdog: leave (rank 0 printing the headline it has) after this many seconds; 0 = off")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one rendered (z, colour, normals: view 0 whole and a seeded "
                         "pixel sample of all views) as float32 .npy files into DIR; rank 0 writes its own views, so compare "
                         "dumps taken with the same number of ranks and --views")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload != "trex_1024_orbit"):
        ap.error("--dump-outputs applies to the headline run (--impl b200, --workload trex_1024_orbit)")
    if args.budget_s > 0:
        start_watchdog(args.budget_s)
    if args.impl == "reference":
        run_reference_arm(args)
    elif args.workload != "trex_1024_orbit":
        run_extra_workload(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
