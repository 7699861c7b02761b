#!/usr/bin/env python
"""Turns the scratch captures under gpurun_out/ into the tracked summaries under profiles/ (run here, after a gpurun call):
  gpurun_out/<tag>_kr_{trex,sphere,bunny}.ncu-rep  ->  profiles/<tag>_k_raster_{raw,phases,lines}_<workload>.txt, <tag>_k_raster_traffic.json
  gpurun_out/<tag>_launches_bench.csv              ->  profiles/<tag>_launches_bench.csv + <tag>_launches_summary.txt
usage: tools/make_profile_summaries.py r02"""
import collections, csv, io, json, os, re, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
tag = sys.argv[1] if len(sys.argv) > 1 else "r02"
G, P, T = os.path.join(ROOT, "gpurun_out"), os.path.join(ROOT, "profiles"), os.path.join(ROOT, "tools")
SRC = os.path.join(ROOT, "cython3dmodelrenderer_b200", "csrc", "crender_b200.cu")


def phase_ranges():
    """Line ranges of k_raster's phases, found from markers in the source (so the table survives edits)."""
    src = open(SRC).read().splitlines()
    def find(pat, start=0):
        for i in range(start, len(src)):
            if re.search(pat, src[i]):
                return i + 1
        raise SystemExit("marker not found: " + pat)
    rt = find(r"void raster_tile\(")
    vis = find(r"---- visibility:", rt)
    trip = find(r"unsigned qn = 0, trip = 0;", vis)
    pass1 = find(r"// pass 1: which pixels", trip)
    pub = find(r"__syncwarp\(\);\s+// the slots are published", pass1)
    ev = find(r"const bool flush =", pub)
    left = find(r"if \(b\) \{\s+// what is left", ev)
    shade = find(r"---- deferred shading", left)
    out = find(r"^\s+PH\(7\);", shade)
    end = find(r"^// The fused clear through TMA", out)
    kr = find(r"^__global__ void __launch_bounds__\(C::RT, C::MIN_CTAS\) k_raster")
    kend = find(r"^// The two shapes of the tile rasterizer", kr)
    sf = find(r"bool shade_fragment\("); sfe = find(r"^// Colour of a pixel no triangle covers", sf)
    dv = find(r"float div_rn_by\("); dve = find(r"^// pyx:215-242", dv)
    km = find(r"void smem_key_min\("); kme = find(r"^// Tensor maps", km)
    dk = find(r"unsigned depth_key\("); dke = find(r"^// mu:5-34", dk)
    sb = find(r"void span_bound\("); sbe = find(r"^// bits of a staged triangle", sb)
    sc = find(r"unsigned block_exclusive_scan\("); sce = find(r"^__global__ void __launch_bounds__\(NT\) k_alloc", sc)
    return [("head (CTA prologue, roles, clear CTAs)", [(kr, kend - 1), (rt, vis - 1)]),
            ("staging + row scan", [(vis, trip - 1), (sc, sce - 1)]),
            ("row set-up", [(trip, pass1 - 1)]),
            ("span pass", [(pass1, pub - 1), (sb, sbe - 1)]),
            ("compaction (queue)", [(pub, ev - 1)]),
            ("exact pass", [(ev, left - 1), (dv, dve - 1), (km, kme - 1), (dk, dke - 1)]),
            ("queue leftovers", [(left, shade - 1)]),
            ("shading", [(shade, out - 1), (sf, sfe - 1)]),
            ("row output (staged uint8 image)", [(out, end - 1)])]


def run(cmd):
    return subprocess.run(cmd, capture_output=True, text=True).stdout


def raster_reports():
    for wl in ("trex", "sphere", "bunny"):
        rep = os.path.join(G, f"{tag}_kr_{wl}.ncu-rep")
        if os.path.exists(rep):
            yield wl, rep


WL = {"trex": "128 T-Rex views at 1024^2 in one launch", "sphere": "10 M-triangle sphere at 8192^2, one frame", "bunny": "bunny at 4096^2, one frame"}
traffic = {}
for wl, rep in raster_reports():
    hdr = f"# k_raster, {WL[wl]}: ncu --set full --clock-control none --import-source on (tools/scratch/prof_trex128.py {wl}), launch 3\n"
    open(os.path.join(P, f"{tag}_k_raster_raw_{wl}.txt"), "w").write(hdr + run([sys.executable, os.path.join(T, "ncu_key.py"), rep]))
    specs = [name.split(" (")[0].replace(" ", "_") + ":" + ",".join(f"{a}-{b}" for a, b in rg) for name, rg in phase_ranges()]
    open(os.path.join(P, f"{tag}_k_raster_phases_{wl}.txt"), "w").write(
        hdr + "# warp instructions by phase (source line ranges of crender_b200.cu found by tools/make_profile_summaries.py)\n" +
        run([sys.executable, os.path.join(T, "ncu_ranges.py"), rep, "0"] + specs))
    open(os.path.join(P, f"{tag}_k_raster_lines_{wl}.txt"), "w").write(hdr + run([sys.executable, os.path.join(T, "ncu_lines.py"), rep, "0", "60"]))
    raw = list(csv.reader(io.StringIO(run(["ncu", "-i", rep, "--page", "raw", "--csv"]))))
    h, u, r = raw[0], raw[1], raw[2]
    def val(name):
        v = float(r[h.index(name)].replace(",", "")); unit = u[h.index(name)]
        return v * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1, "ms": 1e3, "us": 1, "ns": 1e-3}.get(unit, 1)
    traffic[wl] = {"launch": WL[wl], "grid": r[h.index("Grid Size")], "dram_bytes_read": val("dram__bytes_read.sum"),
                   "dram_bytes_write": val("dram__bytes_write.sum"), "dram_bytes_per_launch": val("dram__bytes_read.sum") + val("dram__bytes_write.sum"),
                   "gpu_time_us_under_ncu": val("gpu__time_duration.sum"), "warp_instructions": val("smsp__inst_executed.sum"),
                   "issue_active_pct": val("smsp__issue_active.avg.pct_of_peak_sustained_active"),
                   "lsu_data_pipe_pct": val("l1tex__data_pipe_lsu_wavefronts.avg.pct_of_peak_sustained_elapsed"),
                   "dram_throughput_pct": val("gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed"),
                   "source": f"gpurun_out/{os.path.basename(rep)} (scratch; ncu --set full --clock-control none --import-source on)"}
if traffic:
    alg = {"trex": 3949061120, "sphere": 2959393792, "bunny": 473038552}
    for wl in traffic:
        traffic[wl]["algorithmic_bytes_per_launch"] = alg[wl]
    out = dict(traffic.get("trex", {})); out["kernel"] = "k_raster"; out["other_workloads"] = {k: v for k, v in traffic.items() if k != "trex"}
    json.dump(out, open(os.path.join(P, f"{tag}_k_raster_traffic.json"), "w"), indent=1)

lc = os.path.join(G, f"{tag}_launches_bench.csv")
if os.path.exists(lc):
    rows = [r for r in csv.reader(open(lc)) if len(r) > 14 and r[0].isdigit()]
    open(os.path.join(P, f"{tag}_launches_bench.csv"), "w").write(open(lc).read())
    agg = collections.OrderedDict()
    for r in rows:
        name = re.sub(r"<unnamed>::", "", r[4]); key = (name, r[8])
        a = agg.setdefault(key, [0, 0.0]); a[0] += 1; a[1] += float(r[14]) / 1000.0
    with open(os.path.join(P, f"{tag}_launches_summary.txt"), "w") as fo:
        fo.write("ncu --metrics gpu__time_duration.sum --clock-control none -c 400, python bench.py --steps 2 --warmup 1 --no-cpu --no-secondary "
                 "(serialised, cold-cache per-launch times)\n")
        for (name, grid), (n, us) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
            fo.write(f"{name[:46]:46s} grid {grid:24s} launches {n:4d}  avg {us / n:8.1f} us  total {us / 1000:8.2f} ms\n")
print("profiles written for", tag, "->", sorted(f for f in os.listdir(P) if f.startswith(tag)))
