"""Per-phase warp-cycle split of k_raster (needs csrc/libcrender_b200_timing.so = the library built with -DCRB_PHASE_TIMING)."""
import ctypes, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
os.environ["CRB_LIB_OVERRIDE"] = os.path.join(ROOT, "cython3dmodelrenderer_b200", "csrc", "libcrender_b200_timing.so")
import torch
from conftest import load_indexed
from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller, views as VW, _lib
name = sys.argv[1] if len(sys.argv) > 1 else "trex"
res = int(sys.argv[2]) if len(sys.argv) > 2 else 1024
V = int(sys.argv[3]) if len(sys.argv) > 3 else 32
m = load_indexed(name)
dv, dc, dn = (torch.from_numpy(a).cuda() for a in (m._vertices_by_triangles, m._colors_by_triangles, m._normals_by_triangles))
views = torch.from_numpy(VW.orbit_views(128, 0, V)).cuda()
f = AdvancedPixelBufferFiller(res, res, fov=45.0)
out = f.render_views(dv, dc, dn, views, chunk=V)
for _ in range(3):
    f.render_views(dv, dc, dn, views, chunk=V, z_out=out["z"], color_out=out["color"], normals_out=out["normals"])
torch.cuda.synchronize()
ph = (ctypes.c_uint64 * 16)()
_lib.check(f._L.crb_phase_cycles(ph, 1))
N = 5
for _ in range(N):
    f.render_views(dv, dc, dn, views, chunk=V, z_out=out["z"], color_out=out["color"], normals_out=out["normals"], check_status=False)
torch.cuda.synchronize()
_lib.check(f._L.crb_phase_cycles(ph, 1))
names = {0: "head+clears", 2: "keys init / chunk barrier", 3: "staging+scan+owner", 4: "barrier after staging", 5: "row loop (visibility)",
         6: "barrier before shading", 7: "shading loop", 9: "uint8 row output"}
tot = sum(ph)
print(f"{name} {res}^2 x {V} views: warp-cycles per view {tot / N / V:.0f}")
for k, nm in names.items():
    print(f"  {nm:28s} {100.0 * ph[k] / tot:5.1f}%   {ph[k] / N / V:12.0f} warp-cycles/view")
