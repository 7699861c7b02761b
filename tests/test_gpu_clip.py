"""Near-plane clipping (CRB_CLIP_NEAR, AdvancedPixelBufferFiller(near_clip=True); DESIGN 2) on the GPU, word for word against
oracle/clip_oracle.py: the pieces of the clip rule rendered by the pinned oracles.

Covered: random scenes straddling z_near, the T-Rex with cameras inside and orbiting a centre near the camera, the edge
families, adversarial corners; the tiled and atomic paths, the three rasterizer shapes, TMA on and off, the host-array paths,
batched views with every chunking, the launch pipeline and defer_join, band fillers, the row exchange, supersampling, fused Guro,
every texture mode, the pipelines and the drop-in Renderer, compositing with id_base; the invariance of scenes nothing crosses;
the refusals and an overflowing frame.
"""
import ctypes

import numpy as np
import pytest

from conftest import TriModel, bits_equal, load_indexed, random_scene

F32 = np.float32
LIGHT = [0.3, -0.2, 1.0]
SENTINEL = 0x5EED1D5


def CL():
    from oracle import clip_oracle
    return clip_oracle


def _mv(m):
    return m._vertices_by_triangles, m._colors_by_triangles, m._normals_by_triangles


def _device(*arrays):
    import torch
    return tuple(torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays)


def _filler(h, w, fov, z_near=0.1, opts=None, **kw):
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller, _lib
    f = AdvancedPixelBufferFiller(h, w, fov=fov, z_near=z_near, **kw)
    for opt, val in (opts or {}).items():
        f.set_option(getattr(_lib, "CRB_OPT_" + opt), val)
    return f


def _words(got, want, what, nan_equal=False):
    got = got.cpu().numpy() if hasattr(got, "cpu") else np.asarray(got)
    got, want = np.ascontiguousarray(got), np.ascontiguousarray(want)
    assert got.shape == want.shape, f"{what}: shape {got.shape} != {want.shape}"
    if got.dtype.itemsize == 4:
        ok = got.view(np.uint32) == want.view(np.uint32)
        if nan_equal and got.dtype == np.float32:
            ok |= np.isnan(got) & np.isnan(want)
    else:
        ok = got == want
    if not ok.all():
        bad = np.argwhere(~ok)
        raise AssertionError(f"{what}: {len(bad)} words differ, first {bad[:5].tolist()}: got {got[tuple(bad[0])]!r} "
                             f"want {want[tuple(bad[0])]!r}")


def assert_frame(got, o, ids, what, rows=slice(None), nan_equal=False):
    """got = (z, color, normals[, tri_id]) against the oracle filler o and its tri_id"""
    for name, g, w in zip(("z", "color", "normals", "tri_id"), got,
                          (o.z_buffer[rows], o.color_buffer[rows], o.normals_buffer[rows], ids[rows].astype(np.int32))):
        _words(g, w, f"{what}: {name}", nan_equal)


def u8(colour):
    with np.errstate(invalid="ignore"):
        return np.ascontiguousarray(colour[::-1].astype("uint8"))


def lit(o):
    from oracle import oracle as O
    c = o.color_buffer.copy()
    O.guro(c, o.normals_buffer, LIGHT)
    return c


# ---------------------------------------------------------------------------------------------------------------- scenes
def straddling(seed, zn, T=400):
    """A random scene moved towards the camera so that many triangles cross z = zn and some lie behind the camera"""
    m = random_scene(seed, T=T)
    v = m._vertices_by_triangles.copy()
    v[..., 2] -= F32(1.5)
    return TriModel(v, m._colors_by_triangles, m._normals_by_triangles)


def _edges(h, w):
    import test_gpu_edges as E
    return E.concat(*(E.family(k, h, w) for k in "ABCDEFGH")), E.FOV


def adversarial(zn, T=600):
    from test_clip_oracle import adversarial as adv
    v, c, n = adv(7, T, zn)
    v[..., :2] *= F32(0.3)
    return TriModel(v, c, n)


def inside_views(V):
    """Cameras inside the T-Rex (look-at from points within its bounding box) and orbits about a centre near the camera"""
    from cython3dmodelrenderer_b200 import views as VW
    out = []
    for k in range(V):
        th = 2 * np.pi * k / V
        if k % 2 == 0:
            p = (-0.4 + 0.2 * np.cos(th), 0.02, 1.1 + 0.2 * np.sin(th))        # a point inside the model goes to the camera
            out.append(VW.view_matrix(VW.rot_y(th), p=p, q=(0.0, 0.0, 0.0)))
        else:
            out.append(VW.view_matrix(VW.rot_y(0.6 * np.sin(th)), p=(-0.2, 0.0, 0.35)))   # the model swings about a point near the camera
    return np.stack(out).astype(F32)


SCENES = {"straddle0_zn0.1": lambda: (straddling(0, 0.1), 90.0, 0.1, 256, 256),
          "straddle5_zn0.5": lambda: (straddling(5, 0.5), 90.0, 0.5, 256, 256),
          "straddle14_zn1": lambda: (straddling(14, 1.0), 90.0, 1.0, 256, 256),
          "edges256": lambda: _edges(256, 256) + (0.1, 256, 256),
          "edges200x333": lambda: _edges(200, 333) + (0.1, 200, 333),
          "adversarial": lambda: (adversarial(0.25), 90.0, 0.25, 128, 160)}
_CACHE = {}


def scene(name):
    if name not in _CACHE:
        m, fov, zn, h, w = SCENES[name]()
        o, ids = CL().render(h, w, *_mv(m), fov=fov, z_near=zn)
        _CACHE[name] = (m, fov, zn, h, w, o, ids)
    return _CACHE[name]


CONFIGS = {"default": {}, "atomic": {}, "shape1": {"RASTER_SHAPE": 1}, "shape2": {"RASTER_SHAPE": 2},
           "shape3": {"RASTER_SHAPE": 3}, "tma0": {"TMA": 0}}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(SCENES))
@pytest.mark.parametrize("config", sorted(CONFIGS))
def test_scenes_on_every_path(config, name):
    """Device inputs through crb_render: the tiled path in every shape, TMA on and off, and the atomic path"""
    m, fov, zn, h, w, o, ids = scene(name)
    f = _filler(h, w, fov, zn, CONFIGS[config], near_clip=True, triangle_ids=True)
    f.render_arrays(*_device(*_mv(m)), path="atomic" if config == "atomic" else "tiled")
    got = (f.get_z_buffer(), f.get_color_buffer(), f.get_normals_buffer(), f.get_triangle_id_buffer())
    assert_frame(got, o, ids, f"{name} {config}", nan_equal=name == "adversarial")
    assert (o.z_buffer < 1e6).sum() > 0


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["staged", "pageable", "sync", "no_sync"])
def test_host_array_paths(mode):
    """NumPy inputs: staged through pinned memory, the library's pageable ring (large arrays), and crb_render_host called
    synchronously and with CRB_NO_SYNC"""
    import torch
    from cython3dmodelrenderer_b200 import _lib
    if mode == "pageable":        # 20 shifted copies of the straddling scene: more than PAGEABLE_MIN_BYTES
        base = straddling(3, 0.1, T=12000)
        v = np.concatenate([base._vertices_by_triangles + F32(0.01 * k) for k in range(20)]).astype(F32)
        m = TriModel(v, np.tile(base._colors_by_triangles, (20, 1, 1)), np.tile(base._normals_by_triangles, (20, 1, 1)))
    else:
        m = straddling(3, 0.1)
    h, w = 256, 256
    o, ids = CL().render(h, w, *_mv(m), fov=90.0, z_near=0.1)
    f = _filler(h, w, 90.0, near_clip=True, triangle_ids=True)
    if mode in ("staged", "pageable"):
        f.render_arrays(*_mv(m))
        assert_frame((f.get_z_buffer(), f.get_color_buffer(), f.get_normals_buffer(), f.get_triangle_id_buffer()), o, ids, mode)
        return
    L, H = f._L, f._handle
    T = len(m._vertices_by_triangles)
    f._ensure_workspace(T)
    z, c, n = np.empty((h, w), F32), np.empty((h, w, 3), F32), np.empty((h, w, 3), F32)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    flags = _lib.CRB_CLEAR_FIRST | _lib.CRB_CLIP_NEAR | (_lib.CRB_NO_SYNC if mode == "no_sync" else 0)
    v_, c_, n_ = (np.ascontiguousarray(a) for a in _mv(m))
    _lib.check(L.crb_render_host(H, v_.ctypes.data, c_.ctypes.data, n_.ctypes.data, T, flags, _lib.CRB_BUF_ALL,
                                 z.ctypes.data, c.ctypes.data, n.ctypes.data, st))
    if mode == "no_sync":
        torch.cuda.current_stream().synchronize()
    assert_frame((z, c, n, f._tri_id.cpu().numpy()), o, ids, mode)


# ---------------------------------------------------------------------------------------------------------------- views
_VIEWS = {}


def trex_views(V, h=256, w=256, fov=45.0, zn=0.05, light=None):
    key = (V, h, w, fov, zn, light is not None)
    if key not in _VIEWS:
        m = load_indexed("trex")
        views = inside_views(V)
        frames = [CL().render(h, w, *_mv(m), fov=fov, z_near=zn, view=views[k]) for k in range(V)]
        _VIEWS[key] = (m, views, frames)
    return _VIEWS[key]


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [1, 3, 6, 16])
@pytest.mark.parametrize("pipeline", [0, 1])
def test_views_inside_the_model(chunk, pipeline):
    """render_views with cameras inside the T-Rex: every chunking (1, 3, V, > V), the launch pipeline on and off, and
    defer_join + join(); z, colour, normals, tri_id and the uint8 image per view"""
    V = 6
    m, views, frames = trex_views(V)
    f = _filler(256, 256, 45.0, 0.05, {"CHUNK_PIPELINE": pipeline}, near_clip=True)
    dv, dc, dn = _device(*_mv(m))
    for defer in (False, True):
        out = f.render_views(dv, dc, dn, views, want=("z", "color", "normals", "triangle_id"), color_u8_out=True,
                             chunk=chunk, check_status=not defer, defer_join=defer)
        if defer:
            f.join()
        for k, (o, ids) in enumerate(frames):
            what = f"chunk={chunk} pipeline={pipeline} defer={defer} view {k}"
            assert_frame((out["z"][k], out["color"][k], out["normals"][k], out["triangle_id"][k]), o, ids, what)
            _words(out["color_u8"][k], u8(o.color_buffer), what + ": color_u8")
        assert sum(int((o.z_buffer < 1e6).sum()) for o, _ in frames) > 10000


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [1, 2, 3])
def test_views_fused_guro(shape):
    V = 4
    m, views, frames = trex_views(V)
    f = _filler(256, 256, 45.0, 0.05, {"RASTER_SHAPE": shape}, near_clip=True)
    out = f.render_views(*_device(*_mv(m)), views, want=("color",), color_u8_out=True, guro_light=LIGHT, chunk=2)
    for k, (o, _) in enumerate(frames):
        _words(out["color"][k], lit(o), f"shape {shape} view {k}: lit colour")
        _words(out["color_u8"][k], u8(lit(o)), f"shape {shape} view {k}: lit uint8")


@pytest.mark.gpu
@pytest.mark.parametrize("s", [2, 4])
def test_views_supersampled(s):
    from oracle import ssaa_oracle as SS
    V = 3
    m, views, frames = trex_views(V, h=128 * s, w=128 * s)
    f = _filler(128 * s, 128 * s, 45.0, 0.05, near_clip=True)
    for light in (None, LIGHT):
        out = f.render_views(*_device(*_mv(m)), views, color_u8_out=True, supersample=s, guro_light=light, chunk=2)
        for k, (o, _) in enumerate(frames):
            want = SS.resolve(o.color_buffer if light is None else lit(o), s)
            _words(out["color_u8"][k], want, f"SS{s} light={light} view {k}")


@pytest.mark.gpu
def test_views_row_exchange_into_two_buffers():
    import torch
    V, h, w = 4, 256, 256
    m, views, frames = trex_views(V)
    f = _filler(h, w, 45.0, 0.05, near_clip=True)
    bufs = [torch.zeros((V, h // 2, w, 3), dtype=torch.uint8, device="cuda") for _ in range(2)]
    f.render_views(*_device(*_mv(m)), views, want=(), chunk=3, u8_exchange=(h // 2, [b.data_ptr() for b in bufs]))
    torch.cuda.synchronize()
    img = torch.cat(bufs, dim=1)
    for k, (o, _) in enumerate(frames):
        _words(img[k], u8(o.color_buffer), f"row exchange view {k}")


@pytest.mark.gpu
@pytest.mark.parametrize("bands", [((0, 128), (128, 256)), ((0, 77), (77, 150), (150, 256))])
def test_band_fillers(bands):
    """Band fillers (tile-aligned and not) concatenate to the full clipped frame, single view and batched views"""
    m, fov, zn, h, w, o, ids = scene("straddle5_zn0.5")
    got = [[], [], [], []]
    for r0, r1 in bands:
        f = _filler(h, w, fov, zn, band=(r0, r1), near_clip=True, triangle_ids=True)
        f.render_arrays(*_device(*_mv(m)))
        for g, a in zip(got, (f.get_z_buffer(), f.get_color_buffer(), f.get_normals_buffer(), f.get_triangle_id_buffer())):
            g.append(a.copy())
    assert_frame([np.concatenate(g) for g in got], o, ids, f"bands {bands}")
    V = 3
    tm, views, frames = trex_views(V)
    parts = []
    for r0, r1 in bands:
        f = _filler(256, 256, 45.0, 0.05, band=(r0, r1), near_clip=True)
        parts.append(f.render_views(*_device(*_mv(tm)), views, want=("z", "color", "normals", "triangle_id"), chunk=2))
    for k, (ok, ik) in enumerate(frames):
        got = [torch_cat([p[name][k] for p in parts]) for name in ("z", "color", "normals", "triangle_id")]
        assert_frame(got, ok, ik, f"band views {bands} view {k}")


def torch_cat(ts):
    import torch
    return torch.cat(ts, dim=0)


# ---------------------------------------------------------------------------------------------------------------- texturing
def _texture_case(seed=3, T=300):
    rng = np.random.default_rng(seed)
    m = straddling(seed, 0.2, T=T)
    uv = rng.uniform(-1.5, 2.5, (T, 3, 2)).astype(F32)
    tex = rng.integers(0, 256, (37, 53, 3), dtype=np.uint8)
    return m, uv, tex


@pytest.mark.gpu
@pytest.mark.parametrize("wrap", ["clamp", "repeat", "mirror"])
@pytest.mark.parametrize("perspective", [False, True])
@pytest.mark.parametrize("filt", ["nearest", "bilinear", "trilinear"])
def test_textured(filt, perspective, wrap):
    from oracle import texture_wrap_oracle as WR
    m, uv, tex = _texture_case()
    h, w, zn = 192, 224, 0.2
    uv3 = np.concatenate([uv, np.zeros(uv.shape[:2] + (1,), F32)], axis=2)
    ofill = WR.TexturedOracleFiller(h, w, fov=90.0, z_near=zn, wrap=wrap)
    o, ids = CL().render(h, w, m._vertices_by_triangles, uv3, m._normals_by_triangles, fov=90.0, z_near=zn, filler=ofill,
                         texture=tex, perspective=perspective, filter=filt)
    f = _filler(h, w, 90.0, zn, near_clip=True, triangle_ids=True, texture_filter=filt, perspective_correct=perspective,
                texture_wrap=wrap)
    f.render_arrays(m._vertices_by_triangles, uv, m._normals_by_triangles, texture=tex)
    what = f"{filt} perspective={perspective} {wrap}"
    _words(f.get_z_buffer(), o.z_buffer, what + ": z")
    _words(f.get_color_buffer(), o.color_buffer, what + ": colour")
    _words(f.get_normals_buffer(), o.normals_buffer, what + ": normals")
    _words(f.get_triangle_id_buffer(), ids.astype(np.int32), what + ": tri_id")
    # and through batched views (identity view: the arrays as passed are camera space)
    ident = np.array([[1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0, 0, 0, 0, 0]], F32)
    fv = _filler(h, w, 90.0, zn, near_clip=True, texture_filter=filt, perspective_correct=perspective, texture_wrap=wrap)
    out = fv.render_views(*_device(m._vertices_by_triangles, uv3, m._normals_by_triangles), ident, texture=tex,
                          want=("color",), color_u8_out=True)
    _words(out["color"][0], o.color_buffer, what + ": views colour")
    _words(out["color_u8"][0], u8(o.color_buffer), what + ": views uint8")


# ---------------------------------------------------------------------------------------------------------------- pipelines
@pytest.mark.gpu
def test_host_image_pipeline_with_overflow_redraw():
    import torch
    from cython3dmodelrenderer_b200.pipeline import HostImagePipeline
    m = straddling(5, 0.5)
    h = w = 256
    o, _ = CL().render(h, w, *_mv(m), fov=90.0, z_near=0.5)
    pipe = HostImagePipeline(h, w, fov=90.0, z_near=0.5, depth=2, light=LIGHT, near_clip=True)
    block = torch.from_numpy(np.stack(_mv(m))).pin_memory()
    T = block.shape[1]
    f0 = pipe.slots[0].filler
    f0._ensure_workspace(T, 1, 64)                   # slot 0's first frame overflows: it must come back drawn
    assert f0._ws_T == 2 * T
    for _ in range(3):
        i = pipe.submit(block)
        _words(pipe.result(i), u8(lit(o)), "HostImagePipeline")
    assert f0._pair_cap > 1000
    pipe.drain()


@pytest.mark.gpu
def test_host_frame_pipeline():
    from cython3dmodelrenderer_b200.pipeline import HostFramePipeline
    h = w = 256
    pipe = HostFramePipeline(h, w, fov=90.0, z_near=0.5, depth=2, near_clip=True)
    for seed in (5, 6, 7):
        m = straddling(seed, 0.5)
        o, _ = CL().render(h, w, *_mv(m), fov=90.0, z_near=0.5)
        r = pipe.result(pipe.submit(*_mv(m)))
        for name, want in (("z", o.z_buffer), ("color", o.color_buffer), ("normals", o.normals_buffer)):
            _words(r[name], want, f"HostFramePipeline seed {seed}: {name}")
    pipe.drain()


@pytest.mark.gpu
def test_drop_in_renderer_and_compositing_with_id_base():
    from cython3dmodelrenderer_b200 import GuroIllumination, Renderer
    m, fov, zn, h, w, o, ids = scene("straddle0_zn0.1")
    f = _filler(h, w, fov, zn, near_clip=True)
    got = Renderer(f, GuroIllumination(LIGHT), None, h, w).render(m)
    _words(got, lit(o), "Renderer + GuroIllumination")
    # two calls into one frame: the second call's tri_id = 5000 + parent wherever it wrote
    under = straddling(9, 0.1, T=250)
    fi = _filler(h, w, fov, zn, near_clip=True, triangle_ids=True)
    fi.render_model(under)
    fi.render_model(m, id_base=5000)
    ou, iu = CL().render(h, w, *_mv(under), fov=fov, z_near=zn)
    pv, pc, pn, parent = CL().clip(*_mv(m), zn)
    ou.render_arrays(pv, pc, pn)
    ids2 = np.where(CL().clipped_ids(ou, pv, pn, parent, base=5000) >= 0, CL().clipped_ids(ou, pv, pn, parent, base=5000), iu)
    assert_frame((fi.get_z_buffer(), fi.get_color_buffer(), fi.get_normals_buffer(), fi.get_triangle_id_buffer()), ou, ids2,
                 "composited")
    assert (ids2 >= 5000).any() and ((ids2 >= 0) & (ids2 < 5000)).any()


# ---------------------------------------------------------------------------------------------------------------- invariance
@pytest.mark.gpu
def test_invariance_trex_orbit_1024_128_views():
    """Nothing of the T-Rex orbit crosses z_near: with and without the bit every output is bit-identical"""
    import torch
    from cython3dmodelrenderer_b200 import views as VW
    m = load_indexed("trex")
    dv, dc, dn = _device(*_mv(m))
    views = VW.orbit_views(128)
    outs = []
    for clip in (False, True):
        f = _filler(1024, 1024, 45.0, near_clip=clip)
        outs.append(f.render_views(dv, dc, dn, views, want=("z", "color", "normals", "triangle_id"), color_u8_out=True,
                                   chunk=32))
        torch.cuda.synchronize()
    for name in outs[0]:
        a, b = outs[0][name], outs[1][name]
        if a.dtype == torch.float32:
            a, b = a.view(torch.int32), b.view(torch.int32)
        assert torch.equal(a, b), f"orbit: {name} differs with the bit"
    assert int((outs[0]["z"] < 1e5).sum()) > 1000000


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [1, 5, 14])
def test_invariance_scenes_lifted_past_the_plane(seed):
    m = random_scene(seed, T=400)
    v = m._vertices_by_triangles.copy()
    v[..., 2] = np.abs(v[..., 2]) + F32(0.5)
    lifted = TriModel(v, m._colors_by_triangles, m._normals_by_triangles)
    res = []
    for clip in (False, True):
        for path in ("tiled", "atomic"):
            f = _filler(256, 256, 90.0, 0.5, near_clip=clip, triangle_ids=True)
            f.render_arrays(*_device(*_mv(lifted)), path=path)
            res.append((f.get_z_buffer().copy(), f.get_color_buffer().copy(), f.get_normals_buffer().copy(),
                        f.get_triangle_id_buffer()))
    for r in res[1:]:
        for a, b in zip(res[0], r):
            assert bits_equal(a, b)


# ---------------------------------------------------------------------------------------------------------------- refusals
@pytest.mark.gpu
def test_refusals():
    import torch
    from cython3dmodelrenderer_b200 import _lib
    m = straddling(5, 0.5, T=64)
    T = 64
    dv, dc, dn = _device(*_mv(m))
    INV, STATE = _lib.CRB_ERR_INVALID, _lib.CRB_ERR_STATE
    CLIP = _lib.CRB_CLIP_NEAR | _lib.CRB_CLEAR_FIRST
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    # a bary output with the bit
    f = _filler(64, 64, 90.0, triangle_ids=True, barycentrics=True)
    f._ensure_workspace(2 * T)
    L, H = f._L, f._handle
    assert L.crb_render(H, dv.data_ptr(), dc.data_ptr(), dn.data_ptr(), T, CLIP, st) == INV
    bary = torch.zeros((1, 64, 64, 3), dtype=torch.float32, device="cuda")
    views = torch.from_numpy(np.array([[1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0, 0, 0, 0, 0]], F32)).cuda()
    assert L.crb_render_views_ids(H, dv.data_ptr(), dc.data_ptr(), dn.data_ptr(), T, views.data_ptr(), 1, None, None, None,
                                  None, None, bary.data_ptr(), CLIP, None, st) == INV
    # z_near of 0, negative or NaN
    for zn in (0.0, -0.1, float("nan"), float("inf")):
        fz = _filler(64, 64, 90.0, zn)
        fz._ensure_workspace(2 * T)
        assert fz._L.crb_render(fz._handle, dv.data_ptr(), dc.data_ptr(), dn.data_ptr(), T, CLIP, st) == INV
        with pytest.raises(ValueError):
            _filler(64, 64, 90.0, zn, near_clip=True)
    # a workspace bound for T but not 2T: refused on every entry point; 2T is enough
    fw = _filler(64, 64, 90.0)
    Lw, Hw = fw._L, fw._handle
    nbytes = Lw.crb_workspace_bytes(Hw, T, 1, 0)
    ws = torch.empty(nbytes + 256, dtype=torch.uint8, device="cuda")
    _lib.check(Lw.crb_bind_workspace(Hw, (ws.data_ptr() + 255) // 256 * 256, nbytes, T, 1, 0, st))
    assert Lw.crb_render(Hw, dv.data_ptr(), dc.data_ptr(), dn.data_ptr(), T, CLIP, st) == STATE
    assert Lw.crb_render_views(Hw, dv.data_ptr(), dc.data_ptr(), dn.data_ptr(), T, views.data_ptr(), 1, None, None, None,
                               None, CLIP, None, st) == STATE
    v_, c_, n_ = (np.ascontiguousarray(a) for a in _mv(m))
    assert Lw.crb_render_host(Hw, v_.ctypes.data, c_.ctypes.data, n_.ctypes.data, T, CLIP, 0, None, None, None, st) == STATE
    img_dev = torch.empty((64, 64, 3), dtype=torch.uint8, device="cuda")
    img_host = torch.empty((64, 64, 3), dtype=torch.uint8).pin_memory()
    assert Lw.crb_render_image_host(Hw, v_.ctypes.data, c_.ctypes.data, n_.ctypes.data, T, CLIP, None, img_dev.data_ptr(),
                                    img_host.data_ptr(), None, st) == STATE
    _lib.check(Lw.crb_render(Hw, dv.data_ptr(), dc.data_ptr(), dn.data_ptr(), T // 2, CLIP, st))
    torch.cuda.synchronize()
    # the Python surface, before anything is queued
    with pytest.raises(ValueError):
        _filler(64, 64, 90.0, near_clip=True, barycentrics=True)
    with pytest.raises(ValueError):
        _filler(64, 64, 90.0, near_clip="yes")
    fc = _filler(64, 64, 90.0, near_clip=True)
    launches = fc.launch_count
    with pytest.raises(ValueError):
        fc.render_views(dv, dc, dn, views, want=("z", "barycentrics"))
    with pytest.raises(ValueError):
        fc.render_views(dv, dc, dn, views, barycentrics_out=bary)
    assert fc.launch_count == launches
    from cython3dmodelrenderer_b200.pipeline import HostFramePipeline, HostImagePipeline
    with pytest.raises(ValueError):
        HostImagePipeline(64, 64, z_near=0.0, near_clip=True)
    with pytest.raises(ValueError):
        HostFramePipeline(64, 64, z_near=-1.0, near_clip=True)


@pytest.mark.gpu
def test_overflowing_frame_leaves_outputs_untouched_and_host_path_redraws():
    import torch
    from cython3dmodelrenderer_b200 import _lib
    m, fov, zn, h, w, o, ids = scene("straddle0_zn0.1")
    dv, dc, dn = _device(*_mv(m))
    T = dv.shape[0]
    f = _filler(h, w, fov, zn)
    L, H = f._L, f._handle
    nbytes = L.crb_workspace_bytes(H, 2 * T, 1, 64)
    ws = torch.empty(nbytes + 256, dtype=torch.uint8, device="cuda")
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(L.crb_bind_workspace(H, (ws.data_ptr() + 255) // 256 * 256, nbytes, 2 * T, 1, 64, st))
    z, c, n = f.device_buffers()
    z.fill_(7.0); c.fill_(7.0); n.fill_(7.0)
    tri = torch.full((h, w), SENTINEL, dtype=torch.int32, device="cuda")
    _lib.check(L.crb_bind_id_buffers(H, tri.data_ptr(), None, 0))
    _lib.check(L.crb_render(H, dv.data_ptr(), dc.data_ptr(), dn.data_ptr(), T, _lib.CRB_CLEAR_FIRST | _lib.CRB_CLIP_NEAR, st))
    need, cap = ctypes.c_int64(), ctypes.c_int64()
    assert L.crb_status(H, ctypes.byref(need), ctypes.byref(cap), st) == _lib.CRB_ERR_OVERFLOW
    assert (tri.cpu().numpy() == SENTINEL).all()
    assert (z.cpu().numpy() == 7.0).all() and (c.cpu().numpy() == 7.0).all() and (n.cpu().numpy() == 7.0).all()
    # the filler's host path with a pair list too small: the frame is drawn again with the room it asked for
    fh = _filler(h, w, fov, zn, near_clip=True, triangle_ids=True)
    fh._ensure_workspace(T, 1, 64)
    assert fh._pair_cap < 1000
    fh.render_arrays(*_mv(m))
    assert_frame((fh.get_z_buffer(), fh.get_color_buffer(), fh.get_normals_buffer(), fh.get_triangle_id_buffer()), o, ids,
                 "host path after overflow")
    assert fh._pair_cap > 1000
