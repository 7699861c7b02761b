"""Triangle-id and barycentric outputs (crb_bind_id_buffers, crb_render_views_ids; DESIGN 2) on the GPU, word for word.

tri_id is compared as int32 with the oracle's (oracle/ids_oracle.py), bary with bits_equal.  In every configuration the z,
colour, normals (and uint8) buffers of the same render with the id outputs off are compared too: turning them on must change
no bit of those.
"""
import ctypes

import numpy as np
import pytest

from conftest import TriModel, bits_equal, load_indexed, random_scene

F32 = np.float32
SENTINEL = 0x5EED1D5


def _ids():
    from oracle import ids_oracle
    return ids_oracle


def _edges(h, w):
    import test_gpu_edges as E
    return E.concat(*(E.family(k, h, w) for k in "ACDEFG")), E.FOV


def _mv(m):
    return m._vertices_by_triangles, m._colors_by_triangles, m._normals_by_triangles


def _device(m):
    import torch
    return tuple(torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in _mv(m))


def _quad_pair(z, colours):
    """Two copies of one triangle pair at depth z, a colour per copy: every covered pixel is an equal-depth tie."""
    v = np.array([[[-1, -1, z], [1, -1, z], [-1, 1, z]], [[1, -1, z], [1, 1, z], [-1, 1, z]]], F32)
    v = np.concatenate([v, v])
    n = np.zeros_like(v)
    n[..., 2] = -1
    return TriModel(v, np.concatenate([np.full((2, 3, 3), c, F32) for c in colours]), n)


SCENES = {"trex1024": lambda: (load_indexed("trex"), 45.0, 1024, 1024),
          "scene5": lambda: (random_scene(5, T=400), 90.0, 256, 256),
          "scene14": lambda: (random_scene(14, T=400), 90.0, 256, 256),
          "edges256": lambda: _edges(256, 256) + (256, 256),
          "edges200x333": lambda: _edges(200, 333) + (200, 333),
          "ties": lambda: (_quad_pair(2.0, (10.0, 20.0)), 90.0, 64, 96)}
_SCENE_CACHE, _ORACLE = {}, {}


def scene(name):
    if name not in _SCENE_CACHE:
        _SCENE_CACHE[name] = SCENES[name]()
    return _SCENE_CACHE[name]


def underlay(name):
    """The scene a composited frame was drawn onto first (base 0); the scene itself then gets base 5000."""
    return _quad_pair(2.5, (30.0, 40.0)) if name == "ties" else random_scene(17, T=300)


def oracle(name, composite):
    key = (name, composite)
    if key not in _ORACLE:
        m, fov, h, w = scene(name)
        o = _ids().IdsOracleFiller(h, w, fov=fov)
        if composite:
            o.render_model(underlay(name), base=0)
        o.render_model(m, base=5000 if composite else 0)
        _ORACLE[key] = o
    return _ORACLE[key]


def _assert_words(got, want, what):
    got, want = np.ascontiguousarray(got), np.ascontiguousarray(want)
    assert got.shape == want.shape, f"{what}: shape {got.shape} != {want.shape}"
    g, w = got.view(np.uint32), want.view(np.uint32)
    if not np.array_equal(g, w):
        bad = np.argwhere(g != w)
        raise AssertionError(f"{what}: {len(bad)} words differ, first {bad[:5].tolist()}: got {got[tuple(bad[0])]!r} "
                             f"want {want[tuple(bad[0])]!r}")


def assert_ids(tri_id, bary, o, what, rows=slice(None)):
    _assert_words(tri_id, o.tri_id[rows].astype(np.int32), f"{what}: tri_id")
    _assert_words(bary, o.bary[rows], f"{what}: bary")


def _buffers(f):
    return f.get_z_buffer().copy(), f.get_color_buffer().copy(), f.get_normals_buffer().copy()


def assert_same_buffers(got, want, what):
    for name, g, w in zip(("z", "color", "normals"), got, want):
        _assert_words(g, w, f"{what}: {name}")


CONFIGS = {"default": {}, "atomic": {}, "shape1": {"RASTER_SHAPE": 1}, "shape2": {"RASTER_SHAPE": 2},
           "shape3": {"RASTER_SHAPE": 3}, "tma0": {"TMA": 0}, "split_heavy0": {"SPLIT_HEAVY": 0}}


def _filler(h, w, fov, config=None, **kw):
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller, _lib
    f = AdvancedPixelBufferFiller(h, w, fov=fov, **kw)
    for opt, val in CONFIGS.get(config or "default", {}).items():
        f.set_option(getattr(_lib, "CRB_OPT_" + opt), val)
    return f


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(SCENES))
@pytest.mark.parametrize("config", sorted(CONFIGS))
def test_ids_on_every_path_and_switch(config, name):
    """Tiled and atomic paths, the three rasterizer shapes, TMA clear on / off, split heavy tiles on / off; fresh and
    composited (a second call with id_base 5000): ids equal the oracle, z / colour / normals equal the render without ids."""
    m, fov, h, w = scene(name)
    path = "atomic" if config == "atomic" else "tiled"
    for composite in (False, True):
        what = f"{name} {config} composite={composite}"
        fi = _filler(h, w, fov, config, triangle_ids=True, barycentrics=True)
        f0 = _filler(h, w, fov, config)
        for f, kw in ((fi, {"id_base": 5000 if composite else 0}), (f0, {})):
            if composite:
                f.render_arrays(*_mv(underlay(name)), path=path)
            f.render_arrays(*_mv(m), path=path, **kw)
        assert_ids(fi.get_triangle_id_buffer(), fi.get_barycentric_buffer(), oracle(name, composite), what)
        assert_same_buffers(_buffers(fi), _buffers(f0), what)
        assert_same_buffers(_buffers(fi), (oracle(name, composite).z_buffer, oracle(name, composite).color_buffer,
                                           oracle(name, composite).normals_buffer), what + " vs oracle")


@pytest.mark.gpu
def test_either_output_alone_and_ties():
    o = oracle("ties", True)
    assert set(np.unique(o.tri_id)) <= {-1, 5002, 5003}       # the later call and, within it, the highest index win
    m, fov, h, w = scene("ties")
    for kw in ({"triangle_ids": True}, {"barycentrics": True}):
        f = _filler(h, w, fov, **kw)
        f.render_model(underlay("ties"))
        f.render_model(m, id_base=5000)
        if "triangle_ids" in kw:
            _assert_words(f.get_triangle_id_buffer(), o.tri_id.astype(np.int32), "tri_id alone")
            assert f.device_id_buffers()[1] is None
            with pytest.raises(ValueError):
                f.get_barycentric_buffer()
        else:
            _assert_words(f.get_barycentric_buffer(), o.bary, "bary alone")
            assert f.device_id_buffers()[0] is None
            with pytest.raises(ValueError):
                f.get_triangle_id_buffer()


@pytest.mark.gpu
def test_drop_in_flow_of_two_models_and_clear():
    """render_model of two models with id_base, then clear() and a read with no render (crb_init_buffers resets the ids)."""
    trex, other = load_indexed("trex"), random_scene(9, T=300)
    T0 = len(trex._vertices_by_triangles)
    f = _filler(256, 256, 45.0, triangle_ids=True, barycentrics=True)
    o = _ids().IdsOracleFiller(256, 256, fov=45.0)
    for m, base in ((trex, 0), (other, T0)):
        f.render_model(m, id_base=base)
        o.render_model(m, base=base)
    ids = f.get_triangle_id_buffer()
    assert (ids >= T0).sum() > 100 and ((ids >= 0) & (ids < T0)).sum() > 100
    assert_ids(ids, f.get_barycentric_buffer(), o, "two models")
    assert_same_buffers(_buffers(f), (o.z_buffer, o.color_buffer, o.normals_buffer), "two models")
    f.clear()
    assert (f.get_triangle_id_buffer() == -1).all()
    assert bits_equal(f.get_barycentric_buffer(), np.zeros((256, 256, 3), F32))
    assert (f.get_z_buffer() == F32(1e6)).all()


def _orbit(V):
    from cython3dmodelrenderer_b200 import views as VW
    return VW.orbit_views(V, first=0, count=V, stride=7)


@pytest.mark.gpu
@pytest.mark.parametrize("pipeline", [0, 1])
@pytest.mark.parametrize("chunk", [1, 3, 5, 8])
def test_render_views_ids(chunk, pipeline):
    """Batched views, chunk 1 / 3 / V / > V, the launch pipeline off and on, defer_join + join() and the uint8 image: each
    view's ids equal the oracle on crb_transform_view's arrays; every other output equals the batch without ids."""
    from cython3dmodelrenderer_b200 import _lib
    m = load_indexed("trex")
    h, w, fov, V = 256, 256, 45.0, 5
    views = _orbit(V)
    dv, dc, dn = _device(m)
    want = ("z", "color", "normals", "triangle_id", "barycentrics")
    for defer in (False, True):
        fi, f0 = _filler(h, w, fov), _filler(h, w, fov)
        for f in (fi, f0):
            f.set_option(_lib.CRB_OPT_CHUNK_PIPELINE, pipeline)
        kw = {"check_status": False, "defer_join": True} if defer else {}
        out = fi.render_views(dv, dc, dn, views, want=want, chunk=chunk, color_u8_out=True, **kw)
        ref = f0.render_views(dv, dc, dn, views, chunk=chunk, color_u8_out=True, **kw)
        if defer:
            fi.join()
            f0.join()
        assert set(out) == {"z", "color", "normals", "triangle_id", "barycentrics", "color_u8"} and "triangle_id" not in ref
        for name in ("z", "color", "normals", "color_u8"):
            assert np.array_equal(out[name].cpu().numpy().view(np.uint8), ref[name].cpu().numpy().view(np.uint8)), name
        for k in range(V):
            gv, gn = (a.cpu().numpy() for a in fi.transform_view(dv, dn, views[k]))
            o = _ids().IdsOracleFiller(h, w, fov=fov)
            o.render_arrays(gv, m._colors_by_triangles, gn)
            assert_ids(out["triangle_id"][k].cpu().numpy(), out["barycentrics"][k].cpu().numpy(), o,
                       f"view {k} chunk={chunk} pipeline={pipeline} defer={defer}")


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [0, 1, 2, 3])
def test_render_views_ids_with_fused_guro(shape):
    """CRB_GURO fused into the shading pass (render_views' guro_light), every rasterizer shape: the ids equal the oracle's,
    the lit colour equals the oracle's lit colour, and every output equals the same lit batch without ids."""
    from cython3dmodelrenderer_b200 import _lib
    from oracle import oracle as O
    m = load_indexed("trex")
    h, w, fov, V, light = 256, 256, 45.0, 4, [0.3, -0.2, 1.0]
    views = _orbit(V)
    dv, dc, dn = _device(m)
    fi, f0 = _filler(h, w, fov), _filler(h, w, fov)
    for f in (fi, f0):
        f.set_option(_lib.CRB_OPT_RASTER_SHAPE, shape)
    out = fi.render_views(dv, dc, dn, views, want=("z", "color", "normals", "triangle_id", "barycentrics"), chunk=3,
                          color_u8_out=True, guro_light=light)
    ref = f0.render_views(dv, dc, dn, views, chunk=3, color_u8_out=True, guro_light=light)
    for name in ("z", "color", "normals", "color_u8"):
        assert np.array_equal(out[name].cpu().numpy().view(np.uint8), ref[name].cpu().numpy().view(np.uint8)), name
    for k in range(V):
        gv, gn = (a.cpu().numpy() for a in fi.transform_view(dv, dn, views[k]))
        o = _ids().IdsOracleFiller(h, w, fov=fov)
        o.render_arrays(gv, m._colors_by_triangles, gn)
        assert_ids(out["triangle_id"][k].cpu().numpy(), out["barycentrics"][k].cpu().numpy(), o, f"guro view {k} shape {shape}")
        lit = O.guro(o.color_buffer.copy(), o.normals_buffer, light)
        _assert_words(out["color"][k].cpu().numpy(), lit, f"guro view {k} shape {shape}: lit colour")


@pytest.mark.gpu
def test_render_views_caller_slabs_and_edges():
    """Caller-owned id slabs, one output alone, the plain-store clear size (200 x 333) and the edge families."""
    import torch
    from cython3dmodelrenderer_b200 import views as VW
    for h, w in ((256, 256), (200, 333)):
        m, fov = _edges(h, w)
        views = np.stack([VW.view_matrix(), VW.view_matrix(VW.rot_y(-3e-4), p=(0.0, 0.0, 2.0)), VW.view_matrix(q=(1e-4, -2e-4, 0.0))])
        dv, dc, dn = _device(m)
        tri = torch.full((3, h, w), SENTINEL, dtype=torch.int32, device="cuda")
        f = _filler(h, w, fov)
        out = f.render_views(dv, dc, dn, views, want=("z",), triangle_id_out=tri, chunk=2)
        assert out["triangle_id"] is tri and "barycentrics" not in out
        for k in range(3):
            gv, gn = (a.cpu().numpy() for a in f.transform_view(dv, dn, views[k]))
            o = _ids().IdsOracleFiller(h, w, fov=fov)
            o.render_arrays(gv, m._colors_by_triangles, gn)
            _assert_words(tri[k].cpu().numpy(), o.tri_id.astype(np.int32), f"view {k} {h}x{w}")
            _assert_words(out["z"][k].cpu().numpy(), o.z_buffer, f"view {k} {h}x{w} z")


@pytest.mark.gpu
@pytest.mark.parametrize("size", [(256, 256), (200, 333)], ids=lambda s: f"{s[0]}x{s[1]}")
def test_band_fillers(size):
    """Row bands, tile-aligned and not, one-row bands: each band equals the oracle's rows, so their concatenation is the frame."""
    h, w = size
    m, fov = _edges(h, w)
    o = _ids().IdsOracleFiller(h, w, fov=fov)
    o.render_model(m)
    dv, dc, dn = _device(m)
    cuts = sorted({0, 1, 31, 32, 33, 100, h // 2 + 3, h - 1, h})
    got_t, got_b = [], []
    for r0, r1 in zip(cuts[:-1], cuts[1:]):
        f = _filler(h, w, fov, band=(r0, r1), triangle_ids=True, barycentrics=True)
        f0 = _filler(h, w, fov, band=(r0, r1))
        f.render_arrays(dv, dc, dn)
        f0.render_arrays(dv, dc, dn)
        assert_ids(f.get_triangle_id_buffer(), f.get_barycentric_buffer(), o, f"band {r0}:{r1}", rows=slice(r0, r1))
        assert_same_buffers(_buffers(f), _buffers(f0), f"band {r0}:{r1}")
        got_t.append(f.get_triangle_id_buffer())
        got_b.append(f.get_barycentric_buffer())
    assert_ids(np.concatenate(got_t), np.concatenate(got_b), o, "concatenated bands")


@pytest.mark.gpu
def test_out_ptrs_filler_keeps_local_id_buffers():
    import torch
    m, fov, h, w = scene("scene5")
    r0, r1 = 40, 170
    z = torch.full((h, w), 1e6, dtype=torch.float32, device="cuda")
    c = torch.zeros((h, w, 3), dtype=torch.float32, device="cuda")
    n = torch.zeros((h, w, 3), dtype=torch.float32, device="cuda")
    ptrs = (z[r0:].data_ptr(), c[r0:].data_ptr(), n[r0:].data_ptr())
    f = _filler(h, w, fov, band=(r0, r1), out_ptrs=ptrs, triangle_ids=True, barycentrics=True)
    assert (f.get_triangle_id_buffer() == -1).all()
    f.render_model(m)
    assert_ids(f.get_triangle_id_buffer(), f.get_barycentric_buffer(), oracle("scene5", False), "out_ptrs", rows=slice(r0, r1))


TEX_MODES = [(flt, persp, wrap) for flt in ("nearest", "bilinear", "trilinear") for persp in (False, True)
             for wrap in ("clamp", "repeat", "mirror")]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", TEX_MODES, ids=lambda m: f"{m[0]}-{'persp' if m[1] else 'affine'}-{m[2]}")
def test_texture_modes_leave_ids_as_per_vertex(mode):
    """Per-pixel texturing: ids and bary equal those of the per-vertex render of the same v, n (screen-space barycentrics,
    also with perspective-correct coordinates), and the textured buffers equal the textured render without ids."""
    flt, persp, wrap = mode
    m = load_indexed("trex")
    h, w, fov = 256, 256, 45.0
    rng = np.random.default_rng(7)
    uv = rng.uniform(-1.5, 2.5, (len(m._vertices_by_triangles), 3, 2)).astype(F32)
    tex = rng.integers(0, 256, (64, 48, 3), dtype=np.uint8)
    v, c, n = _mv(m)
    for path in ("tiled", "atomic"):
        kw = dict(texturing="vertex", texture_filter=flt, perspective_correct=persp, texture_wrap=wrap)
        ft = _filler(h, w, fov, triangle_ids=True, barycentrics=True, **kw)
        f0 = _filler(h, w, fov, **kw)
        fv = _filler(h, w, fov, triangle_ids=True, barycentrics=True)
        ft.render_arrays(v, uv, n, texture=tex, path=path)
        f0.render_arrays(v, uv, n, texture=tex, path=path)
        fv.render_arrays(v, c, n, path=path)
        what = f"{mode} {path}"
        _assert_words(ft.get_triangle_id_buffer(), fv.get_triangle_id_buffer(), what + ": tri_id")
        _assert_words(ft.get_barycentric_buffer(), fv.get_barycentric_buffer(), what + ": bary")
        assert_same_buffers(_buffers(ft), _buffers(f0), what)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["trex1024", "scene14", "edges256"])
def test_attributes_restated_on_the_device(name):
    """The use the outputs are for: z, normals and colour interpolated in torch from (ids, bary) and the per-corner arrays --
    one operation per kernel, (a0*b1 + a1*b2) + a2*b3 -- reproduce the buffers (per-vertex colours, no Guro)."""
    import torch
    from oracle import oracle as O
    m, fov, h, w = scene(name)
    f = _filler(h, w, fov, triangle_ids=True, barycentrics=True)
    f.render_model(m)
    tri, bary = f.device_id_buffers()
    z, col, nrm = (t.cpu().numpy() for t in f.device_buffers())
    v, c, n = _mv(m)
    sz = O.project(h, w, O.projection_matrix(h, w, fov), v)[..., 2:3]
    drawn = tri >= 0
    t = tri[drawn].long()
    b = bary[drawn]
    assert int(drawn.sum()) > 100
    for attr, buf, name_ in ((sz, z[..., None], "z"), (n, nrm, "normals"), (c, col, "colour")):
        a = torch.from_numpy(np.ascontiguousarray(attr)).cuda()[t]
        s = torch.mul(a[:, 0], b[:, 0:1])
        s = torch.add(s, torch.mul(a[:, 1], b[:, 1:2]))
        s = torch.add(s, torch.mul(a[:, 2], b[:, 2:3]))
        _assert_words(s.cpu().numpy(), buf[drawn.cpu().numpy()], f"{name}: {name_} restated")


def _raw(f):
    from cython3dmodelrenderer_b200 import _lib
    return f._L, f._handle, _lib


@pytest.mark.gpu
def test_overflowing_frame_leaves_ids_untouched():
    """A caller-owned workspace whose pair list is too small: CRB_ERR_OVERFLOW, and the id buffers keep a sentinel."""
    import torch
    m = load_indexed("trex")
    h = w = 256
    f = _filler(h, w, 45.0)
    L, H, lib = _raw(f)
    dv, dc, dn = _device(m)
    T = dv.shape[0]
    nbytes = L.crb_workspace_bytes(H, T, 1, 64)
    ws = torch.empty(nbytes + 256, dtype=torch.uint8, device="cuda")
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    lib.check(L.crb_bind_workspace(H, (ws.data_ptr() + 255) // 256 * 256, nbytes, T, 1, 64, st))
    tri = torch.full((h, w), SENTINEL, dtype=torch.int32, device="cuda")
    bary = torch.full((h, w, 3), 7.0, dtype=torch.float32, device="cuda")
    lib.check(L.crb_bind_id_buffers(H, tri.data_ptr(), bary.data_ptr(), 0))
    lib.check(L.crb_render(H, dv.data_ptr(), dc.data_ptr(), dn.data_ptr(), T, lib.CRB_CLEAR_FIRST, st))
    need, cap = ctypes.c_int64(), ctypes.c_int64()
    assert L.crb_status(H, ctypes.byref(need), ctypes.byref(cap), st) == lib.CRB_ERR_OVERFLOW
    assert (tri.cpu().numpy() == SENTINEL).all() and (bary.cpu().numpy() == 7.0).all()


@pytest.mark.gpu
def test_render_image_host_leaves_bound_ids_untouched():
    import torch
    m = load_indexed("trex")
    h = w = 256
    f = _filler(h, w, 45.0, triangle_ids=True, barycentrics=True)
    L, H, lib = _raw(f)
    T = len(m._vertices_by_triangles)
    f._ensure_workspace(T)
    tri, bary = f._tri_id, f._bary
    tri.fill_(SENTINEL)
    bary.fill_(7.0)
    v, c, n = (torch.from_numpy(a).pin_memory() for a in _mv(m))
    img_dev = torch.empty((h, w, 3), dtype=torch.uint8, device="cuda")
    img_host = torch.empty((h, w, 3), dtype=torch.uint8).pin_memory()
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    lib.check(L.crb_render_image_host(H, v.data_ptr(), c.data_ptr(), n.data_ptr(), T, 0, None, img_dev.data_ptr(),
                                      img_host.data_ptr(), None, st))
    assert img_host.numpy().any()
    assert (tri.cpu().numpy() == SENTINEL).all() and (bary.cpu().numpy() == 7.0).all()


@pytest.mark.gpu
def test_refusals():
    import torch
    m = _quad_pair(2.0, (10.0, 20.0))
    f = _filler(32, 32, 90.0)
    L, H, lib = _raw(f)
    tri = torch.zeros((32, 32), dtype=torch.int32, device="cuda")
    assert L.crb_bind_id_buffers(H, tri.data_ptr(), None, -1) == lib.CRB_ERR_INVALID
    assert L.crb_bind_id_buffers(H, tri.data_ptr() + 4, None, 0) == lib.CRB_ERR_INVALID
    dv, dc, dn = _device(m)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    f._ensure_workspace(4)
    lib.check(L.crb_bind_id_buffers(H, tri.data_ptr(), None, 2 ** 31 - 4))     # base + T - 1 = 2^31 - 1: the last valid id
    lib.check(L.crb_render(H, dv.data_ptr(), dc.data_ptr(), dn.data_ptr(), 4, lib.CRB_CLEAR_FIRST, st))
    assert set(np.unique(tri.cpu().numpy())) == {-1, 2 ** 31 - 2, 2 ** 31 - 1}
    lib.check(L.crb_bind_id_buffers(H, tri.data_ptr(), None, 2 ** 31 - 3))     # one more: refused, nothing drawn
    before = tri.cpu().numpy().copy()
    assert L.crb_render(H, dv.data_ptr(), dc.data_ptr(), dn.data_ptr(), 4, lib.CRB_CLEAR_FIRST, st) == lib.CRB_ERR_INVALID
    assert np.array_equal(tri.cpu().numpy(), before)
    lib.check(L.crb_bind_id_buffers(H, None, None, 0))                          # unbound: renders as before
    lib.check(L.crb_render(H, dv.data_ptr(), dc.data_ptr(), dn.data_ptr(), 4, lib.CRB_CLEAR_FIRST, st))
    # the Python surface
    fi = _filler(32, 32, 90.0, triangle_ids=True)
    for bad in (-1, 2 ** 31 - 3, 1.5, True):
        with pytest.raises(ValueError):
            fi.render_model(m, id_base=bad)
    with pytest.raises(ValueError):
        f.get_triangle_id_buffer()
    with pytest.raises(ValueError):
        f.device_id_buffers()
    with pytest.raises(ValueError):
        _filler(32, 32, 90.0, triangle_ids="yes")
