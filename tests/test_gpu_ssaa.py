"""Supersampled images (CRB_SS2 / CRB_SS4, render_views(supersample=s), HostImagePipeline(supersample=s),
crb_color_u8_resolved; DESIGN 2) on the GPU, byte for byte against the oracle (oracle/ssaa_oracle.py): T-Rex orbit views,
quads and the edge families at sizes that are not tile or 16-pixel multiples, every rasterizer shape, the launch pipeline and
defer_join, lit and unlit, textured in every filter, interpolation and wrap mode; the fused resolve against the unfused one on a
large single-view frame (split heavy tiles); HostImagePipeline with a frame drawn again after an overflow; the refusals; and
an overflowing frame that leaves the image untouched.
"""
import ctypes

import numpy as np
import pytest

from conftest import load_indexed

F32 = np.float32
LIGHT = [0.3, -0.2, 1.0]
SS_BIT = {2: 65536, 4: 131072}
IDENTITY = np.array([[1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0, 0, 0, 0, 0]], F32)     # R = I, p = q = 0


def SS():
    from oracle import ssaa_oracle
    return ssaa_oracle


def _device(*arrays):
    import torch
    return tuple(torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays)


def _mv(m):
    return m._vertices_by_triangles, m._colors_by_triangles, m._normals_by_triangles


def _filler(h, w, fov, shape=0, **kw):
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller, _lib
    f = AdvancedPixelBufferFiller(h, w, fov=fov, **kw)
    if shape:
        f.set_option(_lib.CRB_OPT_RASTER_SHAPE, shape)
    return f


def _assert_bytes(got, want, what):
    got = got.cpu().numpy() if hasattr(got, "cpu") else np.asarray(got)
    assert got.shape == want.shape, f"{what}: shape {got.shape} != {want.shape}"
    if not np.array_equal(got, want):
        bad = np.argwhere(got != want)
        raise AssertionError(f"{what}: {len(bad)} bytes differ, first {bad[:5].tolist()}: got {got[tuple(bad[0])]} "
                             f"want {want[tuple(bad[0])]}")


def _orbit(V, stride=16):
    from cython3dmodelrenderer_b200 import views as VW
    return VW.orbit_views(128, first=0, count=V, stride=stride)


def _oracle_views(m, views, h, w, s, fov, light=None, uv=None, **tex):
    """Per view: the oracle's supersampled image of the camera-space arrays of views.transform_arrays_host"""
    from cython3dmodelrenderer_b200 import views as VW
    out = []
    for k in range(len(views)):
        vk, nk = VW.transform_arrays_host(views[k], m._vertices_by_triangles, m._normals_by_triangles)
        out.append(SS().render_resolved(h, w, s, vk, m._colors_by_triangles if uv is None else uv, nk, fov=fov, light=light, **tex))
    return out


def _edges(h, w):
    import test_gpu_edges as E
    return E.concat(*(E.family(k, h, w) for k in "ACDEFG")), E.FOV


def _quads():
    from test_gpu_ids import _quad_pair
    from conftest import TriModel
    a, b = _quad_pair(2.0, (10.0, 200.0)), _quad_pair(3.0, (90.0, 250.0))
    return TriModel(*(np.concatenate([x, y]) for x, y in zip(_mv(a), _mv(b)))), 90.0


@pytest.mark.gpu
@pytest.mark.parametrize("lit", [False, True])
@pytest.mark.parametrize("s", [2, 4])
def test_trex_orbit_views(s, lit):
    """256^2 images of 6 T-Rex orbit views from 512^2 (s = 2) or 1024^2 (s = 4) samples, in chunks of 4 (two launches)"""
    m = load_indexed("trex")
    views = _orbit(6)
    dv, dc, dn = _device(*_mv(m))
    f = _filler(256 * s, 256 * s, 45.0)
    out = f.render_views(dv, dc, dn, views, color_u8_out=True, supersample=s, chunk=4, guro_light=LIGHT if lit else None)
    assert set(out) == {"color_u8"}
    want = _oracle_views(m, views, 256, 256, s, 45.0, light=LIGHT if lit else None)
    for k in range(len(views)):
        _assert_bytes(out["color_u8"][k], want[k], f"s={s} lit={lit} view {k}")
        assert int((want[k] > 0).any(axis=2).sum()) > 3000


# (scene, s): output h x w from s*h x s*w samples.  200 x 344 samples are no tile multiples, and w/s = 172 or 86 no 16-multiple
SCENES = {("quads", 2): lambda: _quads() + (64, 96), ("quads", 4): lambda: _quads() + (64, 96),
          ("edges", 2): lambda: _edges(200, 344) + (100, 172), ("edges", 4): lambda: _edges(200, 344) + (50, 86),
          ("edges256", 4): lambda: _edges(256, 256) + (64, 64)}


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [0, 1, 2, 3])
@pytest.mark.parametrize("scene", sorted(SCENES))
def test_scenes_every_shape(scene, shape):
    """Quads and the edge families, one view each, in every rasterizer shape, unlit and lit"""
    name, s = scene
    m, fov, h, w = SCENES[scene]()
    dv, dc, dn = _device(*_mv(m))
    for light in (None, LIGHT):
        f = _filler(h * s, w * s, fov, shape)
        out = f.render_views(dv, dc, dn, IDENTITY, color_u8_out=True, supersample=s, guro_light=light)
        want = _oracle_views(m, IDENTITY, h, w, s, fov, light=light)[0]
        _assert_bytes(out["color_u8"][0], want, f"{name} shape {shape} s={s} light={light}")


@pytest.mark.gpu
@pytest.mark.parametrize("pipeline", [0, 1])
@pytest.mark.parametrize("chunk", [1, 3, 8])
def test_chunks_pipeline_and_defer_join(chunk, pipeline):
    """5 T-Rex views at 128^2 from 256^2 samples: chunk 1 / 3 / > V, the launch pipeline off and on, defer_join + join(), a
    caller tensor; equal to the oracle"""
    import torch
    from cython3dmodelrenderer_b200 import _lib
    m = load_indexed("trex")
    views = _orbit(5, stride=25)
    dv, dc, dn = _device(*_mv(m))
    want = _oracle_views(m, views, 128, 128, 2, 45.0, light=LIGHT)
    for defer in (False, True):
        f = _filler(256, 256, 45.0)
        f.set_option(_lib.CRB_OPT_CHUNK_PIPELINE, pipeline)
        img = torch.full((5, 128, 128, 3), 77, dtype=torch.uint8, device="cuda")
        kw = {"check_status": False, "defer_join": True} if defer else {}
        out = f.render_views(dv, dc, dn, views, color_u8_out=img, supersample=2, chunk=chunk, guro_light=LIGHT, **kw)
        assert out["color_u8"] is img
        if defer:
            f.join()
        for k in range(5):
            _assert_bytes(img[k], want[k], f"chunk {chunk} pipeline {pipeline} defer {defer} view {k}")


MODES = {"nearest": ("nearest", False), "nearest_persp": ("nearest", True), "bilinear": ("bilinear", False),
         "bilinear_persp": ("bilinear", True), "trilinear": ("trilinear", False), "trilinear_persp": ("trilinear", True)}


@pytest.mark.gpu
@pytest.mark.parametrize("wrap", ["clamp", "repeat", "mirror"])
@pytest.mark.parametrize("mode", sorted(MODES))
def test_textured(mode, wrap):
    """Two T-Rex views at 128^2, textured with spherical coordinates tiled 3 x 3 (wrap modes act), s = 2; trilinear also s = 4
    (its level of detail drops by log2 s: per-sample derivatives)"""
    from test_gpu_texture import _trex_uvs
    from test_texture_oracle import random_texture
    m = load_indexed("trex")
    uv = _trex_uvs(m) * F32(3) - F32(1)
    tex = random_texture(31, 97, 131)
    filt, persp = MODES[mode]
    views = _orbit(2, stride=40)
    dv, dn = _device(m._vertices_by_triangles, m._normals_by_triangles)
    for s in ((2, 4) if filt == "trilinear" else (2,)):
        f = _filler(128 * s, 128 * s, 45.0, texture_filter=filt, perspective_correct=persp, texture_wrap=wrap)
        out = f.render_views(dv, uv, dn, views, color_u8_out=True, supersample=s, texture=tex, guro_light=LIGHT)
        want = _oracle_views(m, views, 128, 128, s, 45.0, light=LIGHT, uv=uv, texture=tex, filter=filt, perspective=persp,
                             wrap=wrap)
        for k in range(len(views)):
            _assert_bytes(out["color_u8"][k], want[k], f"{mode} {wrap} s={s} view {k}")


@pytest.mark.gpu
@pytest.mark.parametrize("s", [2, 4])
def test_fused_equals_unfused_on_a_large_frame(s):
    """The bunny at 4096^2 samples with Guro, one view (split heavy tiles): the fused image of render_views equals
    crb_color_u8_resolved of the float32 render of the same frame; and crb_render_image_host's fused image equals the drop-in
    flow (render_model, the device lighting of illuminate_guro, color_u8_flipped(supersample=s))"""
    import torch
    from cython3dmodelrenderer_b200 import _lib
    m = load_indexed("bunny")
    dv, dc, dn = _device(*_mv(m))
    f = _filler(4096, 4096, 45.0)
    fused = f.render_views(dv, dc, dn, IDENTITY, color_u8_out=True, supersample=s, guro_light=LIGHT)["color_u8"][0]
    g = _filler(4096, 4096, 45.0)
    g.render_views(dv, dc, dn, IDENTITY, want=("color",), color_out=g._color[None], guro_light=LIGHT)
    unfused = torch.empty((4096 // s, 4096 // s, 3), dtype=torch.uint8, device="cuda")
    _lib.check(g._L.crb_color_u8_resolved(g._handle, s, unfused.data_ptr(), g._stream()))
    unfused = unfused.cpu().numpy()
    assert tuple(fused.shape) == (4096 // s, 4096 // s, 3)
    _assert_bytes(fused, unfused, f"bunny s={s}")
    assert int((unfused > 0).any(axis=2).sum()) > 100000 // (s * s)
    # untransformed: the drop-in flow against crb_render_image_host
    l = -np.asarray(LIGHT, dtype=F32)           # GuroIllumination's light_direction: negated, normalised
    l = l / np.linalg.norm(l)
    la = (ctypes.c_float * 3)(*[float(x) for x in l])
    d = _filler(4096, 4096, 45.0)
    d.render_model(m)
    d.illuminate_guro(l)
    dropin = d.color_u8_flipped(supersample=s)
    T = len(m._vertices_by_triangles)
    f._ensure_workspace(T)
    v, c, n = (torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in _mv(m))
    host = torch.zeros((4096 // s, 4096 // s, 3), dtype=torch.uint8).pin_memory()
    dev = torch.empty((4096 // s, 4096 // s, 3), dtype=torch.uint8, device="cuda")
    _lib.check(f._L.crb_render_image_host(f._handle, v.data_ptr(), c.data_ptr(), n.data_ptr(), T, _lib.CRB_GURO | SS_BIT[s],
                                          la, dev.data_ptr(), host.data_ptr(), None, f._stream()))
    _assert_bytes(dropin, host.numpy(), f"bunny drop-in s={s}")


@pytest.mark.gpu
@pytest.mark.parametrize("s", [1, 2, 4])
def test_host_image_pipeline(s):
    """HostImagePipeline(256, 256, supersample=s): every frame equals the oracle; a first frame whose pair list is too small is
    skipped and drawn again"""
    import torch
    from cython3dmodelrenderer_b200.pipeline import HostImagePipeline
    from cython3dmodelrenderer_b200 import views as VW
    m = load_indexed("trex")
    views = _orbit(3, stride=33)
    pipe = HostImagePipeline(256, 256, fov=45.0, depth=2, light=LIGHT, supersample=s)
    assert pipe.slots[0].filler.get_size() == (256 * s, 256 * s)
    T = len(m._vertices_by_triangles)
    f0 = pipe.slots[0].filler
    f0._ensure_workspace(T, 1, 64)                     # slot 0's first frame overflows: it must come back drawn
    assert f0._pair_cap < 1000
    blocks = []
    for k in range(len(views)):
        vk, nk = VW.transform_arrays_host(views[k], m._vertices_by_triangles, m._normals_by_triangles)
        blocks.append(torch.from_numpy(np.stack([vk, m._colors_by_triangles, nk])).pin_memory())
    want = _oracle_views(m, views, 256, 256, s, 45.0, light=LIGHT)
    for k in range(len(views)):
        i = pipe.submit(blocks[k])
        _assert_bytes(pipe.result(i).copy(), want[k], f"pipeline s={s} frame {k}")
    assert f0._pair_cap > 1000


def _raw_args(f, m):
    dv, dc, dn = _device(*_mv(m))
    f._ensure_workspace(dv.shape[0])
    st = ctypes.c_void_p(__import__("torch").cuda.current_stream().cuda_stream)
    return dv, dc, dn, st


@pytest.mark.gpu
def test_refusals():
    import torch
    from cython3dmodelrenderer_b200 import _lib
    m = load_indexed("trex")
    T = len(m._vertices_by_triangles)
    SS2, SS4, INV = _lib.CRB_SS2, _lib.CRB_SS4, _lib.CRB_ERR_INVALID
    f = _filler(256, 256, 45.0)
    L, H = f._L, f._handle
    dv, dc, dn, st = _raw_args(f, m)
    img = torch.zeros((128, 128, 3), dtype=torch.uint8, device="cuda")
    flt = torch.zeros((256, 256, 3), dtype=torch.float32, device="cuda")
    ids = torch.zeros((256, 256), dtype=torch.int32, device="cuda")

    def views(z=None, c=None, n=None, u8=img, tri=None, bary=None, flags=SS2, handle=H):
        p = lambda t: None if t is None else t.data_ptr()
        return L.crb_render_views_ids(handle, dv.data_ptr(), dc.data_ptr(), dn.data_ptr(), T, None, 1, p(z), p(c), p(n),
                                      p(u8), p(tri), p(bary), flags, None, st)

    assert views() == _lib.CRB_OK
    assert views(flags=SS2 | SS4) == INV
    assert views(u8=None) == INV
    for kw in ({"z": flt[..., 0]}, {"c": flt}, {"n": flt}, {"tri": ids}, {"bary": flt}):
        assert views(**kw) == INV, kw
    assert L.crb_render_views(H, dv.data_ptr(), dc.data_ptr(), dn.data_ptr(), T, None, 1, None, flt.data_ptr(), None, None,
                              SS4, None, st) == INV
    for flags in (SS2, SS4, SS2 | SS4):
        assert L.crb_render(H, dv.data_ptr(), dc.data_ptr(), dn.data_ptr(), T, flags | _lib.CRB_CLEAR_FIRST, st) == INV
        v, c, n = (np.ascontiguousarray(a) for a in _mv(m))
        assert L.crb_render_host(H, v.ctypes.data, c.ctypes.data, n.ctypes.data, T, flags, 0, None, None, None, st) == INV
    odd = _filler(258, 256, 45.0)                      # rows % 4 != 0 (258 % 2 == 0: s = 2 is fine)
    odd._ensure_workspace(T)
    img_odd = torch.zeros((129, 128, 3), dtype=torch.uint8, device="cuda")
    assert views(u8=img_odd, handle=odd._handle) == _lib.CRB_OK
    assert views(u8=img_odd, handle=odd._handle, flags=SS4) == INV
    odd_w = _filler(256, 250, 45.0)                    # w % 4 != 0
    odd_w._ensure_workspace(T)
    assert views(handle=odd_w._handle, flags=SS4) == INV
    band = _filler(256, 256, 45.0, band=(0, 128))
    band._ensure_workspace(T)
    assert views(handle=band._handle) == INV
    recv = torch.zeros((256, 256, 3), dtype=torch.uint8, device="cuda")
    arr = (ctypes.c_void_p * 1)(recv.data_ptr())
    _lib.check(L.crb_set_u8_exchange(H, 1, 256, arr))
    assert views() == INV and views(u8=None) == INV
    _lib.check(L.crb_set_u8_exchange(H, 0, 0, None))
    assert views() == _lib.CRB_OK
    for s in (0, 3, 8, -2):
        assert L.crb_color_u8_resolved(H, s, img.data_ptr(), st) == INV
    assert L.crb_color_u8_resolved(odd._handle, 4, img.data_ptr(), st) == INV
    assert L.crb_color_u8_resolved(band._handle, 2, img.data_ptr(), st) == INV
    # crb_render_image_host: refused like crb_render_views, and (rows/s) * (w/s) * 3 bytes written
    v, c, n = (torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in _mv(m))
    host = torch.full((256, 256, 3), 9, dtype=torch.uint8).pin_memory()
    dev = torch.zeros((256, 256, 3), dtype=torch.uint8, device="cuda")
    assert L.crb_render_image_host(H, v.data_ptr(), c.data_ptr(), n.data_ptr(), T, SS2 | SS4, None, dev.data_ptr(),
                                   host.data_ptr(), None, st) == INV
    _lib.check(L.crb_render_image_host(H, v.data_ptr(), c.data_ptr(), n.data_ptr(), T, SS4, None, dev.data_ptr(),
                                       host.data_ptr(), None, st))
    flat = host.numpy().reshape(-1)
    assert (flat[64 * 64 * 3:] == 9).all()
    want = SS().render_resolved(64, 64, 4, *_mv(m), fov=45.0)
    assert np.array_equal(flat[:64 * 64 * 3].reshape(64, 64, 3), want)


@pytest.mark.gpu
def test_python_refusals():
    import torch
    m = load_indexed("trex")
    dv, dc, dn = _device(*_mv(m))
    f = _filler(256, 256, 45.0)
    bad = [{"supersample": 3}, {"supersample": True}, {"supersample": 2.0},
           {"supersample": 2, "want": ("z",)}, {"supersample": 2, "want": ("triangle_id",)},
           {"supersample": 2, "want": (), "color_u8_out": None},
           {"supersample": 2, "color_out": torch.zeros((1, 256, 256, 3), device="cuda")},
           {"supersample": 2, "color_u8_out": torch.zeros((1, 256, 256, 3), dtype=torch.uint8, device="cuda")},
           {"supersample": 4, "color_u8_out": torch.zeros((1, 64, 64, 3), dtype=torch.float32, device="cuda")},
           {"supersample": 2, "color_u8_out": True, "u8_exchange": (256, [0])}]
    for kw in bad:
        kw.setdefault("color_u8_out", True)
        with pytest.raises(ValueError):
            f.render_views(dv, dc, dn, IDENTITY, **kw)
    with pytest.raises(ValueError):
        _filler(256, 256, 45.0, band=(0, 128)).render_views(dv, dc, dn, IDENTITY, color_u8_out=True, supersample=2)
    with pytest.raises(ValueError):
        _filler(254, 256, 45.0).render_views(dv, dc, dn, IDENTITY, color_u8_out=True, supersample=4)
    for s in (3, 0, "2"):
        with pytest.raises(ValueError):
            f.color_u8_flipped(supersample=s)
    with pytest.raises(ValueError):
        _filler(254, 256, 45.0).color_u8_flipped(supersample=4)
    with pytest.raises(ValueError):
        _filler(256, 256, 45.0, band=(0, 128)).color_u8_flipped(supersample=2)
    from cython3dmodelrenderer_b200.pipeline import HostImagePipeline
    with pytest.raises(ValueError):
        HostImagePipeline(64, 64, supersample=8)
    # s = 1 is today's call: the default `want`, and the 1x image
    out = f.render_views(dv, dc, dn, IDENTITY, color_u8_out=True, supersample=1)
    assert set(out) == {"z", "color", "normals", "color_u8"} and tuple(out["color_u8"].shape) == (1, 256, 256, 3)


@pytest.mark.gpu
def test_overflowing_frame_leaves_the_image_untouched():
    import torch
    from cython3dmodelrenderer_b200 import _lib
    m = load_indexed("trex")
    f = _filler(512, 512, 45.0)
    L, H = f._L, f._handle
    dv, dc, dn = _device(*_mv(m))
    T = dv.shape[0]
    nbytes = L.crb_workspace_bytes(H, T, 1, 64)
    ws = torch.empty(nbytes + 256, dtype=torch.uint8, device="cuda")
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(L.crb_bind_workspace(H, (ws.data_ptr() + 255) // 256 * 256, nbytes, T, 1, 64, st))
    img = torch.full((256, 256, 3), 123, dtype=torch.uint8, device="cuda")
    _lib.check(L.crb_render_views(H, dv.data_ptr(), dc.data_ptr(), dn.data_ptr(), T, None, 1, None, None, None,
                                  img.data_ptr(), _lib.CRB_SS2, None, st))
    need, cap = ctypes.c_int64(), ctypes.c_int64()
    assert L.crb_status(H, ctypes.byref(need), ctypes.byref(cap), st) == _lib.CRB_ERR_OVERFLOW
    assert (img.cpu().numpy() == 123).all()
