"""The texturing modes CRB_TEX_PERSPECTIVE and CRB_TEX_BILINEAR on the GPU, word for word against their oracle
(oracle/texture_modes_oracle.py; DESIGN 2), in the three combinations that are new: nearest + perspective, bilinear + affine
and bilinear + perspective.  (Nearest + affine is tests/test_gpu_texture.py.)

The same ground as test_gpu_texture: tiled and atomic paths, each rasterizer shape, fresh and composited, host and device
inputs, the edge-case scene families (the near-camera-plane one gives w = inf and W = 0), batched views with the fused Guro
pass and uint8 output, crb_render_image_host, row bands, the drop-in Model / Renderer flow, and the refusals.
"""
import ctypes
import os

import numpy as np
import pytest

from conftest import GOLDEN, load_indexed
from test_gpu_texture import CONFIGS, SEEDS, SIZES, TEXTURES, _arrays, _assert_same, _base, _buffers, _scene, _trex_uvs
from test_texture_oracle import random_texture, random_uvs

F32 = np.float32
MODES = {"nearest_persp": ("nearest", True), "bilinear": ("bilinear", False), "bilinear_persp": ("bilinear", True)}


def O():
    from oracle import oracle
    return oracle


def TM():
    from oracle import texture_modes_oracle
    return texture_modes_oracle


def _filler(h, w, mode, **kw):
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller
    filt, persp = MODES[mode]
    return AdvancedPixelBufferFiller(h, w, texture_filter=filt, perspective_correct=persp, **kw)


def _oracle(h, w, mode, v, uv, n, tex, fov=90.0, base=None):
    filt, persp = MODES[mode]
    o = TM().TexturedOracleFiller(h, w, fov=fov)
    if base is not None:
        o.render_arrays(*base)
    o.render_arrays(v, uv, n, texture=tex, perspective=persp, filter=filt)
    return o


@pytest.fixture(scope="module")
def oracle_frames():
    cache = {}

    def get(mode, seed, size, tshape, composite):
        key = (mode, seed, size, tshape, composite)
        if key not in cache:
            m, uv = _scene(seed)
            o = _oracle(*size, mode, m._vertices_by_triangles, uv, m._normals_by_triangles, random_texture(seed, *tshape),
                        base=_base() if composite else None)
            cache[key] = _buffers(o)
        return cache[key]
    return get


@pytest.mark.gpu
@pytest.mark.parametrize("mode", sorted(MODES))
@pytest.mark.parametrize("size", SIZES, ids=lambda s: f"{s[0]}x{s[1]}")
@pytest.mark.parametrize("tshape", TEXTURES, ids=lambda s: f"tex{s[0]}x{s[1]}")
@pytest.mark.parametrize("config", sorted(CONFIGS))
def test_texture_modes_scenes_bit_exact(config, tshape, size, mode, oracle_frames):
    """Seeded scenes with in-range and out-of-range coordinates; fresh, and composited onto a per-vertex frame drawn by the
    same filler; host and device inputs, [T,3,3] and [T,3,2] coordinates."""
    import torch
    from cython3dmodelrenderer_b200 import _lib
    h, w = size
    path = "atomic" if config == "atomic" else "tiled"
    for seed in SEEDS:
        m, uv = _scene(seed)
        tex = random_texture(seed, *tshape)
        for composite in (False, True):
            f = _filler(h, w, mode)
            for opt, val in CONFIGS[config].items():
                f.set_option(getattr(_lib, "CRB_OPT_" + opt), val)
            if composite:
                f.render_arrays(*_base(), path=path)
            if seed == SEEDS[1]:     # device-resident inputs, texture as a CUDA tensor, (u, v) pairs
                v, n = (torch.from_numpy(a).cuda() for a in (m._vertices_by_triangles, m._normals_by_triangles))
                f.render_arrays(v, torch.from_numpy(np.ascontiguousarray(uv[..., :2])).cuda(), n, path=path,
                                texture=torch.from_numpy(tex).cuda())
            else:
                f.render_arrays(m._vertices_by_triangles, uv, m._normals_by_triangles, path=path, texture=tex)
            _assert_same(_buffers(f), oracle_frames(mode, seed, size, tshape, composite),
                         f"{mode} seed {seed} {config} tex {tshape} {h}x{w} composite={composite}")


@pytest.mark.gpu
@pytest.mark.parametrize("mode", sorted(MODES))
@pytest.mark.parametrize("size", SIZES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_edge_families_texture_modes(size, mode):
    import test_gpu_edges as E
    h, w = size
    for i, name in enumerate(sorted(E.FAMILIES)):
        m = E.family(name, h, w)
        v, _, n = _arrays(m)
        uv = random_uvs(50 + i, v.shape[0])
        tex = random_texture(i, 61, 83)
        want = _buffers(_oracle(h, w, mode, v, uv, n, tex, fov=E.FOV))
        for path in ("tiled", "atomic"):
            f = _filler(h, w, mode, fov=E.FOV)
            f.render_arrays(v, uv, n, path=path, texture=tex)
            _assert_same(_buffers(f), want, f"{mode} family {name} {path} {h}x{w}")


@pytest.mark.gpu
@pytest.mark.parametrize("mode", sorted(MODES))
@pytest.mark.parametrize("lit", [False, True])
def test_render_views_texture_modes_trex_orbit(lit, mode):
    """8 T-Rex orbit views at 1024^2: float32 slabs and the fused uint8 image, against the oracle on the camera-space arrays
    of views.transform_arrays_host (perspective divides by the transformed z), then oracle.guro, the row flip and
    astype('uint8'); lit, also crb_render_image_host with the mode's bits."""
    import torch
    from cython3dmodelrenderer_b200 import _lib, views as VW
    m = load_indexed("trex")
    uv = _trex_uvs(m)
    tex = random_texture(709, 709, 709)
    h = w = 1024
    light = [0.3, -0.2, 1.0] if lit else None
    views = VW.orbit_views(128, first=0, count=8, stride=16)
    dv, dn = (torch.from_numpy(a).cuda() for a in (m._vertices_by_triangles, m._normals_by_triangles))
    f = _filler(h, w, mode, fov=45.0)
    out = f.render_views(dv, uv, dn, views, chunk=3, color_u8_out=True, guro_light=light, texture=tex)
    for k in range(len(views)):
        vk, nk = VW.transform_arrays_host(views[k], m._vertices_by_triangles, m._normals_by_triangles)
        want = _buffers(_oracle(h, w, mode, vk, uv, nk, tex, fov=45.0))
        if lit:
            O().guro(want[1], want[2], light)
        got = tuple(out[name][k].cpu().numpy() for name in ("z", "color", "normals"))
        _assert_same(got, want, f"{mode} view {k} lit={lit}")
        with np.errstate(invalid="ignore"):
            want_u8 = want[1][::-1].astype("uint8")
        assert np.array_equal(out["color_u8"][k].cpu().numpy(), want_u8), f"{mode} uint8 view {k} lit={lit}"
        assert int((want[0] < F32(1e6)).sum()) > 100000
    if lit:
        filt, persp = MODES[mode]
        bits = _lib.CRB_TEXTURE | (_lib.CRB_TEX_BILINEAR if filt == "bilinear" else 0) | (_lib.CRB_TEX_PERSPECTIVE if persp else 0)
        vk, nk = VW.transform_arrays_host(views[3], m._vertices_by_triangles, m._normals_by_triangles)
        uv3 = np.concatenate([uv, np.zeros(uv.shape[:2] + (1,), F32)], axis=2)
        T = vk.shape[0]
        f._ensure_workspace(T)
        image_dev = torch.empty((h, w, 3), dtype=torch.uint8, device="cuda")
        image_host = np.zeros((h, w, 3), np.uint8)
        l = -np.asarray(light, dtype=F32)
        l = l / np.linalg.norm(l)
        la = (ctypes.c_float * 3)(*[float(x) for x in l])
        _lib.check(f._L.crb_render_image_host(f._handle, vk.ctypes.data, uv3.ctypes.data, nk.ctypes.data, T,
                                              _lib.CRB_GURO | bits, la, image_dev.data_ptr(), image_host.ctypes.data, None,
                                              f._stream()))
        o = _oracle(h, w, mode, vk, uv3, nk, tex, fov=45.0)
        c = o.get_color_buffer().copy()
        O().guro(c, o.get_normals_buffer(), light)
        with np.errstate(invalid="ignore"):
            assert np.array_equal(image_host, c[::-1].astype("uint8"))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", sorted(MODES))
@pytest.mark.parametrize("prepass", [1, 0])
def test_texture_modes_bands_concatenate_to_full_frame(prepass, mode):
    import torch
    from cython3dmodelrenderer_b200 import _lib
    m = load_indexed("trex")
    uv = _trex_uvs(m)
    tex = random_texture(3, 333, 4097)
    h = w = 256
    want = _buffers(_oracle(h, w, mode, m._vertices_by_triangles, uv, m._normals_by_triangles, tex, fov=45.0))
    dv, dn = (torch.from_numpy(a).cuda() for a in (m._vertices_by_triangles, m._normals_by_triangles))
    duv = torch.from_numpy(uv).cuda()
    parts = []
    for r0, r1 in ((0, 90), (90, 171), (171, 256)):
        f = _filler(h, w, mode, fov=45.0, band=(r0, r1))
        f.set_option(_lib.CRB_OPT_BAND_PREPASS, prepass)
        f.render_arrays(dv, duv, dn, texture=tex)
        parts.append(_buffers(f))
    got = tuple(np.concatenate([p[k] for p in parts], axis=0) for k in range(3))
    _assert_same(got, want, f"{mode} bands prepass={prepass}")
    assert int((want[0] < F32(1e6)).sum()) > 3000


@pytest.mark.gpu
@pytest.mark.parametrize("lit", [True, False])
def test_dropin_model_renderer_bilinear_perspective(lit):
    """Model.read_model of the torus fixture through Renderer with a texturing="pixel", texture_filter="bilinear",
    perspective_correct=True filler, rendered twice (the second frame reuses the cached coordinates and texture)."""
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller, GuroIllumination, NoIllumination, Renderer
    from cython3dmodelrenderer_b200.model import Model
    from oracle import ingest as I
    cwd = os.getcwd()
    os.chdir(os.path.join(GOLDEN, "obj"))
    try:
        model = Model.read_model("torus.obj")
    finally:
        os.chdir(cwd)
    vt = np.asarray(model._texture_coords, F32)
    vt3 = np.concatenate([vt[:, :2], np.zeros((vt.shape[0], 1), F32)], axis=1)
    uv = I.gather(vt3, model._triangles_texture_coords)
    o = TM().TexturedOracleFiller(256, 256, fov=45)
    o.render_arrays(model._vertices_by_triangles, uv, model._normals_by_triangles, texture=model._texture, perspective=True,
                    filter="bilinear")
    want = o.get_color_buffer().copy()
    if lit:
        O().guro(want, o.get_normals_buffer(), [0, 0, 1])
    ill = GuroIllumination([0, 0, 1]) if lit else NoIllumination()
    filler = AdvancedPixelBufferFiller(256, 256, fov=45, texturing="pixel", texture_filter="bilinear", perspective_correct=True)
    r = Renderer(filler, ill, None, 256, 256)
    for _ in range(2):
        got = r.render(model).copy()
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), f"lit={lit}"
    assert int((filler.get_z_buffer() < F32(1e6)).sum()) > 2000


@pytest.mark.gpu
def test_refusals():
    import torch
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller, _lib
    L = _lib.load_library()
    m, uv = _scene(4)
    v, c, n = _arrays(m)
    f = AdvancedPixelBufferFiller(64, 64)
    f._ensure_workspace(v.shape[0])
    dv, dc, dn = (torch.from_numpy(a).cuda() for a in (v, c, n))
    st = f._stream()
    img = torch.empty((64, 64, 3), dtype=torch.uint8, device="cuda")
    host = np.zeros((64, 64, 3), np.uint8)

    def calls(flags):
        return {
            "crb_render tiled": L.crb_render(f._handle, dv.data_ptr(), dc.data_ptr(), dn.data_ptr(), v.shape[0],
                                             flags | _lib.CRB_CLEAR_FIRST, st),
            "crb_render atomic": L.crb_render(f._handle, dv.data_ptr(), dc.data_ptr(), dn.data_ptr(), v.shape[0],
                                              flags | _lib.CRB_PATH_ATOMIC, st),
            "crb_render_host": L.crb_render_host(f._handle, v.ctypes.data, c.ctypes.data, n.ctypes.data, v.shape[0], flags, 0,
                                                 None, None, None, st),
            "crb_render_views": L.crb_render_views(f._handle, dv.data_ptr(), dc.data_ptr(), dn.data_ptr(), v.shape[0], None, 1,
                                                   None, None, None, img.data_ptr(), flags, None, st),
            "crb_render_image_host": L.crb_render_image_host(f._handle, v.ctypes.data, c.ctypes.data, n.ctypes.data,
                                                             v.shape[0], flags, None, img.data_ptr(), host.ctypes.data, None, st),
        }
    modes = (_lib.CRB_TEX_PERSPECTIVE, _lib.CRB_TEX_BILINEAR, _lib.CRB_TEX_PERSPECTIVE | _lib.CRB_TEX_BILINEAR)
    # a mode bit without CRB_TEXTURE: refused, with a texture bound or not
    packed = torch.zeros((4, 4), dtype=torch.int32, device="cuda")
    for bound in (False, True):
        if bound:
            assert L.crb_bind_texture(f._handle, packed.data_ptr(), 4, 4) == _lib.CRB_OK
        for bits in modes:
            for name, rc in calls(bits).items():
                assert rc == _lib.CRB_ERR_INVALID, (name, bits, bound, rc)
    # with CRB_TEXTURE and nothing bound: still CRB_ERR_STATE
    assert L.crb_bind_texture(f._handle, None, 0, 0) == _lib.CRB_OK
    for bits in modes:
        for name, rc in calls(bits | _lib.CRB_TEXTURE).items():
            assert rc == _lib.CRB_ERR_STATE, (name, bits, rc)
    torch.cuda.synchronize()
    # Python keywords
    for bad in ("cubic", "linear", None, 2):
        with pytest.raises(ValueError):
            AdvancedPixelBufferFiller(64, 64, texture_filter=bad)
    for bad in ("true", 1, None):
        with pytest.raises(ValueError):
            AdvancedPixelBufferFiller(64, 64, perspective_correct=bad)
    with pytest.raises(ValueError):
        AdvancedPixelBufferFiller(64, 64, texturing="bilinear")
