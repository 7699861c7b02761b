"""Trilinear mip filtering, CRB_TEX_TRILINEAR, on the GPU, word for word against its oracle (oracle/texture_mip_oracle.py;
DESIGN 2), affine ("trilinear") and perspective-correct ("trilinear_persp").

The same ground as test_gpu_texture_filter: tiled and atomic paths, each rasterizer shape, fresh and composited, host and
device inputs, the edge-case scene families, batched T-Rex orbit views at 1024^2 and at 256^2 (where the texture is minified)
with the fused Guro pass and uint8 output, crb_render_image_host, row bands, the drop-in Model / Renderer flow and the
refusals; and the chain kernel against mip_chain, and per-vertex, nearest and bilinear frames unchanged with a chain bound.
"""
import ctypes
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, load_indexed
from test_gpu_texture import (CONFIGS, SEEDS, SIZES, TEXTURES, _arrays, _assert_same, _base, _buffers, _golden_cases, _scene,
                              _trex_uvs, case_model)
from test_texture_oracle import random_texture, random_uvs

F32 = np.float32
MODES = {"trilinear": False, "trilinear_persp": True}


def O():
    from oracle import oracle
    return oracle


def MIP():
    from oracle import texture_mip_oracle
    return texture_mip_oracle


def _filler(h, w, mode, **kw):
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller
    return AdvancedPixelBufferFiller(h, w, texture_filter="trilinear", perspective_correct=MODES[mode], **kw)


def _oracle(h, w, mode, v, uv, n, tex, fov=90.0, base=None):
    o = MIP().TexturedOracleFiller(h, w, fov=fov)
    if base is not None:
        o.render_arrays(*base)
    o.render_arrays(v, uv, n, texture=tex, perspective=MODES[mode], filter="trilinear")
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
def test_trilinear_scenes_bit_exact(config, tshape, size, mode, oracle_frames):
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
def test_edge_families_trilinear(size, mode):
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
@pytest.mark.parametrize("res", [1024, 256])
@pytest.mark.parametrize("lit", [False, True])
def test_render_views_trilinear_trex_orbit(lit, res, mode):
    """8 T-Rex orbit views: float32 slabs and the fused uint8 image against the oracle on the camera-space arrays of
    views.transform_arrays_host, then oracle.guro, the row flip and astype('uint8'); lit, also crb_render_image_host."""
    import torch
    from cython3dmodelrenderer_b200 import _lib, views as VW
    m = load_indexed("trex")
    uv = _trex_uvs(m)
    tex = random_texture(709, 709, 709)
    h = w = res
    light = [0.3, -0.2, 1.0] if lit else None
    views = VW.orbit_views(128, first=0, count=8, stride=16)
    dv, dn = (torch.from_numpy(a).cuda() for a in (m._vertices_by_triangles, m._normals_by_triangles))
    f = _filler(h, w, mode, fov=45.0)
    out = f.render_views(dv, uv, dn, views, chunk=3, color_u8_out=True, guro_light=light, texture=tex)
    minified = 0
    for k in range(len(views)):
        vk, nk = VW.transform_arrays_host(views[k], m._vertices_by_triangles, m._normals_by_triangles)
        o = MIP().TexturedOracleFiller(h, w, fov=45.0)
        ids, lam, lc = MIP().render_textured(o, vk, uv, nk, tex, perspective=MODES[mode], return_lod=True)
        minified += int((lc > 0).sum())
        want = _buffers(o)
        if lit:
            O().guro(want[1], want[2], light)
        got = tuple(out[name][k].cpu().numpy() for name in ("z", "color", "normals"))
        _assert_same(got, want, f"{mode} view {k} lit={lit} {res}")
        with np.errstate(invalid="ignore"):
            want_u8 = want[1][::-1].astype("uint8")
        assert np.array_equal(out["color_u8"][k].cpu().numpy(), want_u8), f"{mode} uint8 view {k} lit={lit} {res}"
    assert minified > 1000
    if lit:
        bits = _lib.CRB_TEXTURE | _lib.CRB_TEX_TRILINEAR | (_lib.CRB_TEX_PERSPECTIVE if MODES[mode] else 0)
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
def test_trilinear_bands_concatenate_to_full_frame(prepass, mode):
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
@pytest.mark.parametrize("mode", sorted(MODES))
@pytest.mark.parametrize("lit", [True, False])
def test_dropin_model_renderer_trilinear(lit, mode):
    """Model.read_model of the torus fixture through Renderer with a texture_filter="trilinear" filler, rendered twice (the
    second frame reuses the cached coordinates and chain)."""
    from cython3dmodelrenderer_b200 import GuroIllumination, NoIllumination, Renderer
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
    o = _oracle(256, 256, mode, model._vertices_by_triangles, uv, model._normals_by_triangles, model._texture, fov=45)
    want = o.get_color_buffer().copy()
    if lit:
        O().guro(want, o.get_normals_buffer(), [0, 0, 1])
    ill = GuroIllumination([0, 0, 1]) if lit else NoIllumination()
    filler = _filler(256, 256, mode, fov=45, texturing="pixel")
    r = Renderer(filler, ill, None, 256, 256)
    for _ in range(2):
        got = r.render(model).copy()
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), f"{mode} lit={lit}"
    assert int((filler.get_z_buffer() < F32(1e6)).sum()) > 2000


@pytest.mark.gpu
@pytest.mark.parametrize("tshape", TEXTURES, ids=lambda s: f"tex{s[0]}x{s[1]}")
def test_chain_kernel_matches_mip_chain(tshape):
    import torch
    from cython3dmodelrenderer_b200 import _lib
    L = _lib.load_library()
    th, tw = tshape
    tex = random_texture(th * 7 + tw, th, tw)
    levels, texels = ctypes.c_int(), ctypes.c_int64()
    assert L.crb_mip_layout(th, tw, ctypes.byref(levels), ctypes.byref(texels)) == _lib.CRB_OK
    want = MIP().pack_chain(MIP().mip_chain(tex))
    assert (levels.value, texels.value) == (MIP().levels_of(th, tw), want.size)
    out = torch.full((want.size + 1,), -1, dtype=torch.int32, device="cuda")
    bgr = torch.from_numpy(tex).cuda()
    _lib.check(L.crb_pack_texture_mips(bgr.data_ptr(), th, tw, out.data_ptr(), None))
    got = out.cpu().numpy().view(np.uint32)
    assert np.array_equal(got[:-1], want), tshape
    assert got[-1] == 0xFFFFFFFF       # nothing written past the chain


@pytest.mark.gpu
@pytest.mark.parametrize("case", _golden_cases())
def test_vertex_mode_unchanged_with_a_chain_bound(case):
    """A per-vertex render of a filler whose previous frame bound a mip chain gives the golden bits."""
    info = json.load(open(os.path.join(GOLDEN, "checksums.json")))["cases"][case]
    m, _ = case_model(info)
    sha = lambda a: hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()    # noqa: E731
    f = _filler(info["h"], info["w"], "trilinear", fov=info["fov"])
    v, c, n = _arrays(m)
    f.render_arrays(v, random_uvs(1, v.shape[0]), n, texture=random_texture(1, 64, 64))
    f.clear()
    f.render_model(m)
    assert (sha(f.get_z_buffer()), sha(f.get_color_buffer()), sha(f.get_normals_buffer())) == \
        (info["z"], info["color"], info["normals"])


@pytest.mark.gpu
@pytest.mark.parametrize("tshape", [(1, 7), (709, 709), (333, 4097)], ids=lambda s: f"tex{s[0]}x{s[1]}")
def test_nearest_and_bilinear_unchanged_with_a_chain_bound(tshape):
    """Nearest and bilinear frames (affine and perspective) sample level 0 of a bound chain exactly as the packed texture
    bound by crb_bind_texture."""
    import torch
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller, _lib
    L = _lib.load_library()
    m, uv = _scene(2)
    v, _, n = _arrays(m)
    th, tw = tshape
    tex = random_texture(5, th, tw)
    bgr = torch.from_numpy(tex).cuda()
    texels = ctypes.c_int64()
    _lib.check(L.crb_mip_layout(th, tw, None, ctypes.byref(texels)))
    chain = torch.empty((texels.value,), dtype=torch.int32, device="cuda")
    single = torch.empty((th, tw), dtype=torch.int32, device="cuda")
    _lib.check(L.crb_pack_texture_mips(bgr.data_ptr(), th, tw, chain.data_ptr(), None))
    _lib.check(L.crb_pack_texture(bgr.data_ptr(), th, tw, single.data_ptr(), None))
    torch.cuda.synchronize()
    dv, dn = (torch.from_numpy(a).cuda() for a in (v, n))
    duv = torch.from_numpy(uv).cuda()
    for bits in (0, _lib.CRB_TEX_PERSPECTIVE, _lib.CRB_TEX_BILINEAR, _lib.CRB_TEX_BILINEAR | _lib.CRB_TEX_PERSPECTIVE):
        frames = []
        for bind, ptr in ((L.crb_bind_texture, single), (L.crb_bind_texture_mips, chain)):
            f = AdvancedPixelBufferFiller(256, 256)
            f._ensure_workspace(v.shape[0])
            _lib.check(bind(f._handle, ptr.data_ptr(), th, tw))
            for path in (_lib.CRB_CLEAR_FIRST, _lib.CRB_CLEAR_FIRST | _lib.CRB_PATH_ATOMIC):
                _lib.check(L.crb_render(f._handle, dv.data_ptr(), duv.data_ptr(), dn.data_ptr(), v.shape[0],
                                        path | _lib.CRB_TEXTURE | bits, f._stream()))
                torch.cuda.synchronize()
                frames.append(_buffers(f))
        for a, b in zip(frames[:2], frames[2:]):
            _assert_same(a, b, f"bits {bits} {tshape}")


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
    TRI, TEXB = _lib.CRB_TEX_TRILINEAR, _lib.CRB_TEXTURE
    chain = torch.zeros((8,), dtype=torch.int32, device="cuda")      # a 4 x 4 chain has 16 + 4 + 1 texels; 2 x 2: 4 + 1
    for bound in (None, "single", "chain"):
        if bound == "single":
            assert L.crb_bind_texture(f._handle, chain.data_ptr(), 2, 2) == _lib.CRB_OK
        elif bound == "chain":
            assert L.crb_bind_texture_mips(f._handle, chain.data_ptr(), 2, 2) == _lib.CRB_OK
        for bits in (TRI, TRI | _lib.CRB_TEX_PERSPECTIVE, TEXB | TRI | _lib.CRB_TEX_BILINEAR):   # invalid combinations
            for name, rc in calls(bits).items():
                assert rc == _lib.CRB_ERR_INVALID, (name, bits, bound, rc)
        if bound != "chain":     # CRB_TEX_TRILINEAR with no chain bound
            for bits in (TEXB | TRI, TEXB | TRI | _lib.CRB_TEX_PERSPECTIVE):
                for name, rc in calls(bits).items():
                    assert rc == _lib.CRB_ERR_STATE, (name, bits, bound, rc)
    # a single level bound after a chain replaces it
    assert L.crb_bind_texture(f._handle, chain.data_ptr(), 2, 2) == _lib.CRB_OK
    for name, rc in calls(TEXB | TRI).items():
        assert rc == _lib.CRB_ERR_STATE, (name, rc)
    assert L.crb_bind_texture_mips(f._handle, None, 0, 0) == _lib.CRB_OK
    for name, rc in calls(TEXB).items():
        assert rc == _lib.CRB_ERR_STATE, (name, rc)
    torch.cuda.synchronize()
    # layout / pack / bind arguments
    lv, tx = ctypes.c_int(), ctypes.c_int64()
    for th, tw in ((0, 4), (4, 0), (-1, 4), (65536, 32768), (1, 1 << 30 | 1)):
        assert L.crb_mip_layout(th, tw, ctypes.byref(lv), ctypes.byref(tx)) == _lib.CRB_ERR_INVALID, (th, tw)
        assert L.crb_bind_texture_mips(f._handle, chain.data_ptr(), th, tw) == _lib.CRB_ERR_INVALID, (th, tw)
        assert L.crb_pack_texture_mips(img.data_ptr(), th, tw, chain.data_ptr(), None) == _lib.CRB_ERR_INVALID, (th, tw)
    assert L.crb_mip_layout(1, (1 << 30) - 1, ctypes.byref(lv), ctypes.byref(tx)) == _lib.CRB_OK
    assert (lv.value, tx.value) == (30, sum((1 << k) - 1 for k in range(1, 31)))
    assert L.crb_pack_texture_mips(None, 2, 2, chain.data_ptr(), None) == _lib.CRB_ERR_INVALID
    assert L.crb_pack_texture_mips(img.data_ptr(), 2, 2, None, None) == _lib.CRB_ERR_INVALID
    assert L.crb_bind_texture_mips(f._handle, ctypes.c_void_p(chain.data_ptr() + 2), 2, 2) == _lib.CRB_ERR_INVALID
    torch.cuda.synchronize()
    # Python keywords
    for bad in ("Trilinear", "mip", "anisotropic"):
        with pytest.raises(ValueError):
            AdvancedPixelBufferFiller(64, 64, texture_filter=bad)
    for persp in (False, True):
        AdvancedPixelBufferFiller(64, 64, texture_filter="trilinear", perspective_correct=persp)
