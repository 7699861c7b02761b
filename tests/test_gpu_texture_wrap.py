"""The wrap modes of per-pixel texturing, CRB_TEX_REPEAT and CRB_TEX_MIRROR, on the GPU, word for word against their oracle
(oracle/texture_wrap_oracle.py; DESIGN 2): every filter (nearest, bilinear, trilinear) from affine and perspective-correct
coordinates, on the tiled path in each rasterizer shape and on the atomic path, for scenes whose coordinates span several
periods and carry adversarial values; batched T-Rex orbit views lit and unlit with float32 and uint8 output; row bands; the
drop-in Model / Renderer flow; texture_wrap="clamp" against a filler built without the keyword; and the refusals.
"""
import ctypes
import os

import numpy as np
import pytest

from conftest import GOLDEN, bits_equal, load_indexed, random_scene
from test_gpu_texture import CONFIGS, _arrays, _assert_same, _base, _buffers, _trex_uvs
from test_texture_oracle import random_texture, random_uvs

F32 = np.float32
# texture_filter, perspective_correct
MODES = {"nearest": ("nearest", False), "nearest_persp": ("nearest", True), "bilinear": ("bilinear", False),
         "bilinear_persp": ("bilinear", True), "trilinear": ("trilinear", False), "trilinear_persp": ("trilinear", True)}
WRAPS = ("repeat", "mirror")
SEEDS = (3, 8)
TEXTURES = {3: (61, 47), 8: (256, 512)}


def O():
    from oracle import oracle
    return oracle


def WR():
    from oracle import texture_wrap_oracle
    return texture_wrap_oracle


def _filler(h, w, mode, wrap, **kw):
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller
    filt, persp = MODES[mode]
    return AdvancedPixelBufferFiller(h, w, texture_filter=filt, perspective_correct=persp, texture_wrap=wrap, **kw)


def _oracle(h, w, mode, wrap, v, uv, n, tex, fov=90.0, base=None):
    filt, persp = MODES[mode]
    o = WR().TexturedOracleFiller(h, w, fov=fov, wrap=wrap)
    if base is not None:
        o.render_arrays(*base)
    o.render_arrays(v, uv, n, texture=tex, perspective=persp, filter=filt)
    return o


def tiled_uvs(seed, T):
    """[T,3,3] coordinates over several periods: random_uvs' (a tenth adversarial: NaN, +-inf, +-1e10, 3e9, ...) stretched
    from [-0.2, 1.2] to about [-3, 4]."""
    uv = random_uvs(seed, T)
    with np.errstate(invalid="ignore", over="ignore"):
        uv[..., :2] = uv[..., :2] * F32(5) - F32(2)
    return uv


def _scene(seed):
    return random_scene(seed, T=600), tiled_uvs(seed, 600)


@pytest.fixture(scope="module")
def oracle_frames():
    cache = {}

    def get(mode, wrap, seed, composite):
        key = (mode, wrap, seed, composite)
        if key not in cache:
            m, uv = _scene(seed)
            o = _oracle(256, 256, mode, wrap, m._vertices_by_triangles, uv, m._normals_by_triangles,
                        random_texture(seed, *TEXTURES[seed]), base=_base() if composite else None)
            cache[key] = _buffers(o)
        return cache[key]
    return get


@pytest.mark.gpu
@pytest.mark.parametrize("wrap", WRAPS)
@pytest.mark.parametrize("mode", sorted(MODES))
@pytest.mark.parametrize("config", sorted(CONFIGS))
def test_wrap_scenes_bit_exact(config, mode, wrap, oracle_frames):
    """Seeded scenes whose coordinates span about seven periods, a tenth of them adversarial; fresh, and composited onto a
    per-vertex frame drawn by the same filler; host and device inputs, [T,3,3] and [T,3,2] coordinates."""
    import torch
    from cython3dmodelrenderer_b200 import _lib
    path = "atomic" if config == "atomic" else "tiled"
    for seed in SEEDS:
        m, uv = _scene(seed)
        tex = random_texture(seed, *TEXTURES[seed])
        for composite in (False, True):
            f = _filler(256, 256, mode, wrap)
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
            _assert_same(_buffers(f), oracle_frames(mode, wrap, seed, composite),
                         f"{mode} {wrap} seed {seed} {config} composite={composite}")


@pytest.mark.gpu
@pytest.mark.parametrize("wrap", WRAPS)
@pytest.mark.parametrize("mode", ["nearest", "bilinear_persp", "trilinear"])
@pytest.mark.parametrize("lit", [False, True])
def test_render_views_wrap_trex_orbit(lit, mode, wrap):
    """8 T-Rex orbit views at 256^2 with the spherical coordinates tiled four times: float32 slabs and the fused uint8 image
    against the oracle on the camera-space arrays of views.transform_arrays_host, then oracle.guro, the row flip and
    astype('uint8'); lit, also crb_render_image_host."""
    import torch
    from cython3dmodelrenderer_b200 import _lib, views as VW
    m = load_indexed("trex")
    uv = _trex_uvs(m) * F32(4) - F32(1.5)
    tex = random_texture(709, 97, 131)
    h = w = 256
    light = [0.3, -0.2, 1.0] if lit else None
    views = VW.orbit_views(128, first=0, count=8, stride=16)
    dv, dn = (torch.from_numpy(a).cuda() for a in (m._vertices_by_triangles, m._normals_by_triangles))
    f = _filler(h, w, mode, wrap, fov=45.0)
    out = f.render_views(dv, uv, dn, views, chunk=3, color_u8_out=True, guro_light=light, texture=tex)
    for k in range(len(views)):
        vk, nk = VW.transform_arrays_host(views[k], m._vertices_by_triangles, m._normals_by_triangles)
        want = _buffers(_oracle(h, w, mode, wrap, vk, uv, nk, tex, fov=45.0))
        if lit:
            O().guro(want[1], want[2], light)
        got = tuple(out[name][k].cpu().numpy() for name in ("z", "color", "normals"))
        _assert_same(got, want, f"{mode} {wrap} view {k} lit={lit}")
        with np.errstate(invalid="ignore"):
            want_u8 = want[1][::-1].astype("uint8")
        assert np.array_equal(out["color_u8"][k].cpu().numpy(), want_u8), f"{mode} {wrap} uint8 view {k} lit={lit}"
        assert int((want[0] < F32(1e6)).sum()) > 3000
    if lit:
        filt, persp = MODES[mode]
        bits = (_lib.CRB_TEXTURE | (_lib.CRB_TEX_PERSPECTIVE if persp else 0)
                | {"nearest": 0, "bilinear": _lib.CRB_TEX_BILINEAR, "trilinear": _lib.CRB_TEX_TRILINEAR}[filt]
                | (_lib.CRB_TEX_REPEAT if wrap == "repeat" else _lib.CRB_TEX_MIRROR))
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
        o = _oracle(h, w, mode, wrap, vk, uv3, nk, tex, fov=45.0)
        c = o.get_color_buffer().copy()
        O().guro(c, o.get_normals_buffer(), light)
        with np.errstate(invalid="ignore"):
            assert np.array_equal(image_host, c[::-1].astype("uint8"))


@pytest.mark.gpu
@pytest.mark.parametrize("wrap", WRAPS)
@pytest.mark.parametrize("mode", ["nearest_persp", "trilinear_persp"])
def test_wrap_bands_concatenate_to_full_frame(mode, wrap):
    import torch
    from cython3dmodelrenderer_b200 import _lib
    m = load_indexed("trex")
    uv = _trex_uvs(m) * F32(3) - F32(1)
    tex = random_texture(3, 333, 4097)
    h = w = 256
    want = _buffers(_oracle(h, w, mode, wrap, m._vertices_by_triangles, uv, m._normals_by_triangles, tex, fov=45.0))
    dv, dn = (torch.from_numpy(a).cuda() for a in (m._vertices_by_triangles, m._normals_by_triangles))
    duv = torch.from_numpy(uv).cuda()
    for prepass in (1, 0):
        parts = []
        for r0, r1 in ((0, 90), (90, 171), (171, 256)):
            f = _filler(h, w, mode, wrap, fov=45.0, band=(r0, r1))
            f.set_option(_lib.CRB_OPT_BAND_PREPASS, prepass)
            f.render_arrays(dv, duv, dn, texture=tex)
            parts.append(_buffers(f))
        got = tuple(np.concatenate([p[k] for p in parts], axis=0) for k in range(3))
        _assert_same(got, want, f"{mode} {wrap} bands prepass={prepass}")
    assert int((want[0] < F32(1e6)).sum()) > 3000


def _torus():
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
    return model, I.gather(vt3, model._triangles_texture_coords)


@pytest.mark.gpu
@pytest.mark.parametrize("wrap", WRAPS)
@pytest.mark.parametrize("mode", ["nearest", "bilinear", "trilinear_persp"])
@pytest.mark.parametrize("lit", [True, False])
def test_dropin_model_renderer_wrap(lit, mode, wrap):
    """Model.read_model of the torus fixture (its vt run from -0.01 to 1.01) through Renderer with a texturing="pixel" filler
    and texture_wrap=, rendered twice (the second frame reuses the cached coordinates and texture)."""
    from cython3dmodelrenderer_b200 import GuroIllumination, NoIllumination, Renderer
    model, uv = _torus()
    o = _oracle(256, 256, mode, wrap, model._vertices_by_triangles, uv, model._normals_by_triangles, model._texture, fov=45)
    want = o.get_color_buffer().copy()
    if lit:
        O().guro(want, o.get_normals_buffer(), [0, 0, 1])
    ill = GuroIllumination([0, 0, 1]) if lit else NoIllumination()
    filler = _filler(256, 256, mode, wrap, fov=45, texturing="pixel")
    r = Renderer(filler, ill, None, 256, 256)
    for _ in range(2):
        got = r.render(model).copy()
        assert bits_equal(got, want), f"{mode} {wrap} lit={lit}"
    assert int((filler.get_z_buffer() < F32(1e6)).sum()) > 2000


@pytest.mark.gpu
@pytest.mark.parametrize("mode", sorted(MODES))
def test_explicit_clamp_is_the_default(mode):
    """texture_wrap="clamp" renders exactly what a filler built without the keyword renders, on coordinates over several
    periods, through render_arrays on both paths and render_views."""
    import torch
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller, views as VW
    filt, persp = MODES[mode]
    m, uv = _scene(3)
    v, _, n = _arrays(m)
    tex = random_texture(3, 61, 47)
    frames = []
    for kw in ({}, {"texture_wrap": "clamp"}):
        for path in ("tiled", "atomic"):
            f = AdvancedPixelBufferFiller(256, 256, texture_filter=filt, perspective_correct=persp, **kw)
            f.render_arrays(v, uv, n, path=path, texture=tex)
            frames.append(_buffers(f))
        f = AdvancedPixelBufferFiller(128, 128, fov=45.0, texture_filter=filt, perspective_correct=persp, **kw)
        t = load_indexed("trex")
        dv, dn = (torch.from_numpy(a).cuda() for a in (t._vertices_by_triangles, t._normals_by_triangles))
        out = f.render_views(dv, _trex_uvs(t) * F32(4) - F32(1.5), dn, VW.orbit_views(128, first=0, count=4, stride=32),
                             color_u8_out=True, texture=tex)
        frames.append(tuple(out[name].cpu().numpy() for name in ("z", "color", "normals")))
        frames.append(out["color_u8"].cpu().numpy())
    for a, b in zip(frames[:4], frames[4:]):
        if isinstance(a, tuple):
            _assert_same(b, a, f"{mode} clamp")
        else:
            assert np.array_equal(a, b), mode


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
    REP, MIR, TEXB = _lib.CRB_TEX_REPEAT, _lib.CRB_TEX_MIRROR, _lib.CRB_TEXTURE
    texels = torch.zeros((4,), dtype=torch.int32, device="cuda")
    invalid = (REP, MIR, REP | MIR, REP | _lib.CRB_TEX_BILINEAR, MIR | _lib.CRB_TEX_PERSPECTIVE, TEXB | REP | MIR,
               TEXB | REP | MIR | _lib.CRB_TEX_TRILINEAR)
    for bound in (False, True):
        if bound:
            assert L.crb_bind_texture(f._handle, texels.data_ptr(), 2, 2) == _lib.CRB_OK
        for bits in invalid:
            for name, rc in calls(bits).items():
                assert rc == _lib.CRB_ERR_INVALID, (name, bits, bound, rc)
        if not bound:     # a valid wrap mode with no texture bound
            for bits in (TEXB | REP, TEXB | MIR):
                for name, rc in calls(bits).items():
                    assert rc == _lib.CRB_ERR_STATE, (name, bits, rc)
    for bits in (TEXB | REP, TEXB | MIR | _lib.CRB_TEX_BILINEAR):     # and with one bound they render
        for path in (_lib.CRB_CLEAR_FIRST, _lib.CRB_PATH_ATOMIC):
            rc = L.crb_render(f._handle, dv.data_ptr(), dc.data_ptr(), dn.data_ptr(), v.shape[0], bits | path, st)
            assert rc == _lib.CRB_OK, (bits, path, rc)
    torch.cuda.synchronize()
    for bad in ("Repeat", "wrap", "border", "clamp_to_edge", None, 1):
        with pytest.raises(ValueError):
            AdvancedPixelBufferFiller(64, 64, texture_wrap=bad)
    for wrap in ("clamp", "repeat", "mirror"):
        AdvancedPixelBufferFiller(64, 64, texture_filter="trilinear", perspective_correct=True, texture_wrap=wrap)
