"""Per-pixel texturing (CRB_TEXTURE) on the GPU, word for word against the textured oracle (oracle/texture_oracle.py).

DESIGN 2 defines the mode: visibility, depth and normals as in per-vertex mode; the colour of the winning fragment is the
texel its interpolated texture coordinates name under model.py:147-150's rule.  tests/test_texture_oracle.py checks the
oracle against that definition on the CPU; here every GPU path must give the oracle's bits: tiled and atomic, each
rasterizer shape, fresh and composited, the edge-case scene families, batched views with the fused Guro pass and uint8
output, row bands, and the drop-in Model / Renderer flow.
"""
import ctypes
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, ROOT, TriModel, bits_equal, case_model, load_indexed, random_scene
from test_texture_oracle import random_texture, random_uvs

F32 = np.float32
SIZES = [(256, 256), (200, 333)]
TEXTURES = [(1, 1), (1, 7), (7, 1), (709, 709), (333, 4097), (2048, 2048)]
CONFIGS = {"default": {}, "atomic": {}, "shape1": {"RASTER_SHAPE": 1}, "shape2": {"RASTER_SHAPE": 2},
           "shape3": {"RASTER_SHAPE": 3}}
SEEDS = (2, 5, 14)


def O():
    from oracle import oracle
    return oracle


def TO():
    from oracle import texture_oracle
    return texture_oracle


def _buffers(f):
    return f.get_z_buffer().copy(), f.get_color_buffer().copy(), f.get_normals_buffer().copy()


def _assert_same(got, want, what):
    for name, g, w in zip(("z", "color", "normals"), got, want):
        g, w = np.ascontiguousarray(g), np.ascontiguousarray(w)
        if not bits_equal(g, w):
            bad = np.argwhere(g.view(np.uint32) != w.view(np.uint32))
            raise AssertionError(f"{what}: {name} differs at {len(bad)} words, first {bad[:5].tolist()}: "
                                 f"got {g[tuple(bad[0])]!r} want {w[tuple(bad[0])]!r}")


def _arrays(m):
    return m._vertices_by_triangles, m._colors_by_triangles, m._normals_by_triangles


def _scene(seed):
    m = random_scene(seed, T=600)
    return m, random_uvs(seed, 600)


def _base():
    """The per-vertex frame the composited cases draw first."""
    return _arrays(random_scene(17, T=300))


@pytest.fixture(scope="module")
def oracle_frames():
    cache = {}

    def get(seed, size, tshape, composite):
        key = (seed, size, tshape, composite)
        if key not in cache:
            h, w = size
            m, uv = _scene(seed)
            o = TO().TexturedOracleFiller(h, w)
            if composite:
                o.render_arrays(*_base())
            o.render_arrays(m._vertices_by_triangles, uv, m._normals_by_triangles, texture=random_texture(seed, *tshape))
            cache[key] = _buffers(o)
        return cache[key]
    return get


@pytest.mark.gpu
@pytest.mark.parametrize("size", SIZES, ids=lambda s: f"{s[0]}x{s[1]}")
@pytest.mark.parametrize("tshape", TEXTURES, ids=lambda s: f"tex{s[0]}x{s[1]}")
@pytest.mark.parametrize("config", sorted(CONFIGS))
def test_textured_scenes_bit_exact(config, tshape, size, oracle_frames):
    """Seeded scenes with in-range and out-of-range coordinates; fresh, and composited onto a per-vertex frame drawn by the
    same filler; host and device inputs, [T,3,3] and [T,3,2] coordinates."""
    import torch
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller, _lib
    h, w = size
    path = "atomic" if config == "atomic" else "tiled"
    for seed in SEEDS:
        m, uv = _scene(seed)
        tex = random_texture(seed, *tshape)
        for composite in (False, True):
            f = AdvancedPixelBufferFiller(h, w)
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
            _assert_same(_buffers(f), oracle_frames(seed, size, tshape, composite),
                         f"seed {seed} {config} tex {tshape} {h}x{w} composite={composite}")


@pytest.mark.gpu
@pytest.mark.parametrize("size", SIZES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_edge_families_textured(size):
    import test_gpu_edges as E
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller
    h, w = size
    for i, name in enumerate(sorted(E.FAMILIES)):
        m = E.family(name, h, w)
        v, _, n = _arrays(m)
        uv = random_uvs(50 + i, v.shape[0])
        tex = random_texture(i, 61, 83)
        o = TO().TexturedOracleFiller(h, w, fov=E.FOV)
        o.render_arrays(v, uv, n, texture=tex)
        for path in ("tiled", "atomic"):
            f = AdvancedPixelBufferFiller(h, w, fov=E.FOV)
            f.render_arrays(v, uv, n, path=path, texture=tex)
            _assert_same(_buffers(f), _buffers(o), f"family {name} {path} {h}x{w}")


def _trex_uvs(m):
    from cython3dmodelrenderer_b200 import synthetic
    return synthetic.spherical_uvs(m._vertices_by_triangles)


@pytest.mark.gpu
@pytest.mark.parametrize("lit", [False, True])
def test_render_views_textured_trex_orbit(lit):
    """8 T-Rex orbit views at 1024^2: float32 slabs and the fused uint8 image, against the oracle on the camera-space arrays
    of views.transform_arrays_host (then oracle.guro, the row flip and astype('uint8'))."""
    import torch
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller, views as VW
    m = load_indexed("trex")
    uv = _trex_uvs(m)
    tex = random_texture(709, 709, 709)
    h = w = 1024
    light = [0.3, -0.2, 1.0] if lit else None
    views = VW.orbit_views(128, first=0, count=8, stride=16)
    dv, dn = (torch.from_numpy(a).cuda() for a in (m._vertices_by_triangles, m._normals_by_triangles))
    f = AdvancedPixelBufferFiller(h, w, fov=45.0)
    out = f.render_views(dv, uv, dn, views, chunk=3, color_u8_out=True, guro_light=light, texture=tex)
    for k in range(len(views)):
        vk, nk = VW.transform_arrays_host(views[k], m._vertices_by_triangles, m._normals_by_triangles)
        o = TO().TexturedOracleFiller(h, w, fov=45.0)
        o.render_arrays(vk, uv, nk, texture=tex)
        want = _buffers(o)
        if lit:
            O().guro(want[1], want[2], light)
        got = tuple(out[name][k].cpu().numpy() for name in ("z", "color", "normals"))
        _assert_same(got, want, f"view {k} lit={lit}")
        with np.errstate(invalid="ignore"):
            want_u8 = want[1][::-1].astype("uint8")
        assert np.array_equal(out["color_u8"][k].cpu().numpy(), want_u8), f"uint8 view {k} lit={lit}"
        assert int((want[0] < F32(1e6)).sum()) > 100000
    if lit:
        # crb_render_image_host with CRB_TEXTURE: host arrays in, run.py's flipped uint8 image out, one view
        from cython3dmodelrenderer_b200 import _lib
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
                                              _lib.CRB_GURO | _lib.CRB_TEXTURE, la, image_dev.data_ptr(),
                                              image_host.ctypes.data, None, f._stream()))
        o = TO().TexturedOracleFiller(h, w, fov=45.0)
        o.render_arrays(vk, uv3, nk, texture=tex)
        c = o.get_color_buffer().copy()
        O().guro(c, o.get_normals_buffer(), light)
        with np.errstate(invalid="ignore"):
            assert np.array_equal(image_host, c[::-1].astype("uint8"))


@pytest.mark.gpu
@pytest.mark.parametrize("prepass", [1, 0])
def test_textured_bands_concatenate_to_full_frame(prepass):
    import torch
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller, _lib
    m = load_indexed("trex")
    uv = _trex_uvs(m)
    tex = random_texture(3, 333, 4097)
    h = w = 256
    o = TO().TexturedOracleFiller(h, w, fov=45.0)
    o.render_arrays(m._vertices_by_triangles, uv, m._normals_by_triangles, texture=tex)
    want = _buffers(o)
    dv, dn = (torch.from_numpy(a).cuda() for a in (m._vertices_by_triangles, m._normals_by_triangles))
    duv = torch.from_numpy(uv).cuda()
    parts = []
    for r0, r1 in ((0, 90), (90, 171), (171, 256)):
        f = AdvancedPixelBufferFiller(h, w, fov=45.0, band=(r0, r1))
        f.set_option(_lib.CRB_OPT_BAND_PREPASS, prepass)
        f.render_arrays(dv, duv, dn, texture=tex)
        parts.append(_buffers(f))
    got = tuple(np.concatenate([p[k] for p in parts], axis=0) for k in range(3))
    _assert_same(got, want, f"bands prepass={prepass}")
    assert int((want[0] < F32(1e6)).sum()) > 3000


def _torus_oracle(model, light):
    from oracle import ingest as I
    vt = np.asarray(model._texture_coords, F32)
    vt3 = np.concatenate([vt[:, :2], np.zeros((vt.shape[0], 1), F32)], axis=1)
    uv = I.gather(vt3, model._triangles_texture_coords)
    o = TO().TexturedOracleFiller(256, 256, fov=45)
    o.render_arrays(model._vertices_by_triangles, uv, model._normals_by_triangles, texture=model._texture)
    c = o.get_color_buffer().copy()
    if light is not None:
        O().guro(c, o.get_normals_buffer(), light)
    return c


@pytest.mark.gpu
@pytest.mark.parametrize("lit", [True, False])
def test_dropin_model_renderer_pixel_texturing(lit):
    """Model.read_model of the torus fixture (its .mtl names checker.png) through Renderer with a texturing="pixel" filler."""
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller, GuroIllumination, NoIllumination, Renderer
    from cython3dmodelrenderer_b200.model import Model
    cwd = os.getcwd()
    os.chdir(os.path.join(GOLDEN, "obj"))
    try:
        model = Model.read_model("torus.obj")
    finally:
        os.chdir(cwd)
    assert model._texture is not None and model._texture.shape[2] == 3      # (the torus sits in front of the camera as read)
    ill = GuroIllumination([0, 0, 1]) if lit else NoIllumination()
    filler = AdvancedPixelBufferFiller(256, 256, fov=45, texturing="pixel")
    r = Renderer(filler, ill, None, 256, 256)
    want = _torus_oracle(model, [0, 0, 1] if lit else None)
    for _ in range(2):      # the second frame reuses the cached coordinates and texture
        got = r.render(model).copy()
        assert bits_equal(got, want), f"lit={lit}"
    assert int((filler.get_z_buffer() < F32(1e6)).sum()) > 2000


def _golden_cases():
    cases = json.load(open(os.path.join(GOLDEN, "checksums.json")))["cases"]
    return sorted(k for k, c in cases.items() if "z" in c and "+" not in c["model"] and not c["model"].startswith("uv_sphere")
                  and c["h"] * c["w"] <= 1024 * 1024)


@pytest.mark.gpu
@pytest.mark.parametrize("case", _golden_cases())
def test_vertex_mode_unchanged_with_a_texture_bound(case):
    """A per-vertex render of a filler that has a texture bound (its previous frame was textured) gives the golden bits."""
    import hashlib
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller
    info = json.load(open(os.path.join(GOLDEN, "checksums.json")))["cases"][case]
    m, _ = case_model(info)
    sha = lambda a: hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()    # noqa: E731
    f = AdvancedPixelBufferFiller(info["h"], info["w"], fov=info["fov"])
    v, c, n = _arrays(m)
    f.render_arrays(v, random_uvs(1, v.shape[0]), n, texture=random_texture(1, 64, 64))
    f.clear()
    f.render_model(m)
    assert (sha(f.get_z_buffer()), sha(f.get_color_buffer()), sha(f.get_normals_buffer())) == \
        (info["z"], info["color"], info["normals"])


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
    # CRB_TEXTURE with nothing bound
    assert L.crb_render(f._handle, dv.data_ptr(), dc.data_ptr(), dn.data_ptr(), v.shape[0],
                        _lib.CRB_TEXTURE | _lib.CRB_CLEAR_FIRST, st) == _lib.CRB_ERR_STATE
    assert L.crb_render(f._handle, dv.data_ptr(), dc.data_ptr(), dn.data_ptr(), v.shape[0],
                        _lib.CRB_TEXTURE | _lib.CRB_PATH_ATOMIC, st) == _lib.CRB_ERR_STATE
    assert L.crb_render_views(f._handle, dv.data_ptr(), dc.data_ptr(), dn.data_ptr(), v.shape[0], None, 1, None, None,
                              None, None, _lib.CRB_TEXTURE, None, st) == _lib.CRB_ERR_STATE
    img = torch.empty((64, 64, 3), dtype=torch.uint8, device="cuda")
    host = np.zeros((64, 64, 3), np.uint8)
    assert L.crb_render_image_host(f._handle, v.ctypes.data, c.ctypes.data, n.ctypes.data, v.shape[0], _lib.CRB_TEXTURE,
                                   None, img.data_ptr(), host.ctypes.data, None, st) == _lib.CRB_ERR_STATE
    assert L.crb_render_host(f._handle, v.ctypes.data, c.ctypes.data, n.ctypes.data, v.shape[0], _lib.CRB_TEXTURE, 0,
                             None, None, None, st) == _lib.CRB_ERR_STATE
    # bad bind / pack arguments
    packed = torch.zeros((4, 4), dtype=torch.int32, device="cuda")
    bgr = torch.zeros((4, 4, 3), dtype=torch.uint8, device="cuda")
    for th, tw in ((0, 4), (4, 0), (-1, 4), (65536, 32768)):
        assert L.crb_bind_texture(f._handle, packed.data_ptr(), th, tw) == _lib.CRB_ERR_INVALID
        assert L.crb_pack_texture(bgr.data_ptr(), th, tw, packed.data_ptr(), st) == _lib.CRB_ERR_INVALID
    assert L.crb_bind_texture(f._handle, packed.data_ptr() + 2, 4, 4) == _lib.CRB_ERR_INVALID
    assert L.crb_bind_texture(None, packed.data_ptr(), 4, 4) == _lib.CRB_ERR_INVALID
    assert L.crb_pack_texture(None, 4, 4, packed.data_ptr(), st) == _lib.CRB_ERR_INVALID
    assert L.crb_pack_texture(bgr.data_ptr(), 4, 4, None, st) == _lib.CRB_ERR_INVALID
    # bound, then unbound again: refused again
    assert L.crb_pack_texture(bgr.data_ptr(), 4, 4, packed.data_ptr(), st) == _lib.CRB_OK
    assert L.crb_bind_texture(f._handle, packed.data_ptr(), 4, 4) == _lib.CRB_OK
    assert L.crb_bind_texture(f._handle, None, 0, 0) == _lib.CRB_OK
    assert L.crb_render(f._handle, dv.data_ptr(), dc.data_ptr(), dn.data_ptr(), v.shape[0],
                        _lib.CRB_TEXTURE | _lib.CRB_CLEAR_FIRST, st) == _lib.CRB_ERR_STATE
    torch.cuda.synchronize()
    # Python: wrong texture dtype / shape, wrong coordinate shape, untextured model in pixel mode
    for bad in (np.zeros((4, 4, 3), np.float32), np.zeros((4, 4), np.uint8), np.zeros((4, 4, 4), np.uint8),
                np.zeros((0, 4, 3), np.uint8)):
        with pytest.raises(ValueError):
            f.render_arrays(v, uv, n, texture=bad)
        with pytest.raises(ValueError):
            f.render_views(dv, torch.from_numpy(uv).cuda(), dn, np.eye(4, dtype=F32).ravel()[None, :16].copy(), texture=bad)
    with pytest.raises(ValueError):
        f.render_arrays(v, np.zeros((v.shape[0], 3, 4), F32), n, texture=np.zeros((4, 4, 3), np.uint8))
    with pytest.raises(ValueError):
        f.render_arrays(v, uv.astype(np.float64), n, texture=np.zeros((4, 4, 3), np.uint8))
    with pytest.raises(ValueError):
        AdvancedPixelBufferFiller(64, 64, texturing="bilinear")
    with pytest.raises(ValueError):
        AdvancedPixelBufferFiller(64, 64, texturing="pixel").render_model(m)       # TriModel: no texture at all
    from cython3dmodelrenderer_b200.model import Model
    tri = np.array([[0, 1, 2]], np.int32)
    untextured = Model(np.array([[0, 0, 1], [1, 0, 1], [0, 1, 1]], F32), tri)
    with pytest.raises(ValueError):
        AdvancedPixelBufferFiller(64, 64, texturing="pixel").render_model(untextured)
