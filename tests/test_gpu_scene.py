"""Scenes in batched views (crb_render_scene_views, render_views(objects=...); DESIGN 2) on the GPU, word for word against
oracle/scene_oracle.py: each view's camera-space triangles, chosen and transformed per object, rendered by the pinned oracles.

Covered: the T-Rex, bunny and basketball with a generated floor and walls (K = 2...8, random rigid poses per view, object
boundaries that are not multiples of 256), 300 one-triangle objects (a chunk spans hundreds of objects), interleaved object
indices with hidden objects and indices outside [0, K); the two equivalences with crb_render_views_ids on the T-Rex orbit at
1024^2 with 128 views, and the slow equivalent path (per view, crb_transform_view per object, then one untransformed view);
every chunking, the launch pipeline and defer_join; the three rasterizer shapes with Guro; every texture filter and
interpolation with a wrap mode; supersampling; near_clip with cameras inside a room; band fillers; an overflowing frame and
its redraw; the refusals.
"""
import ctypes

import numpy as np
import pytest

from conftest import load_indexed, random_scene

F32 = np.float32
LIGHT = [0.3, -0.2, 1.0]
SENTINEL = 0x5EED1D5


def SC():
    from oracle import scene_oracle
    return scene_oracle


def VW():
    from cython3dmodelrenderer_b200 import views
    return views


def _device(*arrays):
    import torch
    return tuple(torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays)


def _filler(h, w, fov=45.0, z_near=0.1, opts=None, **kw):
    from cython3dmodelrenderer_b200 import AdvancedPixelBufferFiller, _lib
    f = AdvancedPixelBufferFiller(h, w, fov=fov, z_near=z_near, **kw)
    for opt, val in (opts or {}).items():
        f.set_option(getattr(_lib, "CRB_OPT_" + opt), val)
    return f


def _words(got, want, what):
    got = got.cpu().numpy() if hasattr(got, "cpu") else np.asarray(got)
    got, want = np.ascontiguousarray(got), np.ascontiguousarray(want)
    assert got.shape == want.shape, f"{what}: shape {got.shape} != {want.shape}"
    ok = got.view(np.uint32) == want.view(np.uint32) if got.dtype.itemsize == 4 else got == want
    if not ok.all():
        bad = np.argwhere(~ok)
        raise AssertionError(f"{what}: {len(bad)} words differ, first {bad[:5].tolist()}: got {got[tuple(bad[0])]!r} "
                             f"want {want[tuple(bad[0])]!r}")


def u8(colour):
    with np.errstate(invalid="ignore"):
        return np.ascontiguousarray(colour[::-1].astype("uint8"))


def lit(o):
    from oracle import oracle as O
    c = o.color_buffer.copy()
    O.guro(c, o.normals_buffer, LIGHT)
    return c


def _torch_equal(a, b):
    import torch
    if a.dtype == torch.float32:
        a, b = a.view(torch.int32), b.view(torch.int32)
    return torch.equal(a, b)


# ---------------------------------------------------------------------------------------------------------------- scenes
def grid(nx, nz, size, rng):
    """A quad grid of 2*nx*nz triangles in the plane y = 0 about the origin, normals +y, random colours"""
    xs = np.linspace(-size / 2, size / 2, nx + 1)
    zs = np.linspace(-size / 2, size / 2, nz + 1)
    tris = []
    for i in range(nx):
        for j in range(nz):
            a, b = (xs[i], 0.0, zs[j]), (xs[i + 1], 0.0, zs[j])
            c, d = (xs[i + 1], 0.0, zs[j + 1]), (xs[i], 0.0, zs[j + 1])
            tris += [(a, c, b), (a, d, c)]
    v = np.array(tris, F32)
    n = np.zeros_like(v)
    n[..., 1] = 1.0
    return v, (rng.random(v.shape) * 255).astype(F32), n


def _model(name, scale):
    m = load_indexed(name)
    v = m._vertices_by_triangles
    ctr = (v.reshape(-1, 3).min(0) + v.reshape(-1, 3).max(0)) / 2
    return ((v - ctr) * F32(scale)).astype(F32), m._colors_by_triangles, m._normals_by_triangles


def _wall(rng, R):
    v, c, n = grid(6, 4, 2.4, rng)
    R = np.asarray(R, F32)
    return (v @ R.T).astype(F32), c, (n @ R.T).astype(F32)


def room_objects(K, seed=0):
    """K (2..8) objects about their own origins: the T-Rex, a floor, the bunny, the basketball, three walls facing inwards
    and a small grid (boundaries 13814, 13942, ... are not multiples of 256)"""
    rng = np.random.default_rng(seed)
    rx = lambda a: np.array([[1, 0, 0], [0, np.cos(a), -np.sin(a)], [0, np.sin(a), np.cos(a)]])
    objs = [_model("trex", 1.0), grid(16, 16, 4.0, rng), _model("bunny", 0.8), _model("basketball", 0.4),
            _wall(rng, rx(-np.pi / 2)), _wall(rng, VW().rot_y(np.pi / 2) @ rx(-np.pi / 2)),
            _wall(rng, VW().rot_y(-np.pi / 2) @ rx(-np.pi / 2)), grid(3, 5, 0.5, rng)]
    return objs[:K]


HOME = [(0.0, 0.2, 0.0), (0.0, -0.4, 0.0), (0.9, 0.1, 0.5), (-0.9, 0.0, -0.4), (0.0, 0.5, 1.8), (-1.8, 0.5, 0.0),
        (1.8, 0.5, 0.0), (0.3, 0.4, -0.9)]


def _rot(axis, angle):
    axis = np.asarray(axis, np.float64) / np.linalg.norm(axis)
    K_ = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    return np.eye(3) + np.sin(angle) * K_ + (1 - np.cos(angle)) * K_ @ K_


def cameras(V, dist=3.2, pitch=-0.4, height=0.0):
    """An orbit about the world origin, looking down by `pitch` (floor normals then face the camera)"""
    rx = np.array([[1, 0, 0], [0, np.cos(pitch), -np.sin(pitch)], [0, np.sin(pitch), np.cos(pitch)]])
    return np.stack([VW().view_matrix(rx @ VW().rot_y(2 * np.pi * k / V + 0.3), p=(0.0, height, 0.0), q=(0.0, 0.0, dist))
                     for k in range(V)]).astype(F32)


def random_poses(V, K, seed):
    """Random rigid poses per view: turns about y (objects 0 and 2..: about a random axis) and jitter about HOME"""
    rng = np.random.default_rng(seed)
    out = np.zeros((V, K, 16), F32)
    for v in range(V):
        for k in range(K):
            R = VW().rot_y(rng.uniform(0, 2 * np.pi)) if k in (1, 4, 5, 6) else _rot(rng.standard_normal(3), rng.uniform(0, 2 * np.pi))
            q = np.asarray(HOME[k]) + (rng.uniform(-0.15, 0.15, 3) if k not in (1, 4, 5, 6) else 0.0)
            out[v, k] = VW().view_matrix(R, p=(0.0, 0.0, 0.0), q=q)
    return out


def models_scene(K, V, seed):
    v, c, n, tri_obj = VW().concat_meshes(room_objects(K, seed))
    return v, c, n, tri_obj, VW().scene_views(cameras(V), random_poses(V, K, seed))


def tiny_scene(V, seed=4, K=300):
    """K one-triangle objects: every chunk of 256 triangles spans 256 objects"""
    m = random_scene(seed, T=K)
    v = m._vertices_by_triangles - np.array([0.0, 0.0, 2.5], F32)
    rng = np.random.default_rng(seed)
    poses = np.zeros((V, K, 16), F32)
    for i in range(V):
        for k in range(K):
            poses[i, k] = VW().view_matrix(_rot(rng.standard_normal(3), rng.uniform(-0.4, 0.4)), p=(0.0, 0.0, 0.0),
                                           q=rng.uniform(-0.1, 0.1, 3))
    cams = np.stack([VW().view_matrix(VW().rot_y(0.2 * k), p=(0.0, 0.0, 0.0), q=(0.0, 0.0, 2.5)) for k in range(V)]).astype(F32)
    return v, m._colors_by_triangles, m._normals_by_triangles, np.arange(K, dtype=np.int32), VW().scene_views(cams, poses)


def interleaved_scene(V, seed=6, K=7):
    """Objects interleaved triangle by triangle, some indices outside [0, K), and hidden objects (pads 1, NaN; -0 shown)"""
    v, c, n, _, views = models_scene(4, V, seed)
    rng = np.random.default_rng(seed)
    tri_obj = rng.integers(0, K, len(v)).astype(np.int32)
    tri_obj[::13] = K
    tri_obj[3::29] = -5
    views = np.concatenate([views, views[:, :K - 4]], axis=1)
    views[0, 2, 15] = F32(1.0)
    views[1 % V, 5, 15] = F32(np.nan)
    views[2 % V, 1, 15] = -F32(0.0)
    return v, c, n, tri_obj, views


SCENES = {"models_K2": lambda V: models_scene(2, V, 1), "models_K5": lambda V: models_scene(5, V, 2),
          "models_K8": lambda V: models_scene(8, V, 3), "tiny300": tiny_scene, "interleaved": interleaved_scene}
H = W = 256
VIEWS = 10
_CACHE = {}


def scene(name, V=VIEWS, h=H, w=W):
    key = (name, V, h, w)
    if key not in _CACHE:
        v, c, n, tri_obj, views = SCENES[name](V)
        frames = [SC().render(h, w, v, c, n, tri_obj, views[k], fov=45.0) for k in range(V)]
        _CACHE[key] = (v, c, n, tri_obj, views, frames)
    return _CACHE[key]


def assert_views(out, frames, what, bary=True):
    for k, (o, ids, b) in enumerate(frames):
        w = f"{what} view {k}"
        _words(out["z"][k], o.z_buffer, w + ": z")
        _words(out["color"][k], o.color_buffer, w + ": colour")
        _words(out["normals"][k], o.normals_buffer, w + ": normals")
        _words(out["triangle_id"][k], ids.astype(np.int32), w + ": tri_id")
        if bary:
            _words(out["barycentrics"][k], b, w + ": bary")
        if "color_u8" in out:
            _words(out["color_u8"][k], u8(o.color_buffer), w + ": color_u8")


ALL = ("z", "color", "normals", "triangle_id", "barycentrics")


# ---------------------------------------------------------------------------------------------------------------- oracle
@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(SCENES))
@pytest.mark.parametrize("chunk", [1, 7, 32, 128])
@pytest.mark.parametrize("pipeline", [0, 1])
def test_scenes_against_oracle(name, chunk, pipeline):
    """Every output of every view, every chunking, the launch pipeline on and off; defer_join + join() once per case"""
    v, c, n, tri_obj, views, frames = scene(name)
    assert sum(int((ids >= 0).sum()) for _, ids, _ in frames) > 20000
    f = _filler(H, W, opts={"CHUNK_PIPELINE": pipeline})
    dv, dc, dn = _device(v, c, n)
    for defer in (False, True):
        out = f.render_views(dv, dc, dn, views, want=ALL, color_u8_out=True, chunk=chunk, objects=tri_obj,
                             check_status=not defer, defer_join=defer)
        if defer:
            f.join()
        assert_views(out, frames, f"{name} chunk={chunk} pipeline={pipeline} defer={defer}")


@pytest.mark.gpu
def test_object_of_a_pixel_is_one_gather():
    import torch
    v, c, n, tri_obj, views, frames = scene("interleaved")
    f = _filler(H, W)
    dv, dc, dn, dobj = _device(v, c, n, tri_obj)
    out = f.render_views(dv, dc, dn, torch.from_numpy(views).cuda(), want=("triangle_id",), objects=dobj)
    ids = out["triangle_id"]
    obj = torch.where(ids >= 0, dobj[ids.clamp(min=0).long()], torch.full_like(ids, -1))
    for k, (_, oids, _) in enumerate(frames):
        want = np.where(oids >= 0, tri_obj[np.maximum(oids, 0)], -1).astype(np.int32)
        _words(obj[k], want, f"view {k}: object of each pixel")
        with np.errstate(invalid="ignore"):
            hidden = np.flatnonzero(~(views[k, :, 15] == 0))
        assert not np.isin(want, hidden).any() and not np.isin(want, [7, -5]).any()


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [1, 2, 3])
def test_raster_shapes_with_guro(shape):
    v, c, n, tri_obj, views, frames = scene("models_K8")
    f = _filler(H, W, opts={"RASTER_SHAPE": shape})
    out = f.render_views(*_device(v, c, n), views, want=("color", "triangle_id"), color_u8_out=True, guro_light=LIGHT,
                         chunk=4, objects=tri_obj)
    for k, (o, ids, _) in enumerate(frames):
        _words(out["color"][k], lit(o), f"shape {shape} view {k}: lit colour")
        _words(out["color_u8"][k], u8(lit(o)), f"shape {shape} view {k}: lit uint8")
        _words(out["triangle_id"][k], ids.astype(np.int32), f"shape {shape} view {k}: tri_id")


@pytest.mark.gpu
@pytest.mark.parametrize("perspective", [False, True])
@pytest.mark.parametrize("filt", ["nearest", "bilinear", "trilinear"])
def test_textured(filt, perspective):
    from oracle import texture_wrap_oracle as WR
    v, c, n, tri_obj, views = models_scene(5, 3, 7)
    rng = np.random.default_rng(5)
    uv = rng.uniform(-1.5, 2.5, (len(v), 3, 2)).astype(F32)
    uv3 = np.concatenate([uv, np.zeros(uv.shape[:2] + (1,), F32)], axis=2)
    tex = rng.integers(0, 256, (37, 53, 3), dtype=np.uint8)
    f = _filler(H, W, texture_filter=filt, perspective_correct=perspective, texture_wrap="repeat")
    out = f.render_views(*_device(v, uv3, n), views, texture=tex, want=("color", "triangle_id"), color_u8_out=True,
                         objects=tri_obj, chunk=2)
    for k in range(3):
        ofill = WR.TexturedOracleFiller(H, W, fov=45.0, wrap="repeat")
        o, ids, _ = SC().render(H, W, v, uv3, n, tri_obj, views[k], fov=45.0, filler=ofill, texture=tex,
                                perspective=perspective, filter=filt)
        what = f"{filt} perspective={perspective} view {k}"
        _words(out["color"][k], o.color_buffer, what + ": colour")
        _words(out["color_u8"][k], u8(o.color_buffer), what + ": uint8")
        _words(out["triangle_id"][k], ids.astype(np.int32), what + ": tri_id")


@pytest.mark.gpu
@pytest.mark.parametrize("s", [2, 4])
def test_supersampled(s):
    v, c, n, tri_obj, views = models_scene(6, 3, 8)
    f = _filler(128 * s, 128 * s)
    for light in (None, LIGHT):
        out = f.render_views(*_device(v, c, n), views, color_u8_out=True, supersample=s, guro_light=light, objects=tri_obj,
                             chunk=2)
        for k in range(3):
            want = SC().render_resolved(128, 128, s, v, c, n, tri_obj, views[k], fov=45.0, light=light)
            _words(out["color_u8"][k], want, f"SS{s} light={light} view {k}")


def inside_room(V, seed=9):
    """Cameras inside the room, 0.25 above the floor and looking down a little: the floor crosses z_near under every camera"""
    v, c, n, tri_obj, _ = models_scene(7, V, seed)
    rng = np.random.default_rng(seed)
    poses = random_poses(V, 7, seed)
    poses[:, 1, 13] = F32(-0.25)                               # floor 0.25 below the cameras' height
    cams = np.stack([VW().view_matrix(np.array([[1, 0, 0], [0, np.cos(-0.3), np.sin(0.3)], [0, np.sin(-0.3), np.cos(-0.3)]])
                                      @ VW().rot_y(rng.uniform(0, 2 * np.pi)), p=(rng.uniform(-0.3, 0.3), 0.0, rng.uniform(-0.3, 0.3)),
                                      q=(0.0, 0.0, 0.0)) for _ in range(V)]).astype(F32)
    return v, c, n, tri_obj, VW().scene_views(cams, poses)


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [1, 4])
def test_near_clip_inside_a_room(chunk):
    V, zn = 4, 0.05
    v, c, n, tri_obj, views = inside_room(V)
    f = _filler(H, W, 60.0, zn, near_clip=True)
    out = f.render_views(*_device(v, c, n), views, want=("z", "color", "normals", "triangle_id"), color_u8_out=True,
                         objects=tri_obj, chunk=chunk)
    crossing = 0
    for k in range(V):
        o, ids, _ = SC().render(H, W, v, c, n, tri_obj, views[k], fov=60.0, z_near=zn, near_clip=True)
        cv, _, _, _ = SC().camera_space(v, c, n, tri_obj, views[k])
        crossing += int(((cv[..., 2] < zn).any(axis=1) & (cv[..., 2] >= zn).any(axis=1)).sum())
        what = f"near_clip chunk={chunk} view {k}"
        _words(out["z"][k], o.z_buffer, what + ": z")
        _words(out["color"][k], o.color_buffer, what + ": colour")
        _words(out["normals"][k], o.normals_buffer, what + ": normals")
        _words(out["triangle_id"][k], ids.astype(np.int32), what + ": tri_id")
        _words(out["color_u8"][k], u8(o.color_buffer), what + ": uint8")
        assert (ids >= 0).sum() > 5000
    assert crossing > 50


@pytest.mark.gpu
@pytest.mark.parametrize("bands", [((0, 128), (128, 256)), ((0, 77), (77, 150), (150, 256))])
def test_band_fillers(bands):
    import torch
    v, c, n, tri_obj, views, frames = scene("models_K5", V=3)
    parts = []
    for r0, r1 in bands:
        f = _filler(H, W, band=(r0, r1))
        parts.append(f.render_views(*_device(v, c, n), views, want=ALL, objects=tri_obj, chunk=2))
    out = {name: torch.cat([p[name] for p in parts], dim=1) for name in ALL}
    assert_views(out, frames, f"bands {bands}")


@pytest.mark.gpu
def test_row_exchange_into_two_buffers():
    import torch
    v, c, n, tri_obj, views, frames = scene("models_K8", V=3)
    f = _filler(H, W)
    bufs = [torch.zeros((3, H // 2, W, 3), dtype=torch.uint8, device="cuda") for _ in range(2)]
    f.render_views(*_device(v, c, n), views, want=(), objects=tri_obj, chunk=2, u8_exchange=(H // 2, [b.data_ptr() for b in bufs]))
    torch.cuda.synchronize()
    img = torch.cat(bufs, dim=1)
    for k, (o, _, _) in enumerate(frames):
        _words(img[k], u8(o.color_buffer), f"row exchange view {k}")


# ---------------------------------------------------------------------------------------------------------------- equivalences
def _orbit_outputs(f, dv, dc, dn, views, objects=None):
    import torch
    out = f.render_views(dv, dc, dn, views, want=ALL, color_u8_out=True, chunk=32, objects=objects)
    torch.cuda.synchronize()
    return out


@pytest.mark.gpu
def test_equivalences_trex_orbit_1024_128_views():
    """K = 1 with tri_obj all 0, and K = 5 (interleaved objects) with every views[v, k] = views[v]: crb_render_views_ids bit for
    bit in every output"""
    import torch
    m = load_indexed("trex")
    dv, dc, dn = _device(m._vertices_by_triangles, m._colors_by_triangles, m._normals_by_triangles)
    T = dv.shape[0]
    views = torch.from_numpy(VW().orbit_views(128)).cuda()
    f = _filler(1024, 1024)
    want = _orbit_outputs(f, dv, dc, dn, views)
    assert int((want["z"] < 1e5).sum()) > 1000000
    one = _orbit_outputs(f, dv, dc, dn, views[:, None, :].contiguous(), torch.zeros(T, dtype=torch.int32, device="cuda"))
    rng = np.random.default_rng(0)
    objs = torch.from_numpy(rng.integers(0, 5, T).astype(np.int32)).cuda()
    five = _orbit_outputs(f, dv, dc, dn, views[:, None, :].expand(128, 5, 16).contiguous(), objs)
    for name in want:
        assert _torch_equal(one[name], want[name]), f"K = 1: {name} differs from crb_render_views_ids"
        assert _torch_equal(five[name], want[name]), f"K = 5, equal transforms: {name} differs from crb_render_views_ids"


def slow_path(f, dv, dc, dn, tri_obj, views):
    """What a caller without scenes does: per view, crb_transform_view per object (contiguous runs of tri_obj) into one
    camera-space buffer, then a single-view crb_render_views with views = NULL into that view's slab"""
    import torch
    from cython3dmodelrenderer_b200 import _lib
    V = views.shape[0]
    T = dv.shape[0]
    runs = np.flatnonzero(np.diff(tri_obj)) + 1
    starts, stops = np.concatenate([[0], runs]), np.concatenate([runs, [T]])
    rows = f.row1 - f.row0
    z = torch.empty((V, rows, f.w), dtype=torch.float32, device="cuda")
    col = torch.empty((V, rows, f.w, 3), dtype=torch.float32, device="cuda")
    nor = torch.empty((V, rows, f.w, 3), dtype=torch.float32, device="cuda")
    cv, cn = torch.empty_like(dv), torch.empty_like(dn)
    f._ensure_workspace(T, 1)
    L, Hd, st = f._L, f._handle, f._stream()
    for k in range(V):
        for a, b in zip(starts, stops):
            _lib.check(L.crb_transform_view(Hd, dv[a:b].data_ptr(), dn[a:b].data_ptr(), int(b - a),
                                            views[k, int(tri_obj[a])].data_ptr(), cv[a:b].data_ptr(), cn[a:b].data_ptr(), st))
        _lib.check(L.crb_render_views(Hd, cv.data_ptr(), dc.data_ptr(), cn.data_ptr(), T, None, 1, z[k].data_ptr(),
                                      col[k].data_ptr(), nor[k].data_ptr(), None, 0, None, st))
    torch.cuda.synchronize()
    return {"z": z, "color": col, "normals": nor}


@pytest.mark.gpu
def test_slow_equivalent_path_models_1024():
    import torch
    V = 16
    v, c, n, tri_obj, views = models_scene(8, V, 12)
    dv, dc, dn = _device(v, c, n)
    dviews = torch.from_numpy(views).cuda()
    f = _filler(1024, 1024)
    out = f.render_views(dv, dc, dn, dviews, objects=tri_obj, chunk=8)
    slow = slow_path(_filler(1024, 1024), dv, dc, dn, tri_obj, dviews)
    for name in ("z", "color", "normals"):
        assert _torch_equal(out[name], slow[name]), f"{name} differs from the slow equivalent path"
    assert int((out["z"] < 1e5).sum()) > V * 200000


# ---------------------------------------------------------------------------------------------------------------- overflow
@pytest.mark.gpu
def test_overflowing_frame_leaves_outputs_untouched_and_is_redrawn():
    import torch
    from cython3dmodelrenderer_b200 import _lib
    v, c, n, tri_obj, views, frames = scene("models_K5", V=3)
    dv, dc, dn, dobj = _device(v, c, n, tri_obj)
    dviews = torch.from_numpy(views).cuda()
    T = dv.shape[0]
    f = _filler(H, W)
    L, Hd = f._L, f._handle
    nbytes = L.crb_workspace_bytes(Hd, T, 3, 64)
    ws = torch.empty(nbytes + 256, dtype=torch.uint8, device="cuda")
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(L.crb_bind_workspace(Hd, (ws.data_ptr() + 255) // 256 * 256, nbytes, T, 3, 64, st))
    z = torch.full((3, H, W), 7.0, device="cuda")
    col = torch.full((3, H, W, 3), 7.0, device="cuda")
    u = torch.full((3, H, W, 3), 7, dtype=torch.uint8, device="cuda")
    tri = torch.full((3, H, W), SENTINEL, dtype=torch.int32, device="cuda")
    _lib.check(L.crb_render_scene_views(Hd, dv.data_ptr(), dc.data_ptr(), dn.data_ptr(), T, dobj.data_ptr(), views.shape[1],
                                        dviews.data_ptr(), 3, z.data_ptr(), col.data_ptr(), None, u.data_ptr(), tri.data_ptr(),
                                        None, 0, None, st))
    need, cap = ctypes.c_int64(), ctypes.c_int64()
    assert L.crb_status(Hd, ctypes.byref(need), ctypes.byref(cap), st) == _lib.CRB_ERR_OVERFLOW
    assert (z == 7.0).all() and (col == 7.0).all() and (u == 7).all() and (tri == SENTINEL).all()
    # the filler's loop with a pair list too small: the frame is drawn again with the room it asked for
    fr = _filler(H, W)
    fr._ensure_workspace(T, 3, 64)
    assert fr._pair_cap < 1000
    out = fr.render_views(dv, dc, dn, dviews, want=ALL, objects=dobj, chunk=3)
    assert fr._pair_cap > 1000
    assert_views(out, frames, "after overflow")


# ---------------------------------------------------------------------------------------------------------------- refusals
@pytest.mark.gpu
def test_refusals():
    import torch
    from cython3dmodelrenderer_b200 import _lib
    v, c, n, tri_obj, views = models_scene(3, 2, 13)
    dv, dc, dn, dobj = _device(v, c, n, tri_obj)
    dviews = torch.from_numpy(views).cuda()
    T, K = dv.shape[0], views.shape[1]
    f = _filler(64, 64, triangle_ids=True)
    f._ensure_workspace(2 * T, 2)
    L, Hd = f._L, f._handle
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    z = torch.empty((2, 64, 64), device="cuda")
    bary = torch.empty((2, 64, 64, 3), device="cuda")
    INV = _lib.CRB_ERR_INVALID
    CF = _lib.CRB_CLEAR_FIRST

    def call(obj=dobj.data_ptr(), k=K, vw=dviews.data_ptr(), nv=2, flags=CF, b=None):
        return L.crb_render_scene_views(Hd, dv.data_ptr(), dc.data_ptr(), dn.data_ptr(), T, obj, k, vw, nv, z.data_ptr(), None,
                                        None, None, None, b, flags, None, st)
    launches = f.launch_count
    assert call(k=0) == INV and call(k=-1) == INV
    assert call(obj=None) == INV and call(vw=None) == INV
    assert call(obj=dobj.data_ptr() + 2) == INV
    assert call(flags=CF | _lib.CRB_PATH_ATOMIC) == INV
    assert call(k=2 ** 31 - 1, nv=2 ** 31 - 1) == INV
    assert call(nv=-1) == INV                                             # crb_render_views_ids' refusals apply
    assert call(flags=CF | _lib.CRB_CLIP_NEAR, b=bary.data_ptr()) == INV
    assert call(flags=CF | _lib.CRB_SS2) == INV
    assert f.launch_count == launches
    _lib.check(call())
    torch.cuda.synchronize()
    # the Python surface, before anything is queued
    launches = f.launch_count
    for bad in (tri_obj.astype(np.int64), tri_obj[:-1], tri_obj[None], tri_obj.astype(F32), torch.from_numpy(tri_obj).long()):
        with pytest.raises(ValueError):
            f.render_views(dv, dc, dn, dviews, objects=bad)
    for bad_views in (views[:, 0], views[..., :15], views.reshape(2, K, 4, 4), np.zeros((2, 0, 16), F32)):
        with pytest.raises(ValueError):
            f.render_views(dv, dc, dn, bad_views, objects=tri_obj)
    with pytest.raises(ValueError):
        f.render_views(dv, dc, dn, dviews)                                   # [V,K,16] without objects
    assert f.launch_count == launches
