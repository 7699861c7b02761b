"""Drop-in `AdvancedPixelBufferFiller` backed by libcrender_b200.so (hand-written sm_100a CUDA).

Mirrors the reference extension type
(crender/cy/pixel_buffer_filler/advanced_pixel_buffer_filler.pyx:20-253): same constructor, `get_size`,
`render_model`, `get_normals_buffer`, `get_color_buffer`, `get_z_buffer`, same errors, same persistent
(compositing) buffers, same live-view contract for the returned arrays.  PyTorch only owns memory
(device buffers, workspace, pinned host mirrors) and supplies the stream; all work happens behind the
C ABI (include/crender_b200.h).  There is no CPU fallback.
"""
import ctypes

import numpy as np

from . import _lib
from ._lib import check


def _require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("cython3dmodelrenderer_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch


def _check_texture(texture):
    """A texture for per-pixel texturing: uint8 [h,w,3] (what cv2.imread returns, BGR), as NumPy array or torch tensor."""
    import torch
    if isinstance(texture, torch.Tensor):
        ok = texture.dtype == torch.uint8 and texture.dim() == 3 and texture.shape[2] == 3
    else:
        texture = np.asarray(texture)
        ok = texture.dtype == np.uint8 and texture.ndim == 3 and texture.shape[2] == 3
    if not ok or texture.shape[0] < 1 or texture.shape[1] < 1:
        raise ValueError("texture must be a uint8 [h,w,3] image (what cv2.imread returns)")
    return texture


def _check_tri_array(a, name):
    """Same acceptance rules as the reference's `float[:, :, :]` memoryviews (pyx:94-96)."""
    if a is None:
        # `model._colors_by_triangles.copy()` on an untextured model (pyx:95)
        raise AttributeError("'NoneType' object has no attribute 'copy'")
    a = np.asarray(a)
    if a.dtype != np.float32:
        got = {"float64": "double", "int32": "int", "int64": "long", "float16": "npy_half",
               "uint8": "unsigned char"}.get(a.dtype.name, a.dtype.name)
        raise ValueError(f"Buffer dtype mismatch, expected 'float' but got '{got}'")
    if a.ndim != 3:
        raise ValueError(f"Buffer has wrong number of dimensions (expected 3, got {a.ndim})")
    if a.shape[1:] != (3, 3):
        raise ValueError(f"{name}: expected shape [T,3,3], got {tuple(a.shape)}")
    return a


class _HostArrays:
    """Host arrays a caller renders again and again (the reference idiom: one Model, a new filler per frame) are page-locked in
    place on their second sighting (crb_host_register) and then read by the GPU directly, instead of being copied into a pinned
    staging buffer every frame (0.15 ms of a 0.9 ms T-Rex frame).  Arrays that are new every frame (a model that is rotated
    between frames) are never registered -- page-locking costs more than one copy.  A weakref finalizer releases the
    registration with the array."""
    MAX_SEEN, MIN_BYTES = 256, 64 << 10
    seen = {}            # (address, nbytes) -> sightings
    registered = {}      # address -> nbytes

    @classmethod
    def pinned(cls, L, a):
        """True if `a` (C-contiguous float32 ndarray) is page-locked by an earlier call; counts the sighting otherwise."""
        import weakref
        ptr, nb = a.ctypes.data, a.nbytes
        if cls.registered.get(ptr) == nb:
            return True
        if nb < cls.MIN_BYTES or not a.flags.writeable:
            return False
        key = (ptr, nb)
        n = cls.seen.get(key, 0) + 1
        if len(cls.seen) > cls.MAX_SEEN:
            cls.seen.clear()
        cls.seen[key] = n
        if n >= 2 and ptr not in cls.registered:
            if L.crb_host_register(ctypes.c_void_p(ptr), ctypes.c_size_t(nb)) == _lib.CRB_OK:
                cls.registered[ptr] = nb
                try:
                    weakref.finalize(a, cls._release, L, ptr)
                except TypeError:          # an object that cannot be weakly referenced: do not keep its memory locked
                    cls._release(L, ptr)
            cls.seen.pop(key, None)
        return False      # (this call still copies: the registration serves the next one)

    @classmethod
    def _release(cls, L, ptr):
        if cls.registered.pop(ptr, None) is not None:
            try:
                L.crb_host_unregister(ctypes.c_void_p(ptr))
            except Exception:
                pass


class _DevicePointer:
    """CUDA array interface over a raw device address (memory owned elsewhere, e.g. a frame mapped from another rank)."""

    def __init__(self, ptr, shape, typestr="<f4"):
        self.__cuda_array_interface__ = {"shape": tuple(int(x) for x in shape), "typestr": typestr, "data": (int(ptr), False),
                                         "version": 3, "strides": None}


def wrap_device_pointer(torch, ptr, shape, device, dtype=None):
    """torch tensor (float32, or uint8 with dtype=torch.uint8) of `shape` over the device address `ptr` (no copy, no ownership)."""
    dtype = dtype or torch.float32
    if any(int(x) == 0 for x in shape):
        return torch.empty(tuple(shape), dtype=dtype, device=device)
    # no device argument: torch takes the device that owns the memory from the pointer itself (for a frame mapped from
    # another rank that is the peer GPU; naming the local device here would make as_tensor copy instead of alias)
    return torch.as_tensor(_DevicePointer(ptr, shape, "|u1" if dtype == torch.uint8 else "<f4"))


class AdvancedPixelBufferFiller:
    """B200 implementation of the Version C filler.  `n_threads` is accepted and ignored.

    Extra keywords (not in the reference): `device` -- CUDA device index (default: torch's current device),
    `band=(row0,row1)` -- own only those rows of the h x w image (screen-band sharding), `out_ptrs=(z, color, normals)` --
    raw device addresses of existing [rows,w], [rows,w,3], [rows,w,3] float32 buffers to render into instead of buffers of
    its own (e.g. this band's rows inside another rank's frame, sharding.PeerFrame); their content is taken as it is.
    `texturing="pixel"` -- render_model samples the model's texture at every pixel (per-pixel texturing, DESIGN 2) instead
    of blending the colours upstream looks up at the vertices ("vertex", the default and upstream's behaviour).
    `texture_filter="nearest" | "bilinear" | "trilinear"` and `perspective_correct=False | True` -- how every textured render of
    this filler (render_model with texturing="pixel", render_arrays / render_views with texture=) samples: the nearest texel, a
    bilinear blend of four (CRB_TEX_BILINEAR), or a blend of bilinear samples of the two levels of the texture's mip chain that
    the pixel's footprint in the texture selects (CRB_TEX_TRILINEAR; the chain is built on the device when the texture is bound),
    from texture coordinates interpolated affinely in screen space or perspective-correctly (CRB_TEX_PERSPECTIVE).
    """

    PAGEABLE_MIN_BYTES = 8 << 20      # host arrays of at least this size go up through the library's threaded staging ring
    # Download prefetch: the buffers the caller fetched after the previous frame (of this filler, or -- a new filler per frame is
    # the reference's idiom, run.py:21 -- of the filler before this one) start travelling to their host mirrors as soon as the
    # frame is rendered, back to back, instead of one by one when get_*_buffer() asks for them.
    _fetched_by_previous = frozenset()
    _fetched_by_current = set()
    _view_owner = {}      # address of a host mirror handed out by get_*_buffer() -> weak reference to its filler (owner_of_views)

    def __init__(self, h, w, fov=90.0, z_near=0.1, z_far=1000.0, n_threads=1, device=None, band=None, out_ptrs=None,
                 texturing="vertex", texture_filter="nearest", perspective_correct=False):
        if texturing not in ("vertex", "pixel"):
            raise ValueError(f"texturing must be 'vertex' or 'pixel', got {texturing!r}")
        if not isinstance(texture_filter, str) or texture_filter not in ("nearest", "bilinear", "trilinear"):
            raise ValueError(f"texture_filter must be 'nearest', 'bilinear' or 'trilinear', got {texture_filter!r}")
        if not isinstance(perspective_correct, (bool, np.bool_)):
            raise ValueError(f"perspective_correct must be True or False, got {perspective_correct!r}")
        self._texturing = texturing
        # render flags of every textured frame (kept in the arguments of a frame, so a redraw of it samples the same way)
        self._tex_flags = (_lib.CRB_TEXTURE | (_lib.CRB_TEX_BILINEAR if texture_filter == "bilinear" else 0)
                           | (_lib.CRB_TEX_TRILINEAR if texture_filter == "trilinear" else 0)
                           | (_lib.CRB_TEX_PERSPECTIVE if perspective_correct else 0))
        # (source texture, its version, packed uint32 CUDA tensor: [th,tw], or with "trilinear" the whole mip chain) bound to the filler
        self._tex = None
        self._uv = None               # (texture coordinates, their triangle indices, UV-by-triangle CUDA tensor [T,3,3])
        torch = _require_cuda()
        self._torch = torch
        self._L = _lib.load_library()
        self.h, self.w = int(h), int(w)   # pyx:40-41 `<int>h`
        self.n_threads = n_threads
        self._device = torch.cuda.current_device() if device is None else int(device)
        self._dev = torch.device("cuda", self._device)
        handle = ctypes.c_void_p()
        check(self._L.crb_create(self.h, self.w, float(fov), float(z_near), float(z_far), self._device,
                                 ctypes.byref(handle)))
        self._handle = handle
        self.row0, self.row1 = (0, self.h) if band is None else (int(band[0]), int(band[1]))
        if band is not None:
            check(self._L.crb_set_band(self._handle, self.row0, self.row1))
        rows = self.row1 - self.row0
        with torch.cuda.device(self._dev):
            # pyx:65-67: normals 0, colour 0, z = 1e6
            if out_ptrs is None:
                self._z = torch.empty((rows, self.w), dtype=torch.float32, device=self._dev)
                self._color = torch.empty((rows, self.w, 3), dtype=torch.float32, device=self._dev)
                self._normals = torch.empty((rows, self.w, 3), dtype=torch.float32, device=self._dev)
            else:
                self._z = wrap_device_pointer(torch, out_ptrs[0], (rows, self.w), self._dev)
                self._color = wrap_device_pointer(torch, out_ptrs[1], (rows, self.w, 3), self._dev)
                self._normals = wrap_device_pointer(torch, out_ptrs[2], (rows, self.w, 3), self._dev)
            check(self._L.crb_bind_buffers(self._handle, self._z.data_ptr(), self._color.data_ptr(),
                                           self._normals.data_ptr()))
        self._ws = None
        self._ws_T = -1
        self._ws_views = 1
        self._pair_cap = 0
        self._stage = None            # pinned host staging for the three input arrays
        self._host = {}               # name -> pinned torch tensor (host mirror); numpy views in _host_np
        self._host_np = {}
        self._stale = {"z": True, "color": True, "normals": True}   # device newer than host mirror
        self._exposed = set()         # mirrors handed to the caller (may have been written through)
        # pyx:65-67 (normals 0, colour 0, z = 1e6): the fresh-filler values are not stored here -- they materialise fused into
        # the first render's tile pass, or with the first read if nothing was rendered (a new filler per frame is the
        # reference's idiom, run.py:21, so the constructor queues no kernel at all)
        self._pending_clear = out_ptrs is None
        self._status = None           # pinned status words of the last frame (crb_status_async)
        self._unchecked = None        # the last render, until its status words have been looked at (see _validate)
        self._deferred_keep = None    # inputs of a batch issued with defer_join (see render_views)
        self._prefetched = set()      # mirrors whose download is already queued behind the last render
        self._fetched = None          # names fetched since this filler's last render (None: nothing rendered yet)
        cls = type(self)
        cls._fetched_by_previous, cls._fetched_by_current = frozenset(cls._fetched_by_current), set()

    # ------------------------------------------------------------------------------------------------ plumbing
    def __del__(self):
        try:
            for t in getattr(self, "_host", {}).values():       # (pinned memory is recycled: drop this filler's addresses)
                r = type(self)._view_owner.get(t.data_ptr())
                if r is not None and r() in (None, self):
                    type(self)._view_owner.pop(t.data_ptr(), None)
        except Exception:
            pass
        try:
            if getattr(self, "_handle", None):
                self._L.crb_destroy(self._handle)
                self._handle = None
        except Exception:
            pass

    def _stream(self):
        return ctypes.c_void_p(self._torch.cuda.current_stream(self._dev).cuda_stream)

    def _ensure_workspace(self, T, views=1, pair_cap=0):
        if self._ws is not None and T <= self._ws_T and views <= self._ws_views and pair_cap <= self._pair_cap:
            return
        torch = self._torch
        T = max(int(T), self._ws_T, 1)
        views = max(int(views), self._ws_views)
        pair_cap = max(int(pair_cap), self._pair_cap if pair_cap else 0)
        if self._ws is not None:
            check(self._L.crb_join(self._handle, self._stream()))     # deferred rasterizer work still uses the old workspace
        torch.cuda.current_stream(self._dev).synchronize()
        nbytes = self._L.crb_workspace_bytes(self._handle, T, views, pair_cap)
        with torch.cuda.device(self._dev):
            ws = torch.empty(nbytes + 256, dtype=torch.uint8, device=self._dev)
        ptr = (ws.data_ptr() + 255) // 256 * 256
        check(self._L.crb_bind_workspace(self._handle, ptr, nbytes, T, views, pair_cap, self._stream()))
        self._ws, self._ws_T, self._ws_views = ws, T, views
        self._pair_cap = int(self._L.crb_pair_capacity(self._handle))

    def _mirror(self, name):
        if name not in self._host:
            src = {"z": self._z, "color": self._color, "normals": self._normals}[name]
            t = self._torch.empty(src.shape, dtype=self._torch.float32, pin_memory=True)
            self._host[name] = t
            self._host_np[name] = t.numpy()
            import weakref
            type(self)._view_owner[t.data_ptr()] = weakref.ref(self)
        return self._host[name]

    @classmethod
    def owner_of_views(cls, color_buffer, n_buffer):
        """The filler whose live views the two arrays are -- the very objects its get_color_buffer() and get_normals_buffer()
        return -- or None.  (illumination.GuroIllumination uses it to light the device buffers behind the views.)"""
        try:
            ref = cls._view_owner.get(int(color_buffer.__array_interface__["data"][0]))
        except (AttributeError, KeyError, TypeError):
            return None
        f = ref() if ref is not None else None
        if f is None or f._host_np.get("color") is not color_buffer or f._host_np.get("normals") is not n_buffer:
            return None
        return f

    def _push_exposed(self):
        """Live-view contract (pyx:246-253 return views of the filler's own memory): whatever the caller wrote
        through a returned array is part of the buffers the next render composites into."""
        if not self._exposed:
            return
        mask, ptrs = 0, {"z": None, "color": None, "normals": None}
        for name, bit in (("z", _lib.CRB_BUF_Z), ("color", _lib.CRB_BUF_COLOR), ("normals", _lib.CRB_BUF_NORMALS)):
            if name in self._exposed and not self._stale[name]:
                mask |= bit
                ptrs[name] = self._host[name].data_ptr()
        if mask:
            check(self._L.crb_upload(self._handle, mask, ptrs["z"], ptrs["color"], ptrs["normals"], self._stream()))

    def _materialize_clear(self):
        if self._pending_clear:          # clear() with no render since: materialise the fresh-filler state
            check(self._L.crb_init_buffers(self._handle, self._stream()))
            self._pending_clear = False

    def _validate(self):
        """The overflow check of the last render, deferred to the first point that looks at its result: the status words
        came back asynchronously (crb_status_async); a frame whose (triangle, tile) pairs did not fit the workspace was
        skipped as a whole (buffers untouched) and is drawn again with the room it asked for."""
        u = self._unchecked
        if u is None:
            return
        self._unchecked = None
        self._torch.cuda.current_stream(self._dev).synchronize()
        st = self._status_np
        while max(int(st[1]), int(st[3])) > self._pair_cap:
            need, cap = ctypes.c_int64(), ctypes.c_int64()
            rc = self._L.crb_status(self._handle, ctypes.byref(need), ctypes.byref(cap), self._stream())   # report + reset
            if rc != _lib.CRB_ERR_OVERFLOW:
                check(rc)
                break
            self._ensure_workspace(u[4], self._ws_views, int(need.value * 1.25) + 1024)
            self._prefetched.clear()      # (downloads queued behind the skipped frame fetched nothing new)
            self._queue_render(*u)
            self._torch.cuda.current_stream(self._dev).synchronize()

    def _get(self, name, bit):
        t = self._mirror(name)
        self._materialize_clear()
        type(self)._fetched_by_current.add(name)
        if self._fetched is not None:
            self._fetched.add(name)
        if self._stale[name] and name in self._prefetched:
            # the download was queued right behind the render: wait for it (and, first read of the frame, for its status words)
            self._prefetched.discard(name)
            cap = self._pair_cap
            if self._unchecked is not None:
                self._validate()
            else:
                self._torch.cuda.current_stream(self._dev).synchronize()
            if self._pair_cap == cap:
                self._stale[name] = False
        if self._stale[name]:
            args = {"z": None, "color": None, "normals": None}
            args[name] = t.data_ptr()
            for attempt in range(2):
                check(self._L.crb_download(self._handle, bit, args["z"], args["color"], args["normals"], self._stream()))
                if self._unchecked is None:
                    self._torch.cuda.current_stream(self._dev).synchronize()
                    break
                # first read after a render: one synchronisation serves the download and the frame's status words; only a
                # frame that had to be drawn again is fetched twice
                cap = self._pair_cap
                self._validate()
                if self._pair_cap == cap:
                    break
            self._stale[name] = False
        self._exposed.add(name)
        return self._host_np[name]

    # ---------------------------------------------------------------------------------------- reference API
    def get_size(self):
        """pyx:80-81"""
        return self.h, self.w

    def render_model(self, model, prefetch=True):
        """pyx:92-104.  Reads model._vertices_by_triangles / _colors_by_triangles / _normals_by_triangles
        ([T,3,3] float32), never mutates them, composites into the persistent buffers.  (`prefetch=False`, not in the
        reference: do not start downloading the buffers the previous frame's caller fetched -- renderer.Renderer lights the
        colour buffer on the device first.)"""
        if self._texturing == "pixel":
            return self._render_model_textured(model, prefetch)
        v = _check_tri_array(getattr(model, "_vertices_by_triangles"), "vertices")
        c = _check_tri_array(getattr(model, "_colors_by_triangles"), "colors")
        n = _check_tri_array(getattr(model, "_normals_by_triangles"), "normals")
        if not (v.shape[0] == c.shape[0] == n.shape[0]):
            raise IndexError("Out of bounds on buffer access (axis 0)")   # what the bounds-checked memoryviews raise
        self.render_arrays(v, c, n, prefetch=prefetch)

    def _render_model_textured(self, model, prefetch):
        """render_model with texturing="pixel": vertices and normals by triangle as upstream, and -- in place of the colours --
        the texture coordinates by triangle, gathered on the device, with the model's texture bound.  Both are made once per
        model (cached on the identity of `_texture_coords`, `_triangles_texture_coords` and `_texture`, which Model never
        changes), so a render loop over one model uploads neither again."""
        torch = self._torch
        v = _check_tri_array(getattr(model, "_vertices_by_triangles"), "vertices")
        n = _check_tri_array(getattr(model, "_normals_by_triangles"), "normals")
        tex = getattr(model, "_texture", None)
        vt = getattr(model, "_texture_coords", None)
        tri = getattr(model, "_triangles_texture_coords", None)
        if tex is None or vt is None or tri is None:
            raise ValueError('texturing="pixel" needs a textured model (_texture, _texture_coords and _triangles_texture_coords); '
                             'this one has none')
        u = self._uv
        if u is None or u[0] is not vt or u[1] is not tri:
            from .model import _wrap_indices
            a = np.asarray(vt, dtype=np.float32)
            if a.ndim != 2 or a.shape[1] < 2:
                raise ValueError(f"texture coordinates must be [n,2] or [n,3], got {tuple(a.shape)}")
            idx = _wrap_indices(tri, a.shape[0])
            if idx.size == 0:
                idx = idx.reshape(0, 3)
            if idx.ndim != 2 or idx.shape[1] != 3:
                raise ValueError(f"texture coordinate indices must be [T,3], got {tuple(idx.shape)}")
            with torch.cuda.device(self._dev):
                d_vt = torch.from_numpy(np.ascontiguousarray(a[:, :2])).to(self._dev)
                d_vt = torch.nn.functional.pad(d_vt, (0, 1)).contiguous()       # [n,2] -> [n,3]: (u, v, 0)
                d_idx = torch.from_numpy(idx).to(self._dev)
                uv = torch.empty((idx.shape[0], 3, 3), dtype=torch.float32, device=self._dev)
                check(self._L.crb_model_gather(d_vt.data_ptr(), d_idx.data_ptr(), idx.shape[0], uv.data_ptr(), self._stream()))
            self._uv = u = (vt, tri, uv)
        if not (v.shape[0] == u[2].shape[0] == n.shape[0]):
            raise IndexError("Out of bounds on buffer access (axis 0)")
        self.render_arrays(v, u[2], n, prefetch=prefetch, texture=tex)

    def _bind_texture(self, texture):
        """Packs (crb_pack_texture) and binds (crb_bind_texture) `texture` -- with texture_filter="trilinear" its mip chain
        (crb_pack_texture_mips, crb_bind_texture_mips) -- unless it is what is bound already: the same NumPy array object, or the
        same torch tensor unchanged since (its version counter)."""
        torch = self._torch
        texture = _check_texture(texture)
        version = texture._version if isinstance(texture, torch.Tensor) else None
        t = self._tex
        if t is not None and t[0] is texture and t[1] == version:
            return
        self._validate()       # the previous frame may have to be drawn again, with the texture it was drawn with
        check(self._L.crb_join(self._handle, self._stream()))      # work in flight on the filler's streams reads the old one
        th, tw = int(texture.shape[0]), int(texture.shape[1])
        with torch.cuda.device(self._dev):
            if isinstance(texture, torch.Tensor):
                d_bgr = texture.to(self._dev).contiguous()
            else:
                d_bgr = torch.from_numpy(np.ascontiguousarray(texture)).to(self._dev)
            if self._tex_flags & _lib.CRB_TEX_TRILINEAR:
                texels = ctypes.c_int64()
                check(self._L.crb_mip_layout(th, tw, None, ctypes.byref(texels)))
                packed = torch.empty((texels.value,), dtype=torch.int32, device=self._dev)
                check(self._L.crb_pack_texture_mips(d_bgr.data_ptr(), th, tw, packed.data_ptr(), self._stream()))
            else:
                packed = torch.empty((th, tw), dtype=torch.int32, device=self._dev)
                check(self._L.crb_pack_texture(d_bgr.data_ptr(), th, tw, packed.data_ptr(), self._stream()))
        bind = self._L.crb_bind_texture_mips if self._tex_flags & _lib.CRB_TEX_TRILINEAR else self._L.crb_bind_texture
        check(bind(self._handle, packed.data_ptr(), th, tw))
        self._tex = (texture, version, packed)

    def _uv_array(self, c, on_device):
        """Texture coordinates by triangle, [T,3,3] (third component ignored) or [T,3,2] float32 -> [T,3,3]."""
        torch = self._torch
        if isinstance(c, torch.Tensor):
            if c.dtype != torch.float32 or c.dim() != 3 or tuple(c.shape[1:]) not in ((3, 3), (3, 2)):
                raise ValueError("texture coordinates must be float32 [T,3,3] or [T,3,2]")
            if c.shape[2] == 2:
                c = torch.nn.functional.pad(c, (0, 1))
            return c.to(self._dev).contiguous() if on_device else c.cpu().numpy()
        c = np.asarray(c)
        if c.dtype != np.float32 or c.ndim != 3 or c.shape[1:] not in ((3, 3), (3, 2)):
            raise ValueError("texture coordinates must be float32 [T,3,3] or [T,3,2]")
        if c.shape[2] == 2:
            c = np.concatenate([c, np.zeros(c.shape[:2] + (1,), np.float32)], axis=2)
        return torch.from_numpy(np.ascontiguousarray(c)).to(self._dev) if on_device else c

    def get_normals_buffer(self):
        """pyx:246-247 -- live float32 [h,w,3] view (same array object on every call)."""
        return self._get("normals", _lib.CRB_BUF_NORMALS)

    def get_color_buffer(self):
        """pyx:249-250"""
        return self._get("color", _lib.CRB_BUF_COLOR)

    def get_z_buffer(self):
        """pyx:252-253"""
        return self._get("z", _lib.CRB_BUF_Z)

    # ---------------------------------------------------------------------------------------- extensions
    def clear(self):
        """Fresh-filler state (pyx:65-67).  The reference has no reset (a new filler per frame is its idiom,
        run.py:21); here the clear is fused into the next frame's tile pass instead of a separate memset."""
        self._pending_clear = True
        self._prefetched.clear()
        self._unchecked = None    # whatever the last frame was, nothing of it remains
        for name in self._stale:
            self._stale[name] = True
        self._exposed.clear()   # arrays handed out earlier are detached until fetched again

    def render_arrays(self, v, c, n, path="tiled", check_status=True, prefetch=True, texture=None):
        """Render [T,3,3] float32 arrays.  numpy inputs are staged through pinned memory and copied H2D;
        torch CUDA tensors are used in place (device-resident inputs).  `texture` (uint8 [h,w,3], BGR; NumPy or torch):
        per-pixel texturing -- `c` then holds texture coordinates by triangle, [T,3,3] (third component ignored) or
        [T,3,2], and every pixel takes the texel they name (CRB_TEXTURE), sampled as the constructor's `texture_filter` and
        `perspective_correct` say."""
        torch = self._torch
        flags = _lib.CRB_PATH_ATOMIC if path == "atomic" else 0
        if texture is not None:
            texture = _check_texture(texture)
            # one residence for all three: on the device if any of them is a CUDA tensor
            on_device = any(isinstance(a, torch.Tensor) and a.is_cuda for a in (v, c, n))
            c = self._uv_array(c, on_device)
            if on_device:
                v, n = (a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a)).to(self._dev) for a in (v, n))
            flags |= self._tex_flags
        on_device = all(isinstance(a, torch.Tensor) for a in (v, c, n))
        if on_device:
            for a in (v, c, n):
                if a.dtype != torch.float32 or a.dim() != 3 or tuple(a.shape[1:]) != (3, 3) or not a.is_cuda:
                    raise ValueError("device inputs must be CUDA float32 tensors of shape [T,3,3]")
            v, c, n = v.contiguous(), c.contiguous(), n.contiguous()
            T = v.shape[0]
        else:
            # (a vertex with camera z == 0: the reference build trips Cython's division check inside a nogil block, prints an
            # unraisable ZeroDivisionError, abandons the projection loop and rasterizes half-projected garbage, pyx:122; here
            # that vertex simply gets IEEE inf / NaN coordinates like on the device-resident path -- stated divergence, DESIGN 2)
            v, c, n = (np.asarray(a) for a in (v, c, n))
            T = v.shape[0]
        self._validate()                 # an earlier frame this one composites onto must have been drawn
        if texture is not None:
            self._bind_texture(texture)
        if self._pending_clear:
            flags |= _lib.CRB_CLEAR_FIRST
        else:
            self._push_exposed()
        self._ensure_workspace(T)
        if not on_device and T * 36 >= self.PAGEABLE_MIN_BYTES:
            # large host arrays: the library stages them itself, chunk by chunk through its pinned ring with worker threads
            # (CRB_HOST_PAGEABLE) -- a single-threaded NumPy copy into pinned memory was 75 ms of the 10 M-triangle frame
            v, c, n = (np.ascontiguousarray(a) for a in (v, c, n))
            flags |= _lib.CRB_HOST_PAGEABLE
        elif not on_device and T > 0 and all(a.flags.c_contiguous and a.dtype == np.float32 for a in (v, c, n)) and \
                all([_HostArrays.pinned(self._L, a) for a in (v, c, n)]):
            # the caller's own arrays, page-locked in place by an earlier frame: the GPU reads them directly, and the call
            # returns once they have been read (CRB_SYNC_UPLOAD) -- the caller may change them afterwards, as upstream
            flags |= _lib.CRB_SYNC_UPLOAD
        elif not on_device:
            if self._stage is None or self._stage.shape[1] < T:
                self._stage = torch.empty((3, max(T, 1), 3, 3), dtype=torch.float32, pin_memory=True)
                self._stage_np = self._stage.numpy()
            s = self._stage_np
            s[0, :T] = v
            s[1, :T] = c
            s[2, :T] = n
            v = c = n = None
        args = (on_device, v, c, n, T, flags)
        self._queue_render(*args)
        self._prefetched.clear()
        want = self._fetched if self._fetched is not None else type(self)._fetched_by_previous
        self._fetched = set()
        if check_status and prefetch and self.row0 == 0 and self.row1 == self.h:
            for name, bit in (("color", _lib.CRB_BUF_COLOR), ("normals", _lib.CRB_BUF_NORMALS), ("z", _lib.CRB_BUF_Z)):
                if name in want and name not in self._exposed:
                    dst = {"z": None, "color": None, "normals": None}
                    dst[name] = self._mirror(name).data_ptr()
                    check(self._L.crb_download(self._handle, bit, dst["z"], dst["color"], dst["normals"], self._stream()))
                    self._prefetched.add(name)
        if check_status:
            self._unchecked = args       # (device inputs stay referenced until the frame is known to have been drawn)
            if flags & (_lib.CRB_HOST_PAGEABLE | _lib.CRB_SYNC_UPLOAD):
                # the frame was read from the caller's own arrays: should it have to be drawn again (pair list overflow), that
                # must happen before the caller gets a chance to change them
                self._validate()
        elif not on_device:
            torch.cuda.current_stream(self._dev).synchronize()     # the pinned staging is reused by the next call
        self._pending_clear = False
        for name in self._stale:
            self._stale[name] = True
        # arrays already handed out are live views upstream: keep them current
        for name, bit in (("z", _lib.CRB_BUF_Z), ("color", _lib.CRB_BUF_COLOR), ("normals", _lib.CRB_BUF_NORMALS)):
            if name in self._exposed:
                self._get(name, bit)

    def _queue_render(self, on_device, v, c, n, T, flags):
        """Queues one frame (upload of the staged host arrays if any, kernels, status words) on the current stream."""
        if on_device:
            check(self._L.crb_render(self._handle, v.data_ptr(), c.data_ptr(), n.data_ptr(), T, flags, self._stream()))
        elif flags & (_lib.CRB_HOST_PAGEABLE | _lib.CRB_SYNC_UPLOAD):
            check(self._L.crb_render_host(self._handle, v.ctypes.data, c.ctypes.data, n.ctypes.data, T,
                                          flags | _lib.CRB_NO_SYNC, 0, None, None, None, self._stream()))
        else:
            st = self._stage
            check(self._L.crb_render_host(self._handle, st[0].data_ptr(), st[1].data_ptr(), st[2].data_ptr(), T,
                                          flags | _lib.CRB_NO_SYNC, 0, None, None, None, self._stream()))
        if self._status is None:
            self._status = self._torch.zeros(4, dtype=self._torch.int64, pin_memory=True)
            self._status_np = self._status.numpy()
        check(self._L.crb_status_async(self._handle, self._status.data_ptr(), self._stream()))

    def set_option(self, option, value):
        """crb_set_option: tuning switches (_lib.CRB_OPT_*), e.g. the store path of the fused clear or a fixed k_raster grid."""
        check(self._L.crb_set_option(self._handle, int(option), int(value)))

    def device_buffers(self):
        """(z, color, normals) torch CUDA tensors -- the device-resident truth (no copy)."""
        self._validate()
        self._materialize_clear()
        self._push_exposed()
        self._prefetched.clear()         # the caller may change the device buffers: what get_*_buffer() returns is read afterwards
        return self._z, self._color, self._normals

    def illuminate_guro(self, light_direction):
        """GuroIllumination.draw_illumination on the device buffers, in place (guro_illumination.py:20-27)."""
        self._validate()
        self._materialize_clear()
        self._push_exposed()
        arr = (ctypes.c_float * 3)(*[float(x) for x in light_direction])
        check(self._L.crb_guro(self._handle, arr, self._stream()))
        self._stale["color"] = True
        self._prefetched.discard("color")

    def color_u8_flipped(self):
        """run.py:26 `image[::-1].astype('uint8')` computed on device; returns a torch CUDA uint8 tensor."""
        self._validate()
        self._materialize_clear()
        self._push_exposed()
        out = self._torch.empty((self.row1 - self.row0, self.w, 3), dtype=self._torch.uint8, device=self._dev)
        check(self._L.crb_color_u8_flipped(self._handle, out.data_ptr(), self._stream()))
        return out

    def render_views(self, v, c, n, views, z_out=None, color_out=None, normals_out=None, color_u8_out=None,
                     want=("z", "color", "normals"), guro_light=None, chunk=32, check_status=True, defer_join=False,
                     u8_exchange=None, texture=None):
        """Batched multi-view render (config C5): every view gets fresh-filler buffers in its own slab.

        v, c, n: torch CUDA float32 [T,3,3] (device-resident base mesh);  views: [V,16] float32 (numpy or CUDA tensor,
        see views.py).  Outputs are torch CUDA tensors [V,rows,w(,3)], allocated here unless passed in; `want` selects
        which float32 buffers are produced, `color_u8_out=True` (or a tensor) adds run.py:26's flipped uint8 image.
        `guro_light` = raw light direction (as given to GuroIllumination) fuses the illumination into the shading pass.
        `defer_join=True` (with check_status=False): the call returns without ordering the current stream behind the
        rasterizer, so the next batch's front end overlaps it; call `join()` before using the outputs.
        `u8_exchange=(rows_per_band, [address, ...])` (sharding.RowExchange.plan): the flipped uint8 images leave the
        rasterizer row band by row band straight into the listed receive buffers (other GPUs' memory) instead of a
        local array -- the view-sharded render and its delivery in one kernel (crb_set_u8_exchange).
        `texture` (uint8 [h,w,3], BGR): per-pixel texturing -- `c` holds texture coordinates by triangle, [T,3,3] or
        [T,3,2], host or CUDA (see render_arrays).
        Returns a dict of the produced tensors."""
        torch = self._torch
        if texture is not None:
            texture = _check_texture(texture)
            c = self._uv_array(c, True)
        for a in (v, c, n):
            if not isinstance(a, torch.Tensor) or not a.is_cuda or a.dtype != torch.float32 or tuple(a.shape[1:]) != (3, 3):
                raise ValueError("render_views needs CUDA float32 tensors of shape [T,3,3]")
        v, c, n = v.contiguous(), c.contiguous(), n.contiguous()
        T = v.shape[0]
        if not isinstance(views, torch.Tensor):
            views = torch.from_numpy(np.ascontiguousarray(views, dtype=np.float32)).to(self._dev)
        views = views.contiguous()
        V = views.shape[0]
        rows = self.row1 - self.row0
        out = {}

        def slab(name, given, shape, dtype):
            if given is None and name not in want:
                return None
            t = given if isinstance(given, torch.Tensor) else torch.empty(shape, dtype=dtype, device=self._dev)
            assert t.is_cuda and t.is_contiguous() and tuple(t.shape) == shape and t.dtype == dtype
            out[name] = t
            return t

        z_out = slab("z", z_out, (V, rows, self.w), torch.float32)
        color_out = slab("color", color_out, (V, rows, self.w, 3), torch.float32)
        normals_out = slab("normals", normals_out, (V, rows, self.w, 3), torch.float32)
        if color_u8_out is True:
            color_u8_out = torch.empty((V, rows, self.w, 3), dtype=torch.uint8, device=self._dev)
        if color_u8_out is not None:
            out["color_u8"] = color_u8_out
        flags, light = 0, None
        if texture is not None:
            self._bind_texture(texture)
            flags |= self._tex_flags
        if guro_light is not None:
            # GuroIllumination.__init__ (guro_illumination.py:17-18): negate, then normalise, in float32
            l = -np.asarray(guro_light, dtype="float32")
            l = l / np.linalg.norm(l)
            light = (ctypes.c_float * 3)(*[float(x) for x in l])
            flags |= _lib.CRB_GURO
        if defer_join and not check_status:
            flags |= _lib.CRB_DEFER_JOIN
            # the front end may still be queued on the filler's internal stream when this call returns: torch's allocator orders
            # the reuse of freed memory on the CALLER's stream only, so temporaries made above stay referenced until join()
            self._deferred_keep = (views, v, c, n)
        self._ensure_workspace(T, views=min(int(chunk), max(V, 1)))
        ptr = lambda t: None if t is None else t.data_ptr()
        if u8_exchange is not None:
            if color_u8_out is not None:
                raise ValueError("u8_exchange replaces color_u8_out")
            hb, bases = u8_exchange
            arr = (ctypes.c_void_p * len(bases))(*[int(b) for b in bases])
            check(self._L.crb_set_u8_exchange(self._handle, len(bases), int(hb), arr))
        try:
            return self._render_views_loop(v, c, n, T, views, V, z_out, color_out, normals_out, color_u8_out, flags, light,
                                           check_status, out, ptr)
        finally:
            if u8_exchange is not None:
                check(self._L.crb_set_u8_exchange(self._handle, 0, 0, None))

    def _render_views_loop(self, v, c, n, T, views, V, z_out, color_out, normals_out, color_u8_out, flags, light, check_status,
                           out, ptr):
        while True:
            check(self._L.crb_render_views(self._handle, v.data_ptr(), c.data_ptr(), n.data_ptr(), T, views.data_ptr(), V,
                                           ptr(z_out), ptr(color_out), ptr(normals_out), ptr(color_u8_out), flags, light,
                                           self._stream()))
            if not check_status:
                break
            need, cap = ctypes.c_int64(), ctypes.c_int64()
            rc = self._L.crb_status(self._handle, ctypes.byref(need), ctypes.byref(cap), self._stream())
            if rc == _lib.CRB_ERR_OVERFLOW:
                self._ensure_workspace(T, self._ws_views, int(need.value * 1.25) + 1024)
                continue
            check(rc)
            break
        return out

    def join(self):
        """Orders the current stream behind batches issued with defer_join=True."""
        check(self._L.crb_join(self._handle, self._stream()))
        self._deferred_keep = None

    def transform_view(self, v, n, view):
        """The camera-space [T,3,3] arrays one view produces (what the reference would be handed for that view)."""
        torch = self._torch
        if not isinstance(view, torch.Tensor):
            view = torch.from_numpy(np.ascontiguousarray(view, dtype=np.float32).ravel()).to(self._dev)
        vo, no = torch.empty_like(v), torch.empty_like(n)
        check(self._L.crb_transform_view(self._handle, v.data_ptr(), n.data_ptr(), v.shape[0], view.data_ptr(),
                                         vo.data_ptr(), no.data_ptr(), self._stream()))
        return vo, no

    def profile(self, enable=True):
        check(self._L.crb_profile(self._handle, int(bool(enable))))

    def profile_read(self):
        """(launches, total_ms) of the tile rasterizer kernel since the last read (CUDA events on the render stream)."""
        n, ms = ctypes.c_int(), ctypes.c_double()
        check(self._L.crb_profile_read(self._handle, ctypes.byref(n), ctypes.byref(ms)))
        return n.value, ms.value

    @property
    def launch_count(self):
        return int(self._L.crb_launch_count(self._handle))
