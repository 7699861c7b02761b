"""Frame pipelining for host-resident callers.

One `render_model` through the host-buffer C-ABI call (crb_render_host) is H2D of the three [T,3,3] arrays, the
render, and D2H of the requested buffers -- at 1024^2 the D2H of z + colour + normals (29.4 MB) is ~90 % of the wall
time and the GPU idles meanwhile.  `HostFramePipeline` keeps `depth` fillers (each with its own CUDA stream, device
buffers, workspace and pinned host outputs) and submits frames round-robin with CRB_NO_SYNC, so frame k+1's upload
and render overlap frame k's download; every frame still gets fresh-filler semantics (pyx:65-67) and the same bits.

The reference has no equivalent (a new filler per frame, synchronous, run.py:21-25); this is the throughput-oriented
way to drive the same path from host memory.
"""
import ctypes

import numpy as np

from . import _lib
from ._lib import check
from .pixel_buffer_filler import SS_FLAGS, AdvancedPixelBufferFiller, _check_supersample, _check_tri_array

_BITS = {"z": _lib.CRB_BUF_Z, "color": _lib.CRB_BUF_COLOR, "normals": _lib.CRB_BUF_NORMALS}


class _Slot:
    pass


class HostFramePipeline:
    def __init__(self, h, w, fov=90.0, z_near=0.1, z_far=1000.0, depth=2, device=None, want=("z", "color", "normals"),
                 sparse=True, near_clip=False):
        """sparse=True: CRB_DL_SPARSE read-back -- each slot's pinned host arrays persist between its frames, so only the
        tiles that are busy in the new frame or were busy in the frame the arrays still show are copied (by a kernel that
        writes into the mapped host memory); the arrays are bit-identical to a full download but READ-ONLY for the caller.
        sparse=False: plain cudaMemcpy of the whole buffers every frame.  near_clip=True: triangles are clipped at z_near
        (CRB_CLIP_NEAR, see AdvancedPixelBufferFiller)."""
        if depth < 1:
            raise ValueError("depth must be >= 1")
        self.sparse = bool(sparse)
        self.want = tuple(want)
        self.mask = 0
        for name in self.want:
            self.mask |= _BITS[name]
        self.slots = []
        for _ in range(depth):
            s = _Slot()
            s.filler = AdvancedPixelBufferFiller(h, w, fov=fov, z_near=z_near, z_far=z_far, device=device, near_clip=near_clip)
            torch = s.filler._torch
            s.stream = torch.cuda.Stream(device=s.filler._dev)
            s.out = {name: s.filler._mirror(name) for name in self.want}      # pinned host tensors
            s.out_np = {name: s.filler._host_np[name] for name in self.want}
            if self.sparse:          # the state CRB_DL_SPARSE assumes before the first frame: fresh-filler values (pyx:65-67)
                for name, arr in s.out_np.items():
                    arr[...] = 1e6 if name == "z" else 0.0
                s.out_np = {name: arr.view() for name, arr in s.out_np.items()}
                for arr in s.out_np.values():
                    arr.flags.writeable = False
            s.stage = None
            s.busy = False
            self.slots.append(s)
        self._torch = torch
        self._next = 0
        self._L = self.slots[0].filler._L

    def _ptr(self, s, name):
        return s.out[name].data_ptr() if name in s.out else None

    def submit(self, v, c, n):
        """Queues one fresh-filler frame; returns the slot index to pass to `result`.  v, c, n: [T,3,3] float32, either
        pinned torch CPU tensors (used in place -- do not modify them before `result`) or NumPy arrays (copied into
        the slot's pinned staging first)."""
        torch = self._torch
        i = self._next
        self._next = (i + 1) % len(self.slots)
        s = self.slots[i]
        if s.busy:       # its host buffers are about to be reused
            self.result(i)
        if all(isinstance(a, torch.Tensor) for a in (v, c, n)):
            for a in (v, c, n):
                if a.is_cuda or a.dtype != torch.float32 or a.dim() != 3 or tuple(a.shape[1:]) != (3, 3) or not a.is_contiguous():
                    raise ValueError("tensor inputs must be contiguous CPU float32 [T,3,3]")
            T = int(v.shape[0])
            pv, pc, pn = v.data_ptr(), c.data_ptr(), n.data_ptr()
        else:
            v = _check_tri_array(v, "vertices"); c = _check_tri_array(c, "colors"); n = _check_tri_array(n, "normals")
            T = int(v.shape[0])
            if s.stage is None or s.stage.shape[1] < T:
                s.stage = torch.empty((3, max(T, 1), 3, 3), dtype=torch.float32, pin_memory=True)
                s.stage_np = s.stage.numpy()
            s.stage_np[0, :T] = v; s.stage_np[1, :T] = c; s.stage_np[2, :T] = n
            pv, pc, pn = s.stage[0].data_ptr(), s.stage[1].data_ptr(), s.stage[2].data_ptr()
        s.filler._ensure_workspace(T)
        s.args = (pv, pc, pn, T)
        s.keep = (v, c, n)
        self._launch(s)
        s.busy = True
        return i

    def _launch(self, s):
        pv, pc, pn, T = s.args
        check(self._L.crb_render_host(s.filler._handle, pv, pc, pn, T, _lib.CRB_CLEAR_FIRST | _lib.CRB_NO_SYNC | (_lib.CRB_DL_SPARSE if self.sparse else 0) |
                                      s.filler._clip_flags, self.mask,
                                      self._ptr(s, "z"), self._ptr(s, "color"), self._ptr(s, "normals"),
                                      ctypes.c_void_p(s.stream.cuda_stream)))

    def result(self, i):
        """Waits for slot i's frame; returns {name: numpy array} (pinned memory, valid until the slot is resubmitted)."""
        s = self.slots[i]
        while s.busy:
            need, cap = ctypes.c_int64(), ctypes.c_int64()
            st = ctypes.c_void_p(s.stream.cuda_stream)
            rc = self._L.crb_status(s.filler._handle, ctypes.byref(need), ctypes.byref(cap), st)   # synchronises the stream
            if rc == _lib.CRB_ERR_OVERFLOW:     # the frame was skipped: enlarge the pair list and queue it again
                f = s.filler
                f._ensure_workspace(s.args[3], f._ws_views, int(need.value * 1.25) + 1024)
                self._launch(s)
                continue
            check(rc)
            s.busy = False
            s.keep = None
        return s.out_np

    def drain(self):
        for i in range(len(self.slots)):
            self.result(i)

    def readback_tiles(self, reset=True):
        """Tiles (32x32 pixels) copied to the host by the sparse read-back since the last reset, over all slots."""
        total = 0
        for s in self.slots:
            n = ctypes.c_int64()
            check(self._L.crb_readback_stats(s.filler._handle, ctypes.byref(n), int(reset), ctypes.c_void_p(s.stream.cuda_stream)))
            total += n.value
        return total

    @property
    def launch_count(self):
        return sum(s.filler.launch_count for s in self.slots)


class HostImagePipeline:
    """run.py's product -- the uint8 image `image[::-1].astype('uint8')` (run.py:26), optionally lit by GuroIllumination
    (renderer.py:48) -- from host triangle arrays to host memory, with only 3 bytes per pixel crossing PCIe (SURVEY 8f N3).

    Per frame, on the slot's own stream, ONE C-ABI call (crb_render_image_host): one H2D copy of the [3,T,3,3] block, one
    fused launch sequence (fresh-filler clear + rasterizer + shading with the light applied + truncation to uint8 + row
    flip, written by the rasterizer itself: no float32 buffer is produced at all), one D2H copy of h*w*3 bytes and of the
    status words.  `depth` frames are in flight.  Inputs: a pinned float32 tensor [3,T,3,3] = (vertices, colours, normals)
    by triangles, not to be modified before `result`.  `supersample=2 | 4`: the image is anti-aliased -- its fillers render
    (s*h, s*w) samples and the rasterizer resolves each s x s block into one pixel of the [h,w,3] image (CRB_SS2 / CRB_SS4).
    `near_clip=True`: triangles are clipped at z_near (CRB_CLIP_NEAR, see AdvancedPixelBufferFiller).
    (The per-frame host work matters: at 10 k images/s the submitting thread is the bottleneck if a frame costs it more than
    a few dozen microseconds.)"""

    def __init__(self, h, w, fov=90.0, z_near=0.1, z_far=1000.0, depth=3, device=None, light=None, supersample=1,
                 near_clip=False):
        if depth < 1:
            raise ValueError("depth must be >= 1")
        ss = _check_supersample(supersample)
        self._flags, self._light = SS_FLAGS[ss], None
        if light is not None:
            # GuroIllumination.__init__ (guro_illumination.py:17-18): negate, then normalise, in float32
            l = -np.asarray(light, dtype="float32")
            l = l / np.linalg.norm(l)
            self._light = (ctypes.c_float * 3)(*[float(x) for x in l])
            self._flags |= _lib.CRB_GURO
        self.slots = []
        for _ in range(depth):
            s = _Slot()
            s.filler = AdvancedPixelBufferFiller(ss * h, ss * w, fov=fov, z_near=z_near, z_far=z_far, device=device,
                                                 near_clip=near_clip)
            torch = s.filler._torch
            dev = s.filler._dev
            s.stream = torch.cuda.Stream(device=dev)
            s.stream_ptr = ctypes.c_void_p(s.stream.cuda_stream)
            s.dev_u8 = torch.empty((h, w, 3), dtype=torch.uint8, device=dev)
            s.host_u8 = torch.empty((h, w, 3), dtype=torch.uint8, pin_memory=True)
            s.host_np = s.host_u8.numpy()
            s.status = torch.zeros(4, dtype=torch.int64, pin_memory=True)
            s.status_np = s.status.numpy()
            s.dev_u8_ptr, s.host_u8_ptr, s.status_ptr = s.dev_u8.data_ptr(), s.host_u8.data_ptr(), s.status.data_ptr()
            s.done = torch.cuda.Event()
            s.busy = False
            self.slots.append(s)
        self._flags |= self.slots[0].filler._clip_flags
        self._torch = torch
        self._L = self.slots[0].filler._L
        self._next = 0

    def submit(self, block):
        torch = self._torch
        if not isinstance(block, torch.Tensor) or block.is_cuda or block.dtype != torch.float32 or block.dim() != 4 or \
                tuple(block.shape[0:1] + block.shape[2:]) != (3, 3, 3) or not block.is_contiguous():
            raise ValueError("input must be a contiguous CPU float32 tensor [3,T,3,3] (pinned for asynchronous copies)")
        i = self._next
        self._next = (i + 1) % len(self.slots)
        s = self.slots[i]
        if s.busy:
            self.result(i)
        T = int(block.shape[1])
        if s.filler._frame_triangles(T) > s.filler._ws_T or s.filler._ws is None:
            with torch.cuda.stream(s.stream):
                s.filler._ensure_workspace(T, views=1)
        s.T = T
        s.keep = block
        base = block.data_ptr()
        s.args = (base, base + 36 * T, base + 72 * T)
        self._launch(s)
        s.busy = True
        return i

    def _launch(self, s):
        # one C call: upload, fused clear + raster + shade (+ light) + uint8 + flip, download of the image and the status words
        check(self._L.crb_render_image_host(s.filler._handle, s.args[0], s.args[1], s.args[2], s.T, self._flags | _lib.CRB_NO_SYNC,
                                            self._light, s.dev_u8_ptr, s.host_u8_ptr, s.status_ptr, s.stream_ptr))
        s.done.record(s.stream)

    def result(self, i):
        """Waits for slot i's frame; returns the uint8 [h,w,3] image (pinned memory, valid until the slot is resubmitted)."""
        s = self.slots[i]
        while s.busy:
            s.done.synchronize()
            f = s.filler
            if max(int(s.status_np[1]), int(s.status_np[3])) > f._pair_cap:
                # the frame was skipped (pair list too small): take the report, enlarge the list and draw it again
                need, cap = ctypes.c_int64(), ctypes.c_int64()
                rc = self._L.crb_status(f._handle, ctypes.byref(need), ctypes.byref(cap), s.stream_ptr)
                if rc != _lib.CRB_ERR_OVERFLOW:
                    check(rc)
                with self._torch.cuda.stream(s.stream):
                    f._ensure_workspace(s.T, f._ws_views, int(max(need.value, s.status_np[1], s.status_np[3]) * 1.25) + 1024)
                self._launch(s)
                continue
            s.busy = False
            s.keep = None
        return s.host_np

    def drain(self):
        for i in range(len(self.slots)):
            self.result(i)

    @property
    def launch_count(self):
        return sum(s.filler.launch_count for s in self.slots)
