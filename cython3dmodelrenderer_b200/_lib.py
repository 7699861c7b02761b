"""ctypes binding of libcrender_b200.so (C ABI: include/crender_b200.h).

There is no CPU fallback: if the shared library has not been built, or no CUDA device is visible,
the product raises.  Build with `python -c "import __graft_entry__ as g; g.build()"` or
`make -C cython3dmodelrenderer_b200/csrc`.
"""
import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.path.join(CSRC, "libcrender_b200.so")
HEADER = os.path.join(os.path.dirname(_HERE), "include", "crender_b200.h")
HEADERS = [HEADER, os.path.join(os.path.dirname(_HERE), "include", "crender_ingest_b200.h")]
SOURCES = [os.path.join(CSRC, "crender_b200.cu"), os.path.join(CSRC, "ingest_b200.cu")]

CRB_OK = 0
CRB_ERR_INVALID, CRB_ERR_CUDA, CRB_ERR_ZERODIV, CRB_ERR_STATE, CRB_ERR_OVERFLOW = -1, -2, -3, -4, -5
CRB_ERR_SYNTAX, CRB_ERR_RANGE = -6, -7
CRB_CLEAR_FIRST, CRB_PATH_ATOMIC, CRB_GURO, CRB_NO_SYNC, CRB_DL_SPARSE, CRB_DEFER_JOIN, CRB_HOST_PAGEABLE, CRB_SYNC_UPLOAD = 1, 2, 4, 8, 16, 32, 64, 128
CRB_TEXTURE, CRB_TEX_PERSPECTIVE, CRB_TEX_BILINEAR, CRB_TEX_TRILINEAR = 1024, 2048, 4096, 8192
CRB_OPT_CHUNK_PIPELINE, CRB_OPT_TMA, CRB_OPT_TMA_ROWS, CRB_OPT_BAND_PREPASS, CRB_OPT_RASTER_CTAS, CRB_OPT_SPLIT_HEAVY, CRB_OPT_WIDE_KERNEL = 1, 2, 3, 4, 5, 6, 7
CRB_OPT_RASTER_SHAPE = 8
CRB_BUF_Z, CRB_BUF_COLOR, CRB_BUF_NORMALS, CRB_BUF_ALL = 1, 2, 4, 7

_vp, _i, _i64, _u, _f, _sz = (ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_uint, ctypes.c_float,
                              ctypes.c_size_t)
_ip, _i64p = ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int64)
_fp = ctypes.POINTER(ctypes.c_float)
_vpp = ctypes.POINTER(ctypes.c_void_p)

# name -> (restype, argtypes); every symbol include/crender_b200.h declares
SIGNATURES = {
    "crb_version": (_i, []),
    "crb_last_error": (ctypes.c_char_p, []),
    "crb_device_count": (_i, [_ip]),
    "crb_projection": (_i, [_i, _i, _f, _f, _f, _fp]),
    "crb_create": (_i, [_i, _i, _f, _f, _f, _i, _vpp]),
    "crb_destroy": (None, [_vp]),
    "crb_get_size": (_i, [_vp, _ip, _ip]),
    "crb_get_projection": (_i, [_vp, _fp]),
    "crb_set_band": (_i, [_vp, _i, _i]),
    "crb_bind_buffers": (_i, [_vp, _vp, _vp, _vp]),
    "crb_workspace_bytes": (_sz, [_vp, _i64, _i, _i64]),
    "crb_bind_workspace": (_i, [_vp, _vp, _sz, _i64, _i, _i64, _vp]),
    "crb_alloc_owned": (_i, [_vp, _i64, _i, _i64]),
    "crb_device_buffers": (_i, [_vp, _vpp, _vpp, _vpp]),
    "crb_init_buffers": (_i, [_vp, _vp]),
    "crb_render": (_i, [_vp, _vp, _vp, _vp, _i64, _u, _vp]),
    "crb_render_host": (_i, [_vp, _vp, _vp, _vp, _i64, _u, _u, _vp, _vp, _vp, _vp]),
    "crb_render_views": (_i, [_vp, _vp, _vp, _vp, _i64, _vp, _i, _vp, _vp, _vp, _vp, _u, _fp, _vp]),
    "crb_set_option": (_i, [_vp, _i, _i]),
    "crb_join": (_i, [_vp, _vp]),
    "crb_set_u8_exchange": (_i, [_vp, _i, _i, ctypes.POINTER(_vp)]),
    "crb_sync": (_i, [_vp, _vp]),
    "crb_readback_stats": (_i, [_vp, _i64p, _i, _vp]),
    "crb_readback_reset": (_i, [_vp, _vp]),
    "crb_transform_view": (_i, [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp]),
    "crb_guro": (_i, [_vp, _fp, _vp]),
    "crb_color_u8_flipped": (_i, [_vp, _vp, _vp]),
    "crb_download": (_i, [_vp, _u, _vp, _vp, _vp, _vp]),
    "crb_upload": (_i, [_vp, _u, _vp, _vp, _vp, _vp]),
    "crb_status": (_i, [_vp, _i64p, _i64p, _vp]),
    "crb_pair_capacity": (_i64, [_vp]),
    "crb_launch_count": (_i64, [_vp]),
    "crb_selftest_fdiv": (_i, [_i, ctypes.c_uint64, _u, ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint32)]),
    "crb_phase_cycles": (_i, [ctypes.POINTER(ctypes.c_uint64), _i]),
    "crb_trace_dump": (_i, [ctypes.c_char_p]),
    "crb_status_async": (_i, [_vp, _vp, _vp]),
    "crb_render_image_host": (_i, [_vp, _vp, _vp, _vp, _i64, _u, _fp, _vp, _vp, _vp, _vp]),
    "crb_host_register": (_i, [_vp, _sz]),
    "crb_host_unregister": (_i, [_vp]),
    "crb_shared_alloc": (_i, [_i, _sz, ctypes.POINTER(_vp), ctypes.c_char_p]),
    "crb_shared_open": (_i, [_i, ctypes.c_char_p, ctypes.POINTER(_vp)]),
    "crb_shared_close": (_i, [_i, _vp]),
    "crb_shared_free": (_i, [_i, _vp]),
    "crb_profile": (_i, [_vp, _i]),
    "crb_profile_read": (_i, [_vp, _ip, ctypes.POINTER(ctypes.c_double)]),
    "crb_pack_texture": (_i, [_vp, _i, _i, _vp, _vp]),
    "crb_bind_texture": (_i, [_vp, _vp, _i, _i]),
    "crb_mip_layout": (_i, [_i, _i, _ip, _i64p]),
    "crb_pack_texture_mips": (_i, [_vp, _i, _i, _vp, _vp]),
    "crb_bind_texture_mips": (_i, [_vp, _vp, _i, _i]),
    # include/crender_ingest_b200.h (model ingest, SURVEY 8f N4)
    "crb_obj_parse": (_i, [ctypes.c_char_p, _sz, _vpp]),
    "crb_obj_free": (None, [_vp]),
    "crb_obj_counts": (_i, [_vp, _i64p]),
    "crb_obj_copy": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "crb_obj_mtllib": (_i, [_vp, _i, ctypes.POINTER(ctypes.c_char_p), ctypes.POINTER(_sz)]),
    "crb_model_normals_workspace_bytes": (_sz, [_i64, _i64]),
    "crb_model_vertex_normals": (_i, [_vp, _i64, _vp, _i64, _i, _vp, _vp, _sz, _vp]),
    "crb_model_vertex_colors": (_i, [_vp, _i64, _i, _vp, _i, _i, _vp, _vp]),
    "crb_model_gather": (_i, [_vp, _vp, _i64, _vp, _vp]),
    "crb_model_launch_count": (_i64, []),
}

_lib = None


class CrenderError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"libcrender_b200: {message} (code {code})")
        self.code = code


def build(force=False, verbose=False):
    """nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -fmad=false ... (cross-compiles without a GPU)."""
    stale = (not os.path.exists(LIB_PATH)
             or os.path.getmtime(LIB_PATH) < max(os.path.getmtime(p) for p in SOURCES + HEADERS))
    if force or stale:
        cmd = ["make", "-C", CSRC, "libcrender_b200.so"] + (["-B"] if force else [])
        subprocess.run(cmd, check=True, stdout=None if verbose else subprocess.DEVNULL)
    return LIB_PATH


def load_library():
    """Loads the shared library and installs the prototypes.  Raises if it is missing -- there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("CRB_LIB_OVERRIDE", LIB_PATH)   # experiments only: an alternative build of the same library
    if not os.path.exists(path):
        raise ImportError(
            f"{path} is missing: the CUDA library has not been built "
            "(run `python -c 'import __graft_entry__ as g; g.build()'`). There is no CPU fallback.")
    lib = ctypes.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc == CRB_OK:
        return
    msg = load_library().crb_last_error().decode("utf-8", "replace")
    if rc == CRB_ERR_ZERODIV:
        raise ZeroDivisionError(msg)
    if rc == CRB_ERR_RANGE:
        raise OverflowError(msg)
    if rc == CRB_ERR_SYNTAX:
        raise ValueError(msg)
    raise CrenderError(rc, msg)


def projection_matrix(h, w, fov=90.0, z_near=0.1, z_far=1000.0):
    """Host-only: the reference's proj_mat (pyx:83-90) as a [4,4] float32 array."""
    import numpy as np
    P = np.zeros(16, dtype=np.float32)
    check(load_library().crb_projection(int(h), int(w), float(fov), float(z_near), float(z_far),
                                        P.ctypes.data_as(_fp)))
    return P.reshape(4, 4)
