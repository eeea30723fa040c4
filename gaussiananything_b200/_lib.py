"""ctypes binding of libga_b200.so (the C ABI in include/ga_b200.h).

There is NO CPU fallback: if the shared library is missing or does not load,
importing anything that computes raises.  Build it with
`python -m gaussiananything_b200.build` (nvcc, sm_100a).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# GA_B200_LIB: load a tuning build (gaussiananything_b200/build.py --variant) instead of the product library
LIB_PATH = os.environ.get("GA_B200_LIB") or os.path.join(_HERE, "libga_b200.so")

_lib = None


class GaRasterLayout(C.Structure):
    _fields_ = [(n, C.c_size_t) for n in (
        "total_bytes", "status", "rec", "depth", "rect", "tile_count", "tile_start",
        "keys", "ids", "final_T", "n_contrib", "inst_off", "inst_cnt", "n_list", "tile_flag", "tile_rec_start", "lists")]


def lib():
    """Returns the loaded library; raises loudly when it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "gaussiananything_b200: %s is missing -- build it with "
            "`python -m gaussiananything_b200.build` (there is no CPU fallback)" % LIB_PATH)
    import torch  # noqa: F401  (loads libcudart / libcuda into the process first)
    L = C.CDLL(LIB_PATH)
    vp, i32, i64, f32, sz = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_size_t
    L.ga_raster_layout.argtypes = [i32, i32, i32, i32, i32, i64, C.POINTER(GaRasterLayout)]
    L.ga_raster_layout.restype = i32
    L.ga_raster_layout_ex.argtypes = [i32, i32, i32, i32, i32, i64, i32, C.POINTER(GaRasterLayout)]
    L.ga_raster_layout_ex.restype = i32
    L.ga_raster_forward_ex.argtypes = [vp, i32, i32, i32, vp, vp, vp, i32, i32, f32, vp, vp, vp, vp, sz, i64, i32, vp, vp, vp]
    L.ga_raster_forward_ex.restype = i32
    L.ga_raster_backward_ex.argtypes = [vp, i32, i32, i32, vp, vp, vp, i32, i32, f32, vp, vp, vp, vp, sz, i64, i32, vp, sz, vp, vp]
    L.ga_raster_backward_ex.restype = i32
    L.ga_raster_forward.argtypes = [vp, i32, i32, i32, vp, vp, vp, i32, i32, f32,
                                    vp, vp, vp, vp, sz, i64, vp]
    L.ga_raster_forward.restype = i32
    for n in ("ga_raster_forward_bin", "ga_raster_forward_render"):
        getattr(L, n).argtypes = L.ga_raster_forward.argtypes
        getattr(L, n).restype = i32
    L.ga_raster_forward_async.argtypes = L.ga_raster_forward.argtypes[:-1] + [vp, vp, vp]
    L.ga_raster_forward_async.restype = i32
    L.ga_raster_backward_scratch_bytes.argtypes = [i32, i32, i32]
    L.ga_raster_backward_scratch_bytes.restype = sz
    L.ga_raster_backward_records.argtypes = [i32, i32, i32, i32, i32, vp, sz, i64, i32, vp, sz,
                                             C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), vp]
    L.ga_raster_backward_records.restype = i32
    L.ga_raster_backward.argtypes = [vp, i32, i32, i32, vp, vp, vp, i32, i32, f32,
                                     vp, vp, vp, vp, sz, i64, vp, sz, vp, vp]
    L.ga_raster_backward.restype = i32
    L.ga_render_post_forward.argtypes = [vp, vp, vp, i32, i32, i32, vp, vp, vp, vp, vp, vp]
    L.ga_render_post_forward.restype = i32
    L.ga_render_post_backward.argtypes = [vp, vp, vp, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp]
    L.ga_render_post_backward.restype = i32
    L.ga_b200_version.restype = C.c_char_p
    _lib = L
    return L


def check(rc, what):
    if rc != 0:
        raise RuntimeError("%s failed with code %d" % (what, rc))
