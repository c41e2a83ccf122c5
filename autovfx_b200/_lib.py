"""ctypes binding of the C-ABI library (include/gsr_b200.h).

There is NO fallback: if libgsr_b200.so cannot be loaded (and cannot be built because nvcc is absent)
importing this module raises, and every operator of the package fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

_f32p = C.c_void_p  # device pointers travel as plain integers


class gsr_frame(C.Structure):
    _fields_ = [
        ("P", C.c_int32), ("D", C.c_int32), ("M", C.c_int32), ("W", C.c_int32), ("H", C.c_int32),
        ("scale_modifier", C.c_float), ("tanfovx", C.c_float), ("tanfovy", C.c_float),
        ("prefiltered", C.c_int32), ("debug", C.c_int32),
        ("bg", _f32p), ("means3D", _f32p), ("shs", _f32p), ("colors_precomp", _f32p), ("opacities", _f32p),
        ("scales", _f32p), ("rotations", _f32p), ("cov3D_precomp", _f32p), ("viewmatrix", _f32p),
        ("projmatrix", _f32p), ("campos", _f32p),
    ]


class gsr_workspace(C.Structure):
    _fields_ = [("geom", C.c_void_p), ("geom_bytes", C.c_size_t), ("binning", C.c_void_p), ("binning_bytes", C.c_size_t),
                ("image", C.c_void_p), ("image_bytes", C.c_size_t)]


class gsr_counters(C.Structure):
    _fields_ = [("num_rendered", C.c_uint32), ("overflow", C.c_uint32), ("max_tile", C.c_uint32), ("trapped", C.c_uint32),
                ("num_visible", C.c_uint32), ("foot_total", C.c_uint32), ("exact_redos", C.c_uint32),
                ("blend_next", C.c_uint32)]


class gsr_grads(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("dL_dmeans2D", "dL_dconic", "dL_dopacity", "dL_dcolors", "dL_ddepths", "dL_dmeans3D",
                                          "dL_dcov3D", "dL_dsh", "dL_dscales", "dL_drotations")]


class gsr_views(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("records", "cov3D", "clamped", "point_list", "sorted_keys", "ranges", "n_contrib",
                                          "tile_count", "tile_big", "counters")]


class gsr_object_xform(C.Structure):
    _fields_ = [("rotation", C.c_float * 9), ("quat", C.c_float * 4), ("center", C.c_float * 3), ("initial_center", C.c_float * 3),
                ("scaling", C.c_float), ("log_scaling", C.c_float)]


GSR_FLAG_FOR_BACKWARD = 1
GSR_FLAG_SORTED_KEYS = 2
GSR_FLAG_TIGHT_TILES = 4
GSR_FLAG_REUSE_GEOMETRY = 8
GSR_FLAG_EXACT_IMAGES = 16
GSR_FLAG_BINNING_ONLY = 32
GSR_FLAG_RESUME = 64
ABI_VERSION = 4

EXPORTS = ("gsr_abi_version", "gsr_last_error", "gsr_geom_bytes", "gsr_binning_bytes", "gsr_binning_capacity", "gsr_image_bytes",
           "gsr_forward", "gsr_backward", "gsr_mark_visible", "gsr_dist2_bytes", "gsr_dist2", "gsr_get_views",
           "gsr_profile_begin", "gsr_profile_begin_strided", "gsr_profile_end", "gsr_forward_multi", "gsr_axis_normals", "gsr_normal_maps",
           "gsr_pack_frame", "gsr_activate_gaussians", "gsr_set_option", "gsr_backward_multi")


def _load() -> C.CDLL:
    path = _build.SO_PATH
    if _build.is_stale():
        # rebuild where a toolkit exists; a stale prebuilt library is still used on a box without nvcc
        try:
            _build.build()
        except Exception as ex:  # noqa: BLE001
            if not os.path.exists(path):
                raise ImportError("autovfx_b200: CUDA library %s is missing and cannot be built (%s). "
                                  "There is no CPU fallback." % (path, ex)) from ex
    lib = C.CDLL(path)
    for name in EXPORTS:
        if not hasattr(lib, name):
            raise ImportError("autovfx_b200: %s does not export %s" % (path, name))
    lib.gsr_abi_version.restype = C.c_int
    if lib.gsr_abi_version() != ABI_VERSION:
        raise ImportError("autovfx_b200: ABI mismatch, rebuild with `python -m autovfx_b200.build --force`")
    lib.gsr_last_error.restype = C.c_char_p
    for n in ("gsr_geom_bytes", "gsr_image_bytes", "gsr_binning_bytes", "gsr_binning_capacity", "gsr_dist2_bytes"):
        getattr(lib, n).restype = C.c_size_t
    lib.gsr_geom_bytes.argtypes = [C.c_int32]
    lib.gsr_image_bytes.argtypes = [C.c_int32, C.c_int32]
    lib.gsr_binning_bytes.argtypes = [C.c_size_t]
    lib.gsr_binning_capacity.argtypes = [C.c_size_t]
    lib.gsr_dist2_bytes.argtypes = [C.c_int32]
    lib.gsr_forward.restype = C.c_int
    lib.gsr_forward.argtypes = [C.POINTER(gsr_frame), C.POINTER(gsr_workspace), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_int, C.c_void_p]
    lib.gsr_forward_multi.restype = C.c_int
    lib.gsr_forward_multi.argtypes = [C.POINTER(gsr_frame), C.POINTER(gsr_workspace), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    lib.gsr_axis_normals.restype = C.c_int
    lib.gsr_axis_normals.argtypes = [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    lib.gsr_normal_maps.restype = C.c_int
    lib.gsr_normal_maps.argtypes = [C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_float, C.c_float,
                                    C.c_void_p, C.c_void_p, C.c_void_p]
    lib.gsr_pack_frame.restype = C.c_int
    lib.gsr_pack_frame.argtypes = [C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p]
    lib.gsr_activate_gaussians.restype = C.c_int
    lib.gsr_activate_gaussians.argtypes = [C.c_int32, C.c_int32] + [C.c_void_p] * 6 + [C.POINTER(gsr_object_xform)] + [C.c_void_p] * 6
    lib.gsr_backward.restype = C.c_int
    lib.gsr_backward.argtypes = [C.POINTER(gsr_frame), C.POINTER(gsr_workspace), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.POINTER(gsr_grads), C.c_void_p]
    lib.gsr_backward_multi.restype = C.c_int
    lib.gsr_backward_multi.argtypes = [C.POINTER(gsr_frame), C.POINTER(gsr_workspace), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(gsr_grads), C.c_void_p, C.c_void_p]
    lib.gsr_mark_visible.restype = C.c_int
    lib.gsr_mark_visible.argtypes = [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.gsr_dist2.restype = C.c_int
    lib.gsr_dist2.argtypes = [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.gsr_get_views.restype = C.c_int
    lib.gsr_get_views.argtypes = [C.POINTER(gsr_workspace), C.c_int32, C.c_int32, C.c_int32, C.POINTER(gsr_views)]
    lib.gsr_profile_begin.restype = C.c_int
    lib.gsr_profile_begin.argtypes = [C.c_int]
    lib.gsr_profile_begin_strided.restype = C.c_int
    lib.gsr_profile_begin_strided.argtypes = [C.c_int, C.c_int]
    lib.gsr_set_option.restype = C.c_int
    lib.gsr_set_option.argtypes = [C.c_char_p, C.c_int]
    lib.gsr_profile_end.restype = C.c_int
    lib.gsr_profile_end.argtypes = [C.POINTER(C.c_float), C.POINTER(C.c_int)]
    return lib


lib = _load()

# GSR_OPTIONS="name=value,name=value": gsr_set_option calls at import (experiment harnesses; every setting renders the same bits)
for _kv in filter(None, os.environ.get("GSR_OPTIONS", "").split(",")):
    _k, _v = _kv.split("=")
    if lib.gsr_set_option(_k.strip().encode(), int(_v)) != 0:
        raise ImportError("autovfx_b200: bad GSR_OPTIONS entry %r" % _kv)


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise RuntimeError("%s failed (%d): %s" % (what, rc, lib.gsr_last_error().decode("utf-8", "replace")))
