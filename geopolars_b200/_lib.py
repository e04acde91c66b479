"""ctypes binding of libgeopolars_b200.so — the C ABI declared in include/geopolars_b200.h.

This is the Python-side twin of the reference's PyO3 module `_geopolars.geo`
(py-geopolars/src/api.rs:13-37): the reference moves Arrow buffers into Rust through the Arrow C Data
Interface (py-geopolars/src/ffi.rs:12-109) and calls `impl GeoSeries for Series`; here the same
buffers go through `gpl_*` entry points into HBM and hand-written sm_100a kernels.

There is NO CPU fallback: if the shared library is missing or no CUDA device is usable the import /
context creation fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# GEOPOLARS_B200_LIB: load another build of the same library.  The library reads no environment itself, so this is how
# two builds (say, before and after a kernel change) are compared on the same inputs.
SO_PATH = os.environ.get("GEOPOLARS_B200_LIB") or os.path.join(_HERE, "libgeopolars_b200.so")

GPL_HOST, GPL_DEVICE = 0, 1
ORIGIN_CENTROID, ORIGIN_CENTER, ORIGIN_POINT = 0, 1, 2

STATUS = {
    0: "GPL_OK",
    -1: "GPL_ERR_INVALID_TYPE",
    -2: "GPL_ERR_LENGTH_MISMATCH",
    -3: "GPL_ERR_CUDA",
    -4: "GPL_ERR_NCCL",
    -5: "GPL_ERR_OOM",
    -6: "GPL_ERR_UNSUPPORTED",
    -7: "GPL_ERR_INVALID_ARG",
}


class GeopolarsError(Exception):
    """Mirror of GeopolarsErrorException (py-geopolars/src/error.rs:13-25)."""

    def __init__(self, code: int, message: str):
        super().__init__(f"{STATUS.get(code, code)}: {message}")
        self.code = code


class MismatchedGeometry(GeopolarsError, TypeError):
    """GeopolarsError::MismatchedGeometry (geopolars/geopolars-geo/src/error.rs:12-16)."""


class ShapeError(GeopolarsError, ValueError):
    """polars ShapeMisMatch as mapped by py-geopolars/src/error.rs:27-60."""


class Buffers(C.Structure):
    _fields_ = [
        ("geom_type", C.c_int32),
        ("offset_width", C.c_int32),
        ("mem", C.c_int32),
        ("reserved", C.c_int32),
        ("n_geoms", C.c_int64),
        ("n_parts", C.c_int64),
        ("n_rings", C.c_int64),
        ("n_coords", C.c_int64),
        ("x", C.c_void_p),
        ("y", C.c_void_p),
        ("geom_offsets", C.c_void_p),
        ("part_offsets", C.c_void_p),
        ("ring_offsets", C.c_void_p),
        ("validity", C.c_void_p),
    ]


class DeviceView(C.Structure):
    _fields_ = [
        ("geom_type", C.c_int32),
        ("reserved", C.c_int32),
        ("n_geoms", C.c_int64),
        ("n_parts", C.c_int64),
        ("n_rings", C.c_int64),
        ("n_coords", C.c_int64),
        ("xy", C.c_void_p),
        ("geom_offsets", C.c_void_p),
        ("part_offsets", C.c_void_p),
        ("ring_offsets", C.c_void_p),
        ("validity", C.c_void_p),
    ]


_P = C.c_void_p
_I64 = C.c_int64
_D = C.c_double
_INT = C.c_int

# name -> (restype, argtypes); every symbol include/geopolars_b200.h declares
SIGNATURES = {
    "gpl_abi_version": (_INT, []),
    "gpl_last_error": (C.c_char_p, []),
    "gpl_ctx_create": (_INT, [_INT, _P, C.POINTER(_P)]),
    "gpl_ctx_set_stream": (_INT, [_P, _P]),
    "gpl_ctx_synchronize": (_INT, [_P]),
    "gpl_ctx_destroy": (None, [_P]),
    "gpl_ctx_trim": (_INT, [_P]),
    "gpl_ctx_launch_count": (_I64, [_P]),
    "gpl_ctx_kernel_timing": (_INT, [_P, _INT]),
    "gpl_ctx_kernel_timing_read": (_INT, [_P, C.POINTER(_D), C.POINTER(_I64)]),
    "gpl_host_alloc": (_INT, [C.c_size_t, C.POINTER(_P)]),
    "gpl_host_free": (None, [_P]),
    "gpl_array_from_buffers": (_INT, [_P, C.POINTER(Buffers), C.POINTER(_P)]),
    "gpl_array_view": (_INT, [_P, C.POINTER(DeviceView)]),
    "gpl_array_copy_out": (_INT, [_P, _P, _P, _P, _P, _P, _P, _INT]),
    "gpl_array_free": (None, [_P]),
    "gpl_array_from_wkb": (_INT, [_P, _P, _P, _P, _I64, C.POINTER(_P)]),
    "gpl_array_to_wkb": (_INT, [_P, _P, _P, _P, C.POINTER(_I64)]),
    "gpl_wkb_decode": (_INT, [_P, _P, _P, _INT, _P, _I64, _INT, C.POINTER(_P)]),
    "gpl_wkb_encode": (_INT, [_P, _P, _P, _INT, _P, C.POINTER(_I64), _INT]),
    "gpl_array_import_arrow": (_INT, [_P, _P, _P, C.POINTER(_P)]),
    "gpl_array_export_arrow": (_INT, [_P, _P, _P, _P]),
    "gpl_export_f64_arrow": (_INT, [_P, _P, _I64, _P, _P]),
    "gpl_export_bool_arrow": (_INT, [_P, _P, _I64, _P, _P]),
    "gpl_affine_transform": (_INT, [_P, _P, _D, _D, _D, _D, _D, _D, C.POINTER(_P)]),
    "gpl_translate": (_INT, [_P, _P, _D, _D, C.POINTER(_P)]),
    "gpl_scale": (_INT, [_P, _P, _D, _D, _INT, _D, _D, C.POINTER(_P)]),
    "gpl_rotate": (_INT, [_P, _P, _D, _INT, _D, _D, C.POINTER(_P)]),
    "gpl_skew": (_INT, [_P, _P, _D, _D, _INT, _D, _D, C.POINTER(_P)]),
    "gpl_area": (_INT, [_P, _P, _P, _INT]),
    "gpl_centroid": (_INT, [_P, _P, C.POINTER(_P)]),
    "gpl_envelope": (_INT, [_P, _P, C.POINTER(_P), _P, _INT]),
    "gpl_euclidean_length": (_INT, [_P, _P, _P, _INT]),
    "gpl_geodesic_length": (_INT, [_P, _P, _INT, _P, _P, _INT]),
    "gpl_convex_hull": (_INT, [_P, _P, C.POINTER(_P)]),
    "gpl_simplify": (_INT, [_P, _P, _D, C.POINTER(_P)]),
    "gpl_distance": (_INT, [_P, _P, _P, _P, _P, _INT]),
    "gpl_intersects": (_INT, [_P, _P, _P, _P, _INT]),
    "gpl_contains": (_INT, [_P, _P, _P, _P, _INT]),
    "gpl_geom_type": (_INT, [_P, _P, _P, _INT]),
    "gpl_is_empty": (_INT, [_P, _P, _P, _INT]),
    "gpl_is_ring": (_INT, [_P, _P, _P, _INT]),
    "gpl_x": (_INT, [_P, _P, _P, _INT]),
    "gpl_y": (_INT, [_P, _P, _P, _INT]),
    "gpl_exterior": (_INT, [_P, _P, C.POINTER(_P)]),
    "gpl_explode": (_INT, [_P, _P, C.POINTER(_P)]),
    "gpl_contains_polygon": (_INT, [_P, _P, _P, _P, _INT]),
    "gpl_spatial_join": (_INT, [_P, _P, _P, _INT, C.POINTER(_P)]),
    "gpl_pairs_count": (_I64, [_P]),
    "gpl_pairs_copy": (_INT, [_P, _P, _P, _P, _INT]),
    "gpl_pairs_free": (None, [_P]),
    "gpl_envelope_query": (_INT, [_P, _P, C.c_double, C.c_double, C.c_double, C.c_double, _INT, _P, _INT]),
    "gpl_pip_index_build": (_INT, [_P, _P, C.POINTER(_P)]),
    "gpl_pip_index_free": (None, [_P]),
    "gpl_pip_index_bytes": (_I64, [_P]),
    "gpl_pip_index_stats": (_INT, [_P, _P, _P]),
    "gpl_pip_index_phases": (_INT, [_P, _P, _P]),
    "gpl_contains_join": (_INT, [_P, _P, _P, _I64, _P, _P, _INT]),
    "gpl_contains_join_counts": (_INT, [_P, _P, _P, _I64, _P, _P, _INT]),
    "gpl_contains_join_array": (_INT, [_P, _P, _P, _P, _P, _INT]),
    "gpl_contains_join_pairs": (_INT, [_P, _P, _P, _I64, _P, _P, C.POINTER(_I64), _INT]),
    "gpl_contains_join_pairs_array": (_INT, [_P, _P, _P, C.POINTER(_P)]),
    "gpl_contains_join_host": (_INT, [_P, _P, _P, _I64, _P, _I64]),
    "gpl_join_histogram": (_INT, [_P, _P, _I64, _P, _I64, _INT]),
    "gpl_gen_uniform_points": (_INT, [_P, C.c_uint64, _I64, _I64, _D, _P]),
    "gpl_gen_walk_linestrings": (_INT, [_P, C.c_uint64, _I64, _I64, _I64, C.c_int32, _P, _P]),
    "gpl_gen_blob_polygons": (_INT, [_P, C.c_uint64, _I64, _I64, C.c_int32, _P, _P, _P]),
}

_lib = None


def load() -> C.CDLL:
    """Load the CUDA library; fail loudly when it has not been built (no silent CPU path)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise RuntimeError(
            f"{SO_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). geopolars_b200 has no CPU fallback."
        )
    lib = C.CDLL(SO_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here = header/library mismatch: fail loudly
        fn.restype = res
        fn.argtypes = args
    if lib.gpl_abi_version() != 1:
        raise RuntimeError(f"ABI version mismatch: library reports {lib.gpl_abi_version()}, binding expects 1")
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc == 0:
        return
    msg = load().gpl_last_error().decode("utf-8", "replace")
    if rc == -1:
        raise MismatchedGeometry(rc, msg)
    if rc == -2:
        raise ShapeError(rc, msg)
    raise GeopolarsError(rc, msg)
