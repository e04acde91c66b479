"""Thin object layer over the C ABI: Context (device + stream), DeviceArray (GeoArrow in HBM),
PipIndex (polygon side of a contains join) and one function per GeoSeries op.

Reference boundary mirrored: `impl GeoSeries for Series` (geopolars/geopolars-geo/src/geoseries.rs:10-181)
— same op names and argument meaning; errors map to the reference's exception classes
(py-geopolars/src/error.rs:27-60).  Everything here calls libgeopolars_b200.so; nothing falls back
to the CPU.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence, Tuple

import numpy as np

from . import _lib
from ._lib import GPL_DEVICE, GPL_HOST, check  # noqa: F401 (re-exported for bench.py)
from .geoarrow import GeoArrowArray, GeometryType


def _np_ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data


class Context:
    """One per (host thread, device).  `stream` is a raw cudaStream_t (int) to enqueue on, e.g.
    torch.cuda.current_stream().cuda_stream, or None for a private non-blocking stream."""

    def __init__(self, device: int = 0, stream: Optional[int] = None):
        self.lib = _lib.load()
        self.device = device
        h = C.c_void_p()
        check(self.lib.gpl_ctx_create(device, C.c_void_p(stream) if stream else None, C.byref(h)))
        self._h = h

    def set_stream(self, stream: Optional[int]) -> None:
        check(self.lib.gpl_ctx_set_stream(self._h, C.c_void_p(stream) if stream else None))

    def synchronize(self) -> None:
        check(self.lib.gpl_ctx_synchronize(self._h))

    def trim(self) -> None:
        """return the allocator's cached free blocks to the driver"""
        check(self.lib.gpl_ctx_trim(self._h))

    @property
    def launch_count(self) -> int:
        return int(self.lib.gpl_ctx_launch_count(self._h))

    def kernel_timing(self, enable: bool) -> None:
        """bracket every launch of the streaming join kernel with CUDA events (measurement aid, see the header)"""
        check(self.lib.gpl_ctx_kernel_timing(self._h, 1 if enable else 0))

    def kernel_timing_read(self):
        """(summed ms, launches) of the bracketed launches since the previous read; waits for them"""
        ms, n = C.c_double(0.0), C.c_int64(0)
        check(self.lib.gpl_ctx_kernel_timing_read(self._h, C.byref(ms), C.byref(n)))
        return float(ms.value), int(n.value)

    def close(self) -> None:
        if getattr(self, "_h", None):
            self.lib.gpl_ctx_destroy(self._h)
            self._h = None

    # -- arrays ------------------------------------------------------------------------------------
    def upload(self, arr: GeoArrowArray, offset_width: int = 64) -> "DeviceArray":
        """Copy a host GeoArrow array to HBM once (cudaMemcpyAsync on the context stream)."""
        b = _lib.Buffers()
        keep = []
        b.geom_type = int(arr.type)
        b.offset_width = offset_width
        b.mem = GPL_HOST
        b.n_geoms, b.n_parts, b.n_rings, b.n_coords = len(arr), arr.n_parts, arr.n_rings, arr.n_coords
        b.x = arr.xy.ctypes.data
        b.y = None
        dt = np.int64 if offset_width == 64 else np.int32
        for name, field in (("geom_off", "geom_offsets"), ("part_off", "part_offsets"), ("ring_off", "ring_offsets")):
            v = getattr(arr, name)
            if v is not None:
                vv = np.ascontiguousarray(v, dtype=dt)
                keep.append(vv)
                setattr(b, field, vv.ctypes.data)
        bm = arr.validity_bitmap()
        if bm is not None:
            keep.append(bm)
            b.validity = bm.ctypes.data
        h = C.c_void_p()
        check(self.lib.gpl_array_from_buffers(self._h, C.byref(b), C.byref(h)))
        return DeviceArray(self, h)

    def upload_separated(self, type: GeometryType, x: np.ndarray, y: np.ndarray, geom_off=None, part_off=None, ring_off=None,
                         valid=None, offset_width: int = 32) -> "DeviceArray":
        """GeoArrow Struct{x,y} coordinates (what py-geopolars builds, internals/geoseries.py:87-107)."""
        x = np.ascontiguousarray(x, dtype=np.float64)
        y = np.ascontiguousarray(y, dtype=np.float64)
        b = _lib.Buffers()
        keep = [x, y]
        b.geom_type = int(type)
        b.offset_width = offset_width
        b.mem = GPL_HOST
        b.n_coords = x.shape[0]
        dt = np.int64 if offset_width == 64 else np.int32
        offs = {"geom_offsets": geom_off, "part_offsets": part_off, "ring_offsets": ring_off}
        for field, v in offs.items():
            if v is not None:
                vv = np.ascontiguousarray(v, dtype=dt)
                keep.append(vv)
                setattr(b, field, vv.ctypes.data)
        b.n_geoms = x.shape[0] if int(type) == GeometryType.POINT else len(geom_off) - 1
        b.n_parts = 0 if part_off is None else len(part_off) - 1
        b.n_rings = 0 if ring_off is None else len(ring_off) - 1
        b.x, b.y = x.ctypes.data, y.ctypes.data
        if valid is not None:
            bm = np.packbits(np.asarray(valid, dtype=bool), bitorder="little")
            keep.append(bm)
            b.validity = bm.ctypes.data
        h = C.c_void_p()
        check(self.lib.gpl_array_from_buffers(self._h, C.byref(b), C.byref(h)))
        return DeviceArray(self, h)

    def wrap_device(self, type: GeometryType, n_geoms: int, n_coords: int, xy_ptr: int, geom_off_ptr: int = 0,
                    part_off_ptr: int = 0, ring_off_ptr: int = 0, n_parts: int = 0, n_rings: int = 0, validity_ptr: int = 0,
                    keepalive=None) -> "DeviceArray":
        """Borrow buffers that already live in HBM (interleaved xy, int64 offsets): zero copies."""
        b = _lib.Buffers()
        b.geom_type = int(type)
        b.offset_width = 64
        b.mem = GPL_DEVICE
        b.n_geoms, b.n_parts, b.n_rings, b.n_coords = n_geoms, n_parts, n_rings, n_coords
        b.x = xy_ptr
        b.y = None
        b.geom_offsets = geom_off_ptr or None
        b.part_offsets = part_off_ptr or None
        b.ring_offsets = ring_off_ptr or None
        b.validity = validity_ptr or None
        h = C.c_void_p()
        check(self.lib.gpl_array_from_buffers(self._h, C.byref(b), C.byref(h)))
        d = DeviceArray(self, h)
        d._keepalive = keepalive
        return d

    def import_arrow(self, arr) -> "DeviceArray":
        """pyarrow geometry array (geoarrow nested layout or WKB binary) -> HBM, through the Arrow C Data
        Interface exactly like py-geopolars/src/ffi.rs:12-32 (`_export_to_c` into ArrowArray/ArrowSchema)."""
        import pyarrow as pa

        if isinstance(arr, pa.ChunkedArray):
            arr = arr.combine_chunks()  # the reference rechunks to one chunk first (ffi.rs:56)
        c_array = (C.c_uint8 * 80)()   # struct ArrowArray
        c_schema = (C.c_uint8 * 72)()  # struct ArrowSchema
        arr._export_to_c(C.addressof(c_array), C.addressof(c_schema))
        h = C.c_void_p()
        try:
            check(self.lib.gpl_array_import_arrow(self._h, C.addressof(c_array), C.addressof(c_schema), C.byref(h)))
        finally:
            # import borrows: hand the structs back to pyarrow so that their release callbacks run
            pa.Array._import_from_c(C.addressof(c_array), C.addressof(c_schema))
        return DeviceArray(self, h)

    def from_wkb(self, wkb) -> "DeviceArray":
        """list of WKB bytes (None = null) or a pyarrow binary array, decoded once (util.rs:27-37 decodes per op)"""
        import pyarrow as pa

        if not isinstance(wkb, (pa.Array, pa.ChunkedArray)):
            wkb = pa.array(list(wkb), type=pa.binary())
        return self.import_arrow(wkb)

    def decode_wkb(self, data, offsets, valid=None, n=None, offset_width=None, device=False) -> "DeviceArray":
        """WKB column -> GeoArrow on the GPU (gpl_wkb_decode).  Host form: numpy `data` (uint8), `offsets`
        (int32 / int64, need not start at 0), `valid` (bool array or None).  Device form (`device=True`):
        `data`, `offsets`, `valid` are raw device addresses (ints; `valid` = Arrow bitmap), `n` rows,
        `offset_width` 32 | 64 — e.g. torch tensors' data_ptr()."""
        h = C.c_void_p()
        if device:
            check(self.lib.gpl_wkb_decode(self._h, C.c_void_p(data), C.c_void_p(offsets), int(offset_width),
                                          C.c_void_p(valid) if valid else None, int(n), GPL_DEVICE, C.byref(h)))
            return DeviceArray(self, h)
        offsets = np.ascontiguousarray(offsets)
        if offsets.dtype not in (np.int32, np.int64):
            offsets = offsets.astype(np.int64)
        data = np.ascontiguousarray(data, dtype=np.uint8)
        n = len(offsets) - 1
        bm = None if valid is None else np.packbits(np.asarray(valid, dtype=bool), bitorder="little")
        check(self.lib.gpl_wkb_decode(self._h, _np_ptr(data) if data.size else None, _np_ptr(offsets), 32 if offsets.dtype == np.int32 else 64,
                                      None if bm is None else _np_ptr(bm), n, GPL_HOST, C.byref(h)))
        return DeviceArray(self, h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class DeviceArray:
    """A GeoArrow geometry array resident in HBM (opaque gpl_array handle)."""

    def __init__(self, ctx: Context, handle: C.c_void_p):
        self.ctx = ctx
        self._h = handle
        self._keepalive = None

    def view(self) -> _lib.DeviceView:
        v = _lib.DeviceView()
        check(self.ctx.lib.gpl_array_view(self._h, C.byref(v)))
        return v

    @property
    def type(self) -> GeometryType:
        return GeometryType(self.view().geom_type)

    def __len__(self) -> int:
        return int(self.view().n_geoms)

    def to_host(self) -> GeoArrowArray:
        v = self.view()
        t = GeometryType(v.geom_type)
        xy = np.empty((v.n_coords, 2), dtype=np.float64)
        geom = np.empty(v.n_geoms + 1, dtype=np.int64) if v.geom_offsets else None
        part = np.empty(v.n_parts + 1, dtype=np.int64) if v.part_offsets else None
        ring = np.empty(v.n_rings + 1, dtype=np.int64) if v.ring_offsets else None
        bm = np.empty((v.n_geoms + 7) // 8, dtype=np.uint8) if v.validity else None
        check(self.ctx.lib.gpl_array_copy_out(self.ctx._h, self._h, _np_ptr(xy), _np_ptr(geom), _np_ptr(part), _np_ptr(ring),
                                              _np_ptr(bm), GPL_HOST))
        valid = None
        if bm is not None:
            valid = np.unpackbits(bm, bitorder="little")[: v.n_geoms].astype(bool)
            if valid.all():
                valid = None
        return GeoArrowArray(t, xy, geom_off=geom, part_off=part, ring_off=ring, valid=valid)

    def to_arrow(self):
        """HBM -> pyarrow geoarrow array through the Arrow C Data Interface (ffi.rs:36-49 in reverse)."""
        import pyarrow as pa

        c_array = (C.c_uint8 * 80)()
        c_schema = (C.c_uint8 * 72)()
        check(self.ctx.lib.gpl_array_export_arrow(self.ctx._h, self._h, C.addressof(c_array), C.addressof(c_schema)))
        return pa.Array._import_from_c(C.addressof(c_array), C.addressof(c_schema))

    def to_wkb(self):
        """ISO WKB (little endian) per row as a pyarrow binary array (from_geom_vec, util.rs:11-24)."""
        import pyarrow as pa

        n = len(self)
        off = np.zeros(n + 1, dtype=np.int32)
        nbytes = C.c_int64(0)
        check(self.ctx.lib.gpl_array_to_wkb(self.ctx._h, self._h, _np_ptr(off), None, C.byref(nbytes)))
        buf = np.empty(max(nbytes.value, 1), dtype=np.uint8)
        check(self.ctx.lib.gpl_array_to_wkb(self.ctx._h, self._h, _np_ptr(off), _np_ptr(buf), C.byref(nbytes)))
        host = self.to_host()
        validity = None if host.valid is None else pa.py_buffer(np.packbits(host.valid, bitorder="little").tobytes())
        return pa.Array.from_buffers(pa.binary(), n, [validity, pa.py_buffer(off.tobytes()), pa.py_buffer(buf[: nbytes.value].tobytes())])

    def encode_wkb(self, offset_width: int = 32, device_out=None):
        """GeoArrow -> WKB on the GPU (gpl_wkb_encode).  Returns (offsets, bytes) as numpy arrays; with
        `device_out=(offsets_ptr, bytes_ptr, capacity)` writes into device memory and returns the byte count."""
        n = len(self)
        nbytes = C.c_int64(0)
        lib, cx = self.ctx.lib, self.ctx._h
        if device_out is not None:
            optr, bptr, cap = device_out
            nbytes.value = int(cap)
            check(lib.gpl_wkb_encode(cx, self._h, C.c_void_p(optr), offset_width, C.c_void_p(bptr), C.byref(nbytes), GPL_DEVICE))
            return nbytes.value
        off = np.zeros(n + 1, dtype=np.int32 if offset_width == 32 else np.int64)
        check(lib.gpl_wkb_encode(cx, self._h, _np_ptr(off), offset_width, None, C.byref(nbytes), GPL_HOST))
        buf = np.empty(max(nbytes.value, 1), dtype=np.uint8)
        check(lib.gpl_wkb_encode(cx, self._h, _np_ptr(off), offset_width, _np_ptr(buf), C.byref(nbytes), GPL_HOST))
        return off, buf[: nbytes.value]

    def free(self) -> None:
        if getattr(self, "_h", None) and self.ctx._h:
            self.ctx.lib.gpl_array_free(self._h)
        self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def _out_array(ctx: Context, fn, *args) -> DeviceArray:
    h = C.c_void_p()
    check(fn(ctx._h, *args, C.byref(h)))
    return DeviceArray(ctx, h)


def _bits(bm: np.ndarray, n: int) -> np.ndarray:
    return np.unpackbits(bm, bitorder="little")[:n].astype(bool)


# ---- GeoSeries ops (names follow geoseries.rs:10-181) -------------------------------------------
def affine_transform(a: DeviceArray, m: Sequence[float]) -> DeviceArray:
    """m = (a, b, xoff, d, e, yoff): x' = a*x + b*y + xoff ; y' = d*x + e*y + yoff."""
    aa, b, xoff, d, e, yoff = [float(v) for v in m]
    return _out_array(a.ctx, a.ctx.lib.gpl_affine_transform, a._h, aa, b, xoff, d, e, yoff)


def translate(a: DeviceArray, xoff: float = 0.0, yoff: float = 0.0) -> DeviceArray:
    return _out_array(a.ctx, a.ctx.lib.gpl_translate, a._h, float(xoff), float(yoff))


def _origin(origin) -> Tuple[int, float, float]:
    """TransformOrigin parsing, same rules as py-geopolars/src/utils.rs:5-27."""
    if isinstance(origin, str):
        s = origin.lower()
        if s == "centroid":
            return _lib.ORIGIN_CENTROID, 0.0, 0.0
        if s == "center":
            return _lib.ORIGIN_CENTER, 0.0, 0.0
        raise ValueError("Invalid argument")
    if isinstance(origin, dict):
        return _lib.ORIGIN_POINT, float(origin["x"]), float(origin["y"])
    x, y = origin
    return _lib.ORIGIN_POINT, float(x), float(y)


def scale(a: DeviceArray, xfact: float = 1.0, yfact: float = 1.0, origin="center") -> DeviceArray:
    k, ox, oy = _origin(origin)
    return _out_array(a.ctx, a.ctx.lib.gpl_scale, a._h, float(xfact), float(yfact), k, ox, oy)


def rotate(a: DeviceArray, angle: float, origin="center") -> DeviceArray:
    k, ox, oy = _origin(origin)
    return _out_array(a.ctx, a.ctx.lib.gpl_rotate, a._h, float(angle), k, ox, oy)


def skew(a: DeviceArray, xs: float = 0.0, ys: float = 0.0, origin="center") -> DeviceArray:
    k, ox, oy = _origin(origin)
    return _out_array(a.ctx, a.ctx.lib.gpl_skew, a._h, float(xs), float(ys), k, ox, oy)


def area(a: DeviceArray) -> np.ndarray:
    out = np.empty(len(a), dtype=np.float64)
    check(a.ctx.lib.gpl_area(a.ctx._h, a._h, _np_ptr(out), GPL_HOST))
    return out


def euclidean_length(a: DeviceArray) -> np.ndarray:
    out = np.empty(len(a), dtype=np.float64)
    check(a.ctx.lib.gpl_euclidean_length(a.ctx._h, a._h, _np_ptr(out), GPL_HOST))
    return out


def centroid(a: DeviceArray) -> DeviceArray:
    return _out_array(a.ctx, a.ctx.lib.gpl_centroid, a._h)


def envelope(a: DeviceArray) -> DeviceArray:
    h = C.c_void_p()
    check(a.ctx.lib.gpl_envelope(a.ctx._h, a._h, C.byref(h), None, GPL_HOST))
    return DeviceArray(a.ctx, h)


def bounds(a: DeviceArray) -> np.ndarray:
    """minx, miny, maxx, maxy per geometry (NaN for empty)."""
    out = np.empty((len(a), 4), dtype=np.float64)
    check(a.ctx.lib.gpl_envelope(a.ctx._h, a._h, None, _np_ptr(out), GPL_HOST))
    return out


def envelope_query(a: DeviceArray, box, intersecting: bool = False) -> np.ndarray:
    """SpatialIndex.r_tree.locate_in_envelope(&AABB::from_corners(..)) (spatial_index.rs:385-387): rows whose envelope
    lies inside the closed box; `intersecting=True`: rows whose envelope meets it (the join's candidate test)."""
    n = len(a)
    bm = np.zeros((n + 7) // 8, dtype=np.uint8)
    x0, y0, x1, y1 = (float(v) for v in box)
    check(a.ctx.lib.gpl_envelope_query(a.ctx._h, a._h, x0, y0, x1, y1, 1 if intersecting else 0, _np_ptr(bm), GPL_HOST))
    return _bits(bm, n)


def convex_hull(a: DeviceArray) -> DeviceArray:
    return _out_array(a.ctx, a.ctx.lib.gpl_convex_hull, a._h)


GEODESIC_METHODS = {"geodesic": 0, "haversine": 1, "vincenty": 2}


def geodesic_length(a: DeviceArray, method: str = "geodesic") -> Tuple[np.ndarray, np.ndarray]:
    """GeoSeries::geodesic_length (geoseries.rs:52-58): metres; (values, valid) — a row is invalid when Vincenty fails"""
    m = GEODESIC_METHODS.get(str(method).lower())
    if m is None:
        raise ValueError("Geodesic calculation method not valid. Use one of geodesic, haversine or vincenty")
    n = len(a)
    out = np.empty(n, dtype=np.float64)
    bm = np.zeros((n + 7) // 8, dtype=np.uint8)
    check(a.ctx.lib.gpl_geodesic_length(a.ctx._h, a._h, m, _np_ptr(out), _np_ptr(bm), GPL_HOST))
    return out, _bits(bm, n)


def simplify(a: DeviceArray, tolerance: float) -> DeviceArray:
    """GeoSeries::simplify (geoseries.rs:108-116): geo's Ramer-Douglas-Peucker"""
    return _out_array(a.ctx, a.ctx.lib.gpl_simplify, a._h, C.c_double(float(tolerance)))


def exterior(a: DeviceArray) -> DeviceArray:
    return _out_array(a.ctx, a.ctx.lib.gpl_exterior, a._h)


def explode(a: DeviceArray) -> DeviceArray:
    return _out_array(a.ctx, a.ctx.lib.gpl_explode, a._h)


def distance(a: DeviceArray, b: DeviceArray) -> Tuple[np.ndarray, np.ndarray]:
    n = len(a)
    out = np.empty(n, dtype=np.float64)
    bm = np.zeros((n + 7) // 8, dtype=np.uint8)
    check(a.ctx.lib.gpl_distance(a.ctx._h, a._h, b._h, _np_ptr(out), _np_ptr(bm), GPL_HOST))
    return out, _bits(bm, n)


def intersects(a: DeviceArray, b: DeviceArray) -> np.ndarray:
    n = len(a)
    bm = np.zeros((n + 7) // 8, dtype=np.uint8)
    check(a.ctx.lib.gpl_intersects(a.ctx._h, a._h, b._h, _np_ptr(bm), GPL_HOST))
    return _bits(bm, n)


def contains(a: DeviceArray, b: DeviceArray) -> np.ndarray:
    """row-wise a[i].contains(b[i]): (Multi)Polygon / (Multi)LineString x Point, or (Multi)Polygon x Polygon (the pairs the
    reference's join dispatches, spatial_index.rs:89-135)"""
    n = len(a)
    bm = np.zeros((n + 7) // 8, dtype=np.uint8)
    fn = a.ctx.lib.gpl_contains_polygon if b.type == GeometryType.POLYGON else a.ctx.lib.gpl_contains
    check(fn(a.ctx._h, a._h, b._h, _np_ptr(bm), GPL_HOST))
    return _bits(bm, n)


PREDICATES = {"intersects": 0, "contains": 1}


def _pairs_to_host(ctx: Context, h) -> Tuple[np.ndarray, np.ndarray]:
    try:
        n = int(ctx.lib.gpl_pairs_count(h))
        lhs = np.empty(n, dtype=np.uint64)
        rhs = np.empty(n, dtype=np.uint64)
        if n:
            check(ctx.lib.gpl_pairs_copy(ctx._h, h, _np_ptr(lhs), _np_ptr(rhs), GPL_HOST))
    finally:
        ctx.lib.gpl_pairs_free(h)
    order = np.lexsort((rhs, lhs))  # the reference's order is unspecified (tree traversal): sorted by (lhs, rhs) here
    return lhs[order], rhs[order]


def spatial_join(lhs: DeviceArray, rhs: DeviceArray, predicate: str = "intersects") -> Tuple[np.ndarray, np.ndarray]:
    """(lhs_index, rhs_index) pairs of spatial_join(lhs, rhs, SpatialJoinArgs{predicate, ..}) for any two geometry columns
    (spatial_index.rs:37-157): envelope candidates + the reference's type-pair dispatch."""
    p = PREDICATES.get(str(predicate).lower())
    if p is None:
        raise ValueError("predicate must be 'intersects' or 'contains'")
    h = C.c_void_p()
    check(lhs.ctx.lib.gpl_spatial_join(lhs.ctx._h, lhs._h, rhs._h, p, C.byref(h)))
    return _pairs_to_host(lhs.ctx, h)


def geom_type(a: DeviceArray) -> np.ndarray:
    out = np.empty(len(a), dtype=np.int8)
    check(a.ctx.lib.gpl_geom_type(a.ctx._h, a._h, _np_ptr(out), GPL_HOST))
    return out


def is_empty(a: DeviceArray) -> np.ndarray:
    n = len(a)
    bm = np.zeros((n + 7) // 8, dtype=np.uint8)
    check(a.ctx.lib.gpl_is_empty(a.ctx._h, a._h, _np_ptr(bm), GPL_HOST))
    return _bits(bm, n)


def is_ring(a: DeviceArray) -> np.ndarray:
    n = len(a)
    bm = np.zeros((n + 7) // 8, dtype=np.uint8)
    check(a.ctx.lib.gpl_is_ring(a.ctx._h, a._h, _np_ptr(bm), GPL_HOST))
    return _bits(bm, n)


def x(a: DeviceArray) -> np.ndarray:
    out = np.empty(len(a), dtype=np.float64)
    check(a.ctx.lib.gpl_x(a.ctx._h, a._h, _np_ptr(out), GPL_HOST))
    return out


def y(a: DeviceArray) -> np.ndarray:
    out = np.empty(len(a), dtype=np.float64)
    check(a.ctx.lib.gpl_y(a.ctx._h, a._h, _np_ptr(out), GPL_HOST))
    return out


# ---- spatial join -------------------------------------------------------------------------------
class PipIndex:
    """Polygon side of a points-in-polygons join; stands in for SpatialIndex
    (geopolars/src/spatial_index.rs:314-350)."""

    def __init__(self, polygons: DeviceArray):
        self.ctx = polygons.ctx
        self.polygons = polygons  # keep alive: the index references its coordinates
        h = C.c_void_p()
        check(self.ctx.lib.gpl_pip_index_build(self.ctx._h, polygons._h, C.byref(h)))
        self._h = h

    @property
    def nbytes(self) -> int:
        return int(self.ctx.lib.gpl_pip_index_bytes(self._h))

    def stats(self) -> dict:
        """diagnostics: exact re-evaluations since the build, raster geometry and code census"""
        out = np.zeros(8, dtype=np.int64)
        check(self.ctx.lib.gpl_pip_index_stats(self.ctx._h, self._h, _np_ptr(out)))
        keys = ("deferred", "fine_cells_per_axis", "raster_log2", "raster_walk_cells", "raster_inside_cells", "parts_not_fast",
                "bytes", "coarse_cells_per_axis")
        return dict(zip(keys, (int(v) for v in out)))

    def phases(self):
        """microseconds from the start of the index fill kernel to its phase boundaries (diagnostics)"""
        out = np.zeros(12, dtype=np.float64)
        check(self.ctx.lib.gpl_pip_index_phases(self.ctx._h, self._h, _np_ptr(out)))
        return out[5:].tolist()

    def query(self, points_xy: np.ndarray, with_count: bool = False):
        """first containing polygon row per point (-1 = none) [+ number of containing rows]."""
        pts = np.ascontiguousarray(points_xy, dtype=np.float64).reshape(-1, 2)
        n = pts.shape[0]
        first = np.empty(n, dtype=np.int32)
        cnt = np.empty(n, dtype=np.int32) if with_count else None
        check(self.ctx.lib.gpl_contains_join(self.ctx._h, self._h, _np_ptr(pts), n, _np_ptr(first), _np_ptr(cnt), GPL_HOST))
        return (first, cnt) if with_count else first

    def query_device(self, points_ptr: int, n: int, first_ptr: int, count_ptr: int = 0) -> None:
        """all buffers already in HBM (bench `value` path): one kernel launch, stream ordered."""
        check(self.ctx.lib.gpl_contains_join(self.ctx._h, self._h, C.c_void_p(points_ptr), n, C.c_void_p(first_ptr),
                                             C.c_void_p(count_ptr) if count_ptr else None, GPL_DEVICE))

    def query_device_counts(self, points_ptr: int, n: int, first_ptr: int, counts_ptr: int) -> None:
        """join + per-polygon hit counts (u64 column, accumulated; a histogram of the id column); all buffers in HBM"""
        check(self.ctx.lib.gpl_contains_join_counts(self.ctx._h, self._h, C.c_void_p(points_ptr), n, C.c_void_p(first_ptr),
                                                    C.c_void_p(counts_ptr), GPL_DEVICE))

    def query_counts(self, points_xy: np.ndarray):
        """(first_id, per-polygon hit counts) from host points"""
        pts = np.ascontiguousarray(points_xy, dtype=np.float64).reshape(-1, 2)
        n = pts.shape[0]
        first = np.empty(n, dtype=np.int32)
        counts = np.zeros(len(self.polygons), dtype=np.uint64)
        check(self.ctx.lib.gpl_contains_join_counts(self.ctx._h, self._h, _np_ptr(pts), n, _np_ptr(first), _np_ptr(counts), GPL_HOST))
        return first, counts

    def query_array(self, points: DeviceArray, with_count: bool = False):
        n = len(points)
        first = np.empty(n, dtype=np.int32)
        cnt = np.empty(n, dtype=np.int32) if with_count else None
        check(self.ctx.lib.gpl_contains_join_array(self.ctx._h, self._h, points._h, _np_ptr(first), _np_ptr(cnt), GPL_HOST))
        return (first, cnt) if with_count else first

    def query_host_pipelined(self, points_ptr: int, n: int, first_ptr: int, chunk_points: int = 0) -> None:
        """host (ideally pinned) buffers; H2D / kernel / D2H overlapped in chunks (bench `e2e` path)."""
        check(self.ctx.lib.gpl_contains_join_host(self.ctx._h, self._h, C.c_void_p(points_ptr), n, C.c_void_p(first_ptr),
                                                  chunk_points))

    def pairs(self, points_xy: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
        """(lhs point index, rhs polygon row) pairs, the reference's join output (spatial_index.rs:139-157)."""
        pts = np.ascontiguousarray(points_xy, dtype=np.float64).reshape(-1, 2)
        n = pts.shape[0]
        total = C.c_int64(0)
        check(self.ctx.lib.gpl_contains_join_pairs(self.ctx._h, self._h, _np_ptr(pts), n, None, None, C.byref(total), GPL_HOST))
        lhs = np.empty(total.value, dtype=np.uint64)
        rhs = np.empty(total.value, dtype=np.uint64)
        if total.value:
            check(self.ctx.lib.gpl_contains_join_pairs(self.ctx._h, self._h, _np_ptr(pts), n, _np_ptr(lhs), _np_ptr(rhs),
                                                       C.byref(total), GPL_HOST))
        return lhs, rhs

    def pairs_array(self, points: DeviceArray) -> Tuple[np.ndarray, np.ndarray]:
        """the same pair list for a Point column that already lives in HBM (no host round trip of the points)"""
        h = C.c_void_p()
        check(self.ctx.lib.gpl_contains_join_pairs_array(self.ctx._h, self._h, points._h, C.byref(h)))
        return _pairs_to_host(self.ctx, h)

    def free(self) -> None:
        if getattr(self, "_h", None) and self.ctx._h:
            self.ctx.lib.gpl_pip_index_free(self._h)
        self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass
