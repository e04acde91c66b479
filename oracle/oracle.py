"""ctypes wrapper over oracle/libgeo_oracle.so — TEST INFRASTRUCTURE ONLY.

The oracle restates the CPU arithmetic the reference delegates to geo 0.27 / robust 1.1 (see
oracle/geo_oracle.h for citations and parity status: pinned for contains() only, otherwise
"parity unpinned").  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs may import this module; geopolars_b200/ never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from dataclasses import dataclass
from typing import Optional

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libgeo_oracle.so")

POINT, LINESTRING, POLYGON, MULTIPOINT, MULTILINESTRING, MULTIPOLYGON = 0, 1, 3, 4, 5, 6


class _OgArray(C.Structure):
    _fields_ = [
        ("type", C.c_int32),
        ("n", C.c_int64),
        ("xy", C.c_void_p),
        ("geom_off", C.c_void_p),
        ("part_off", C.c_void_p),
        ("ring_off", C.c_void_p),
        ("valid", C.c_void_p),
    ]


def _cpu_signature():
    """identifies the host CPU (model + ISA flags) and the oracle's source: a -march=native build is only valid where it
    was made, and only for the source it was made from"""
    import hashlib

    h = hashlib.sha1()
    for name in ("geo_oracle.c", "geo_oracle.h", "Makefile"):
        with open(os.path.join(_HERE, name), "rb") as f:
            h.update(f.read())
    model, flags = "", ""
    try:
        with open("/proc/cpuinfo") as f:
            for ln in f:
                if ln.startswith("model name") and not model:
                    model = ln.split(":", 1)[1].strip()
                elif ln.startswith("flags") and not flags:
                    flags = ln.split(":", 1)[1].strip()
                if model and flags:
                    break
    except OSError:
        pass
    h.update((model + "|" + flags).encode())
    return model, h.hexdigest()[:12]


def _private_dir(path: str) -> str:
    """create `path` if needed and return it, but only if it is a real directory (not a link) that belongs to this
    user and that no one else can enter: the temporary directory is shared, and a library found there gets loaded"""
    import stat

    os.makedirs(path, mode=0o700, exist_ok=True)
    st = os.lstat(path)
    if not stat.S_ISDIR(st.st_mode) or st.st_uid != os.getuid() or st.st_mode & 0o077:
        raise PermissionError(f"{path} is not a directory private to this user; the native oracle is not cached there")
    return path


def _build_native(sig: str) -> str:
    """Compile the -march=native build for this host into a private per-user temporary directory (the source tree
    may be read-only) and return its directory.  Each build goes to a fresh directory that is then renamed into
    place, so that concurrent processes never load a half-written library."""
    import shutil
    import tempfile

    base = _private_dir(os.path.join(tempfile.gettempdir(), f"geo_oracle-{os.getuid()}"))
    ndir = os.path.join(base, sig)
    if os.path.exists(os.path.join(ndir, "flags.txt")):
        return ndir
    tmp = tempfile.mkdtemp(dir=base)
    try:
        subprocess.check_call(["make", "-C", _HERE, "-s", "native", f"NATIVE_DIR={tmp}"],
                              stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        os.rename(tmp, ndir)
    except OSError:
        if not os.path.exists(os.path.join(ndir, "flags.txt")):  # not another process's finished build
            raise
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    return ndir


_build_info = {"flags": None, "cpu": None, "so": None, "native": False}


def build(force: bool = False) -> str:
    """Compile the oracle with the recipe in oracle/Makefile (building the checker is not using it).
    Returns the library to load: the -march=native build for THIS host when it can be made (BASELINE.md's
    `-O3 -march=native -ffp-contract=off` CPU arm), else the portable build that ships with the snapshot."""
    src = os.path.join(_HERE, "geo_oracle.c")
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    model, sig = _cpu_signature()
    _build_info.update(cpu=model, so=_SO, native=False)
    try:
        _build_info["flags"] = subprocess.check_output(["make", "-C", _HERE, "-s", "flags"], text=True).strip()
    except Exception:
        _build_info["flags"] = "portable build (flags unknown)"
    if os.environ.get("GEO_ORACLE_NATIVE", "1") != "0":
        try:
            ndir = _build_native(sig)
            with open(os.path.join(ndir, "flags.txt")) as f:
                _build_info.update(flags=f.read().strip(), so=os.path.join(ndir, "libgeo_oracle.so"), native=True)
        except Exception:
            pass  # no compiler on this host: the portable build stands
    return _build_info["so"]


def build_info() -> dict:
    """compiler flags, CPU model and path of the library in use (bench.py prints them next to the CPU arm)"""
    lib()
    return dict(_build_info)


_lib = None


def lib():
    global _lib
    if _lib is None:
        so = build()
        try:
            L = C.CDLL(so)
        except OSError:
            L = C.CDLL(_SO)
            _build_info.update(so=_SO, native=False)
        L.og_orient2d.restype = C.c_double
        L.og_orient2d.argtypes = [C.c_double] * 6
        L.og_orient2d_adapt_calls.restype = C.c_int64
        L.og_splitmix_u.restype = C.c_double
        L.og_splitmix_u.argtypes = [C.c_uint64, C.c_uint64]
        L.og_convex_hull_one.restype = C.c_int64
        L.og_convex_hull.restype = C.c_int64
        L.og_coord_position.restype = C.c_int
        L.og_coord_position.argtypes = [C.c_void_p, C.c_int64, C.c_double, C.c_double]
        L.og_contains_point.restype = C.c_int
        L.og_contains_point.argtypes = [C.c_void_p, C.c_int64, C.c_double, C.c_double]
        L.og_distance_rowwise.restype = C.c_int
        L.og_max_threads.restype = C.c_int
        _lib = L
    return _lib


@dataclass
class OGArray:
    """GeoArrow-nested geometry array on the host: interleaved xy + int64 offsets."""

    type: int
    xy: np.ndarray  # (n_coords, 2) float64 C-contiguous
    geom_off: Optional[np.ndarray] = None
    part_off: Optional[np.ndarray] = None
    ring_off: Optional[np.ndarray] = None
    valid: Optional[np.ndarray] = None  # bool per geometry

    def __post_init__(self):
        self.xy = np.ascontiguousarray(self.xy, dtype=np.float64).reshape(-1, 2)
        for k in ("geom_off", "part_off", "ring_off"):
            v = getattr(self, k)
            if v is not None:
                setattr(self, k, np.ascontiguousarray(v, dtype=np.int64))
        if self.valid is not None:
            self.valid = np.ascontiguousarray(self.valid, dtype=bool)

    def __len__(self) -> int:
        if self.type == POINT:
            return self.xy.shape[0]
        return len(self.geom_off) - 1

    def _c(self):
        keep = []
        s = _OgArray()
        s.type = self.type
        s.n = len(self)
        s.xy = self.xy.ctypes.data
        for k in ("geom_off", "part_off", "ring_off"):
            v = getattr(self, k)
            setattr(s, k, v.ctypes.data if v is not None else None)
        if self.valid is not None:
            bits = np.packbits(self.valid, bitorder="little")
            keep.append(bits)
            s.valid = bits.ctypes.data
        else:
            s.valid = None
        keep.append(s)
        return s, keep


def _p(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def orient2d(a, b, c) -> float:
    return lib().og_orient2d(a[0], a[1], b[0], b[1], c[0], c[1])


def adapt_calls() -> int:
    return lib().og_orient2d_adapt_calls()


def max_threads() -> int:
    return lib().og_max_threads()


def affine_transform(xy: np.ndarray, m, threads: int = 1) -> np.ndarray:
    """m = (a, b, xoff, d, e, yoff) — geo's AffineTransform::new order."""
    xy = np.ascontiguousarray(xy, dtype=np.float64).reshape(-1, 2)
    out = np.empty_like(xy)
    a, b, xoff, d, e, yoff = [float(v) for v in m]
    lib().og_affine_transform(_p(xy), C.c_int64(xy.shape[0]), C.c_double(a), C.c_double(b), C.c_double(xoff),
                              C.c_double(d), C.c_double(e), C.c_double(yoff), _p(out), C.c_int(threads))
    return out


def area(arr: OGArray, threads: int = 1) -> np.ndarray:
    s, keep = arr._c()
    out = np.empty(len(arr), dtype=np.float64)
    lib().og_area(C.byref(s), _p(out), C.c_int(threads))
    return out


def centroid(arr: OGArray, threads: int = 1):
    s, keep = arr._c()
    out = np.empty((len(arr), 2), dtype=np.float64)
    valid = np.empty(len(arr), dtype=np.uint8)
    lib().og_centroid(C.byref(s), _p(out), _p(valid), C.c_int(threads))
    return out, valid.astype(bool)


def envelope(arr: OGArray, threads: int = 1):
    s, keep = arr._c()
    out = np.empty((len(arr), 4), dtype=np.float64)
    valid = np.empty(len(arr), dtype=np.uint8)
    lib().og_envelope(C.byref(s), _p(out), _p(valid), C.c_int(threads))
    return out, valid.astype(bool)


def envelope_query(arr: OGArray, box, mode: int = 0) -> np.ndarray:
    """rstar 0.11 `RTree::locate_in_envelope(&AABB::from_corners(lo, hi))` over the per-row envelopes
    (geopolars/src/spatial_index.rs:206-312 builds them, the tests at :361-430 query them): mode 0 = rows whose
    envelope lies INSIDE the closed box (`AABB::contains_envelope`: lower <= lower' and upper' <= upper per axis);
    mode 1 = rows whose envelope INTERSECTS it (`locate_in_envelope_intersecting`, the candidate test of the join,
    :74-76).  Rows without an envelope (empty / null) never match."""
    b, has = envelope(arr)
    x0, y0, x1, y1 = (float(v) for v in box)
    has = has & ~np.isnan(b).any(axis=1)
    if mode == 0:
        m = (b[:, 0] >= x0) & (b[:, 1] >= y0) & (b[:, 2] <= x1) & (b[:, 3] <= y1)
    else:
        m = (b[:, 0] <= x1) & (b[:, 2] >= x0) & (b[:, 1] <= y1) & (b[:, 3] >= y0)
    return m & has


def euclidean_length(arr: OGArray, threads: int = 1) -> np.ndarray:
    s, keep = arr._c()
    out = np.empty(len(arr), dtype=np.float64)
    lib().og_euclidean_length(C.byref(s), _p(out), C.c_int(threads))
    return out


def coord_position(polys: OGArray, i: int, x: float, y: float) -> int:
    s, keep = polys._c()
    return lib().og_coord_position(C.addressof(s), i, x, y)


def contains_point(polys: OGArray, i: int, x: float, y: float) -> bool:
    s, keep = polys._c()
    return bool(lib().og_contains_point(C.addressof(s), i, x, y))


def contains_join(polys: OGArray, pts_xy: np.ndarray, use_grid: bool = True, threads: int = 1):
    s, keep = polys._c()
    pts = np.ascontiguousarray(pts_xy, dtype=np.float64).reshape(-1, 2)
    first = np.empty(pts.shape[0], dtype=np.int32)
    count = np.empty(pts.shape[0], dtype=np.int32)
    lib().og_contains_join(C.byref(s), _p(pts), C.c_int64(pts.shape[0]), _p(first), _p(count),
                           C.c_int(1 if use_grid else 0), C.c_int(threads))
    return first, count


def intersects_rowwise(a: OGArray, b: OGArray, threads: int = 1) -> np.ndarray:
    sa, ka = a._c()
    sb, kb = b._c()
    out = np.empty(len(a), dtype=np.uint8)
    lib().og_intersects_rowwise(C.byref(sa), C.byref(sb), _p(out), C.c_int(threads))
    return out.astype(bool)


def contains_rowwise(a: OGArray, pts_xy: np.ndarray, threads: int = 1) -> np.ndarray:
    """a[i] contains point i — (Multi)Polygon or (Multi)LineString rows"""
    sa, ka = a._c()
    pts = np.ascontiguousarray(pts_xy, dtype=np.float64)
    out = np.empty(len(a), dtype=np.uint8)
    lib().og_contains_rowwise(C.byref(sa), _p(pts), None, _p(out), C.c_int(threads))
    return out.astype(bool)


def contains_polygon_rowwise(a: OGArray, b: OGArray, threads: int = 1) -> np.ndarray:
    """(Multi)Polygon.contains(Polygon), row-wise (spatial_index.rs:99-110)"""
    sa, ka = a._c()
    sb, kb = b._c()
    out = np.zeros(len(a), dtype=np.uint8)
    rc = lib().og_contains_polygon_rowwise(C.byref(sa), C.byref(sb), _p(out), C.c_int(threads))
    if rc != 0:
        raise ValueError("contains: expected (Multi)Polygon x Polygon columns of equal length")
    return out.astype(bool)


def distance_rowwise(a: OGArray, b: OGArray, threads: int = 1) -> np.ndarray:
    sa, ka = a._c()
    sb, kb = b._c()
    out = np.empty(len(a), dtype=np.float64)
    rc = lib().og_distance_rowwise(C.byref(sa), C.byref(sb), _p(out), C.c_int(threads))
    if rc != 0:
        raise ValueError("unsupported geometry type pair or length mismatch")
    return out


GEODESIC_METHODS = {"geodesic": 0, "haversine": 1, "vincenty": 2}


def geodesic_length(arr: OGArray, method: str = "geodesic", threads: int = 1) -> np.ndarray:
    s, k = arr._c()
    out = np.empty(len(arr), dtype=np.float64)
    rc = lib().og_geodesic_length(C.byref(s), C.c_int(GEODESIC_METHODS[method]), _p(out), C.c_int(threads))
    assert rc == 0
    return out


def geodesic_distance(method: str, lon1, lat1, lon2, lat2) -> float:
    L = lib()
    L.og_geodesic_distance.restype = C.c_double
    L.og_geodesic_distance.argtypes = [C.c_int] + [C.c_double] * 4
    return L.og_geodesic_distance(GEODESIC_METHODS[method], lon1, lat1, lon2, lat2)


def simplify_mask(arr: OGArray, eps: float, threads: int = 1) -> np.ndarray:
    """bool per input coordinate: retained by geo's Ramer-Douglas-Peucker"""
    s, k = arr._c()
    keep = np.zeros(len(arr.xy), dtype=np.uint8)
    rc = lib().og_simplify_mask(C.byref(s), C.c_double(eps), _p(keep), C.c_int(threads))
    if rc != 0:
        raise TypeError("simplify: LineString / MultiLineString / Polygon / MultiPolygon only")
    return keep.astype(bool)


def convex_hull(arr: OGArray, threads: int = 1):
    """returns (ring_off int64[n+1], xy (total,2)) — one closed ring per geometry."""
    s, keep = arr._c()
    n = len(arr)
    off = np.zeros(n + 1, dtype=np.int64)
    total = lib().og_convex_hull(C.byref(s), _p(off), None, C.c_int(threads))
    xy = np.empty((total, 2), dtype=np.float64)
    lib().og_convex_hull(C.byref(s), _p(off), _p(xy), C.c_int(threads))
    return off, xy


def gen_uniform_points(stream: int, first: int, n: int, scale: float) -> np.ndarray:
    out = np.empty((n, 2), dtype=np.float64)
    lib().og_gen_uniform_points(C.c_uint64(stream), C.c_int64(first), C.c_int64(n), C.c_double(scale), _p(out))
    return out
