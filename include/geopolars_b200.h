/*
 * geopolars_b200.h — C ABI of the B200-native GeoSeries engine (libgeopolars_b200.so).
 *
 * This is the drop-in boundary for the reference's GeoSeries hot path: every entry point below is
 * what a reference-side FFI shim binds in place of the per-row `iter_geom(..).map(geo_algo)` loop
 * (reference: geopolars/geopolars-geo/src/util.rs:27-37) behind `impl GeoSeries for Series`
 * (geopolars/geopolars-geo/src/geoseries.rs:183-279).  Plain pointers and sizes only; no torch,
 * polars or C++ types cross this line.  INTEGRATION.md shows the Rust / PyO3 / ctypes binding.
 *
 * Conventions
 *   - every function returns gpl_status (0 = ok, <0 = error); the message for the calling thread is
 *     returned by gpl_last_error().  Error codes mirror GeopolarsError
 *     (geopolars/geopolars-geo/src/error.rs:9-28): INVALID_TYPE = MismatchedGeometry,
 *     LENGTH_MISMATCH = polars ShapeMisMatch.
 *   - geometry arrays use the GeoArrow nesting (coords + geom/part/ring offsets + validity bitmap),
 *     geometry type codes are the reference's GeometryType enum
 *     (py-geopolars/python/geopolars/enums.py:4-15).
 *   - inputs are borrowed for the duration of the call (Arrow C Data Interface ownership rules,
 *     py-geopolars/src/ffi.rs:10-31); outputs are either caller-provided buffers or library-owned
 *     gpl_array handles released with gpl_array_free().
 *   - `mem` arguments say where a caller buffer lives: GPL_HOST (copied with cudaMemcpyAsync on the
 *     context stream; pinned memory from gpl_host_alloc() makes that truly asynchronous) or
 *     GPL_DEVICE (used in place).
 *   - null rows propagate to null outputs (the reference panics on them, util.rs:32): a strict
 *     superset of the reference behaviour.
 *   - all work is enqueued on the context stream; functions that return data to GPL_HOST buffers
 *     synchronise that stream before returning, GPL_DEVICE results are stream-ordered.
 */
#ifndef GEOPOLARS_B200_H
#define GEOPOLARS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GPL_ABI_VERSION 1

typedef enum gpl_status {
    GPL_OK = 0,
    GPL_ERR_INVALID_TYPE = -1,    /* GeopolarsError::MismatchedGeometry (error.rs:12-16) */
    GPL_ERR_LENGTH_MISMATCH = -2, /* polars ShapeMisMatch (py-geopolars/src/error.rs:27-60) */
    GPL_ERR_CUDA = -3,
    GPL_ERR_NCCL = -4,
    GPL_ERR_OOM = -5,
    GPL_ERR_UNSUPPORTED = -6,
    GPL_ERR_INVALID_ARG = -7
} gpl_status;

typedef enum gpl_mem { GPL_HOST = 0, GPL_DEVICE = 1 } gpl_mem;

/* reference: py-geopolars/python/geopolars/enums.py:4-15 ; geoseries.rs:60-73 */
typedef enum gpl_geometry_type {
    GPL_MISSING = -1,
    GPL_POINT = 0,
    GPL_LINESTRING = 1,
    GPL_LINEARRING = 2,
    GPL_POLYGON = 3,
    GPL_MULTIPOINT = 4,
    GPL_MULTILINESTRING = 5,
    GPL_MULTIPOLYGON = 6,
    GPL_GEOMETRYCOLLECTION = 7
} gpl_geometry_type;

/* TransformOrigin of rotate/scale/skew (py-geopolars/src/utils.rs:5-27) */
typedef enum gpl_origin { GPL_ORIGIN_CENTROID = 0, GPL_ORIGIN_CENTER = 1, GPL_ORIGIN_POINT = 2 } gpl_origin;

typedef struct gpl_ctx gpl_ctx;             /* one per (host thread, device) */
typedef struct gpl_array gpl_array;         /* GeoArrow geometry array resident in HBM */
typedef struct gpl_pip_index gpl_pip_index;
typedef struct gpl_pairs gpl_pairs;         /* (lhs_index, rhs_index) pair list of a join, resident on the device */ /* polygon-side index of a contains join */

/* Raw GeoArrow buffers (the zero-dependency form of an Arrow array; replaces the WKB BinaryArray the
 * reference re-parses on every op, util.rs:27-37).
 *   POINT            coords[n_geoms]
 *   LINESTRING       geom_offsets[n_geoms+1] -> coords
 *   POLYGON          geom_offsets[n_geoms+1] -> rings ; ring_offsets[n_rings+1] -> coords
 *   MULTIPOINT       geom_offsets[n_geoms+1] -> coords
 *   MULTILINESTRING  geom_offsets[n_geoms+1] -> lines ; ring_offsets[n_rings+1] -> coords
 *   MULTIPOLYGON     geom_offsets[n_geoms+1] -> polygons ; part_offsets[n_parts+1] -> rings ;
 *                    ring_offsets[n_rings+1] -> coords
 * coords: interleaved (x = xy pairs, y = NULL; GeoArrow FixedSizeList<f64>[2]) or separated
 * (x, y; GeoArrow Struct{x,y}, what py-geopolars builds, internals/geoseries.py:87-107).
 * offsets: int32 (List) or int64 (LargeList), all three the same width. */
typedef struct gpl_buffers {
    int32_t geom_type;    /* gpl_geometry_type */
    int32_t offset_width; /* 32 or 64 */
    int32_t mem;          /* gpl_mem: where every pointer below lives */
    int32_t reserved;
    int64_t n_geoms;
    int64_t n_parts; /* MULTIPOLYGON only */
    int64_t n_rings; /* POLYGON, MULTILINESTRING, MULTIPOLYGON */
    int64_t n_coords;
    const double *x; /* interleaved xy when y == NULL */
    const double *y;
    const void *geom_offsets;
    const void *part_offsets;
    const void *ring_offsets;
    const uint8_t *validity; /* Arrow LSB-first bitmap over geometries, or NULL (= all valid) */
} gpl_buffers;

/* device-side view of a gpl_array (always interleaved coords + int64 offsets); pointers stay valid
 * until the array is freed. */
typedef struct gpl_device_view {
    int32_t geom_type;
    int32_t reserved;
    int64_t n_geoms, n_parts, n_rings, n_coords;
    const double *xy;
    const int64_t *geom_offsets, *part_offsets, *ring_offsets;
    const uint8_t *validity;
} gpl_device_view;

/* ---------------------------------------------------------------- context ---------------- */
int gpl_abi_version(void);
const char *gpl_last_error(void);
/* device: CUDA ordinal.  stream: an existing cudaStream_t to enqueue on (e.g. the caller's current
 * stream) or NULL to let the context create its own non-blocking stream. */
int gpl_ctx_create(int device, void *stream, gpl_ctx **out);
int gpl_ctx_set_stream(gpl_ctx *ctx, void *stream);
int gpl_ctx_synchronize(gpl_ctx *ctx);
/* Measurement aid (bench.py's roofline line): while enabled, every launch of the streaming points-in-polygons kernel
 * (k_pip_stream, the kernel behind gpl_contains_join* — reference path spatial_index.rs:139-157 + geo `Contains`) on this
 * context is bracketed by two CUDA events on the context's stream.  _read waits for the recorded pairs and returns their
 * summed duration (ms) and count since the previous read. */
int gpl_ctx_kernel_timing(gpl_ctx *ctx, int enable);
int gpl_ctx_kernel_timing_read(gpl_ctx *ctx, double *ms_total, int64_t *launches);
void gpl_ctx_destroy(gpl_ctx *ctx);
/* give the cached (free) device blocks of the context's allocator back to the driver */
int gpl_ctx_trim(gpl_ctx *ctx);
/* number of kernels this context has launched (bench.py's gpu_launches) */
int64_t gpl_ctx_launch_count(const gpl_ctx *ctx);
/* pinned host memory for truly asynchronous H2D/D2H */
int gpl_host_alloc(size_t bytes, void **out);
void gpl_host_free(void *p);

/* ---------------------------------------------------------------- arrays ----------------- */
/* Host buffers are copied to HBM once (cudaMemcpyAsync); device buffers are borrowed when they are
 * already interleaved / int64, converted into owned copies otherwise. */
int gpl_array_from_buffers(gpl_ctx *ctx, const gpl_buffers *b, gpl_array **out);
int gpl_array_view(const gpl_array *a, gpl_device_view *out);
/* copy an array back into caller buffers (any pointer may be NULL to skip it); offsets are written
 * as int64. */
int gpl_array_copy_out(gpl_ctx *ctx, const gpl_array *a, double *xy, int64_t *geom_offsets, int64_t *part_offsets,
                       int64_t *ring_offsets, uint8_t *validity, int mem);
void gpl_array_free(gpl_array *a);

/* WKB (ISO, either endianness, XY) -> GeoArrow, decoded ONCE (replaces util.rs:27-37 per-op parse).
 * offsets: int32[n+1] Arrow binary offsets into bytes; all rows must share one geometry type
 * (Polygon rows are promoted when mixed with MultiPolygon, LineString with MultiLineString,
 * Point with MultiPoint).  Host input. */
int gpl_array_from_wkb(gpl_ctx *ctx, const uint8_t *bytes, const int32_t *offsets, const uint8_t *validity,
                       int64_t n, gpl_array **out);
/* GeoArrow -> WKB (from_geom_vec, util.rs:11-24). Two calls: first with bytes == NULL to get
 * *n_bytes and offsets, then with a buffer of that size. Host output. */
int gpl_array_to_wkb(gpl_ctx *ctx, const gpl_array *a, int32_t *offsets, uint8_t *bytes, int64_t *n_bytes);
/* The codec itself, on the GPU (util.rs:11-37 is the per-row, per-op host loop it replaces): bytes / offsets /
 * validity in host OR device memory (`mem`), offsets int32 (`binary`) or int64 (`large_binary`) per
 * `offset_width`; offsets need not start at 0 (sliced arrays).  gpl_wkb_encode follows the two-call protocol
 * of gpl_array_to_wkb (bytes == NULL: offsets and *n_bytes only) and writes little-endian ISO WKB; null rows
 * are zero-length.  gpl_array_from_wkb / gpl_array_to_wkb are the (host, int32) forms of these. */
int gpl_wkb_decode(gpl_ctx *ctx, const uint8_t *bytes, const void *offsets, int offset_width, const uint8_t *validity,
                   int64_t n, int mem, gpl_array **out);
int gpl_wkb_encode(gpl_ctx *ctx, const gpl_array *a, void *offsets, int offset_width, uint8_t *bytes, int64_t *n_bytes,
                   int mem);

/* Arrow C Data Interface (same structs the reference moves across its FFI, py-geopolars/src/ffi.rs:14-49).
 * Accepts geoarrow nested layouts (interleaved or struct coords, List or LargeList) and WKB
 * binary / large_binary columns.  `array`/`schema` are struct ArrowArray* / struct ArrowSchema*;
 * import borrows (never releases) them. export fills caller-allocated structs whose release
 * callbacks free library-owned host memory. */
int gpl_array_import_arrow(gpl_ctx *ctx, const void *array, const void *schema, gpl_array **out);
int gpl_array_export_arrow(gpl_ctx *ctx, const gpl_array *a, void *out_array, void *out_schema);
/* primitive result columns (float64 / bool bitmap / int8 / int32) as Arrow arrays */
int gpl_export_f64_arrow(const double *values_host, const uint8_t *validity, int64_t n, void *out_array, void *out_schema);
int gpl_export_bool_arrow(const uint8_t *bitmap_host, const uint8_t *validity, int64_t n, void *out_array, void *out_schema);

/* ---------------------------------------------------------------- GeoSeries ops ---------- */
/* GeoSeries::affine_transform (geoseries.rs:11-12): x' = a*x + b*y + xoff ; y' = d*x + e*y + yoff.
 * Named scalars, not a [f64;6], because the reference's array order is ambiguous (SURVEY.md §7). */
int gpl_affine_transform(gpl_ctx *ctx, const gpl_array *in, double a, double b, double xoff, double d, double e,
                         double yoff, gpl_array **out);
/* GeoSeries::translate (geoseries.rs:174), scale (:107), rotate (:93, degrees), skew (:139, degrees).
 * origin: per-geometry centroid / bbox centre, or the fixed point (ox, oy). */
int gpl_translate(gpl_ctx *ctx, const gpl_array *in, double xoff, double yoff, gpl_array **out);
int gpl_scale(gpl_ctx *ctx, const gpl_array *in, double xfact, double yfact, int origin, double ox, double oy,
              gpl_array **out);
int gpl_rotate(gpl_ctx *ctx, const gpl_array *in, double angle_deg, int origin, double ox, double oy, gpl_array **out);
int gpl_skew(gpl_ctx *ctx, const gpl_array *in, double xs_deg, double ys_deg, int origin, double ox, double oy,
             gpl_array **out);

/* GeoSeries::area (geoseries.rs:14-16): out[n_geoms] f64 */
int gpl_area(gpl_ctx *ctx, const gpl_array *in, double *out, int mem);
/* GeoSeries::centroid (geoseries.rs:18-21): POINT array; empty geometries -> null */
int gpl_centroid(gpl_ctx *ctx, const gpl_array *in, gpl_array **out);
/* GeoSeries::envelope (geoseries.rs:28-33): POLYGON array of 5-coord rectangles; out4 (optional,
 * may be NULL) additionally receives minx,miny,maxx,maxy per geometry */
int gpl_envelope(gpl_ctx *ctx, const gpl_array *in, gpl_array **out, double *out4, int mem);
/* GeoSeries::euclidean_length (geoseries.rs:35-41) */
int gpl_euclidean_length(gpl_ctx *ctx, const gpl_array *in, double *out, int mem);
/* GeoSeries::geodesic_length (geoseries.rs:52-58; method names py-geopolars/src/geo.rs:64-67): metres, input in
 * (lon, lat) degrees.  method 0 = geodesic (Karney 2013, WGS84), 1 = haversine, 2 = vincenty.  out_validity
 * (optional bitmap): a row is null when a Vincenty segment does not converge (the reference returns Err) */
int gpl_geodesic_length(gpl_ctx *ctx, const gpl_array *in, int method, double *out, uint8_t *out_validity, int mem);
/* GeoSeries::convex_hull (geoseries.rs:23-26): POLYGON array, one closed CCW ring per geometry, in
 * geo's quick_hull vertex order */
int gpl_convex_hull(gpl_ctx *ctx, const gpl_array *in, gpl_array **out);
/* GeoSeries::simplify (geoseries.rs:108-116, impl :240-242): Ramer-Douglas-Peucker with geo 0.27's minimum-size
 * guard (2 points per linestring, 4 per polygon ring); LineString / MultiLineString / Polygon / MultiPolygon;
 * tolerance <= 0 returns the input coordinates.  Outer offsets and validity are shared with the input. */
int gpl_simplify(gpl_ctx *ctx, const gpl_array *in, double tolerance, gpl_array **out);
/* GeoSeries::distance (geoseries.rs:141-146), row-wise 1:1; out[n] f64, out_validity bitmap
 * (may be NULL).  Pairs: any of Point / LineString / Polygon / MultiPoint / MultiLineString / MultiPolygon on
 * either side (geo EuclideanDistance; a Multi* operand is the minimum over its members, f64::MAX when it has none).
 * A row without a single segment where geo needs one (it would panic) is null. */
int gpl_distance(gpl_ctx *ctx, const gpl_array *a, const gpl_array *b, double *out, uint8_t *out_validity, int mem);
/* row-wise intersects (call sites spatial_index.rs:102-123 / geo Intersects); Arrow bitmap out.  Every pair of
 * Point, MultiPoint, LineString, MultiLineString, Polygon, MultiPolygon arrays; null row -> false */
int gpl_intersects(gpl_ctx *ctx, const gpl_array *a, const gpl_array *b, uint8_t *out_bitmap, int mem);
/* row-wise contains of a point: polygons[i] contains points[i] (spatial_index.rs:91-96); `polygons` may also be a
 * (Multi)LineString array (spatial_index.rs:125-135: interior of the line, end points only when closed).
 * Polygon-contains-Polygon (spatial_index.rs:99-101,107-111) is DE-9IM relate in geo and is not provided:
 * GPL_ERR_INVALID_TYPE.  Arrow bitmap out */
int gpl_contains(gpl_ctx *ctx, const gpl_array *polygons, const gpl_array *points, uint8_t *out_bitmap, int mem);
/* secondary trait ops (geoseries.rs:43-83,176-180) */
int gpl_geom_type(gpl_ctx *ctx, const gpl_array *in, int8_t *out, int mem);
int gpl_is_empty(gpl_ctx *ctx, const gpl_array *in, uint8_t *out_bitmap, int mem);
int gpl_is_ring(gpl_ctx *ctx, const gpl_array *in, uint8_t *out_bitmap, int mem);
int gpl_x(gpl_ctx *ctx, const gpl_array *in, double *out, int mem);
int gpl_y(gpl_ctx *ctx, const gpl_array *in, double *out, int mem);
int gpl_exterior(gpl_ctx *ctx, const gpl_array *in, gpl_array **out);
int gpl_explode(gpl_ctx *ctx, const gpl_array *in, gpl_array **out);

/* SpatialIndex envelope queries (spatial_index.rs:206-312 builds one AABB per row, the tests at :361-430 query them
 * with rstar's RTree::locate_in_envelope): out bit i = row i's envelope lies inside the closed box [min,max]
 * (mode 0, `AABB::contains_envelope`) or intersects it (mode 1, closed intervals — the candidate test of the join,
 * :74-76).  Rows without an envelope (null / empty) never match (the reference unwraps and panics on them). */
int gpl_envelope_query(gpl_ctx *ctx, const gpl_array *in, double minx, double miny, double maxx, double maxy, int mode,
                       uint8_t *out_bitmap, int mem);

/* ---------------------------------------------------------------- spatial join ----------- */
/* Replaces SpatialIndex (spatial_index.rs:314-350) for the polygon side of a points-in-polygons
 * join: per-polygon bounding boxes in a uniform grid (candidate generation, closed intervals like
 * rstar's AABB test) plus a per-polygon y-bucketed edge table for the exact test.  Built on the
 * GPU from a POLYGON or MULTIPOLYGON array; keeps a reference to `polygons` (must outlive it). */
int gpl_pip_index_build(gpl_ctx *ctx, const gpl_array *polygons, gpl_pip_index **out);
void gpl_pip_index_free(gpl_pip_index *idx);
int64_t gpl_pip_index_bytes(const gpl_pip_index *idx);
/* diagnostic counters (synchronises the context stream): out8[0] = points the exact kernel re-evaluated since the
 * index was built, [1] = fine raster cells per axis, [2] = log2(fine cells per coarse cell and axis),
 * [3] = raster cells coded "walk", [4] = raster cells coded "inside", [5] = parts without FP32 lists,
 * [6] = index bytes, [7] = coarse cells per axis. */
int gpl_pip_index_stats(gpl_ctx *ctx, const gpl_pip_index *idx, int64_t *out8);
/* diagnostics: microseconds from the start of the index fill kernel to each of its phase boundaries (out12[5..11]) */
int gpl_pip_index_phases(gpl_ctx *ctx, const gpl_pip_index *idx, double *out12);
/* spatial_join(points, polygons, Inner) candidate+exact test (spatial_index.rs:74-143):
 * first_id[p] = lowest polygon row containing point p, or -1; count[p] (may be NULL) = number of
 * containing rows.  points: xy interleaved, n points, in `mem`. */
int gpl_contains_join(gpl_ctx *ctx, const gpl_pip_index *idx, const double *points_xy, int64_t n_points,
                      int32_t *first_id, int32_t *count, int mem);
/* the join and the per-polygon hit counts of config 4: the join (first_id as gpl_contains_join), then a histogram of the
 * id column, both on the context stream: counts[n polygon rows] (u64) += number of points whose first containing row is
 * that polygon (what gpl_join_histogram computes from first_id). */
int gpl_contains_join_counts(gpl_ctx *ctx, const gpl_pip_index *idx, const double *points_xy, int64_t n_points,
                             int32_t *first_id, uint64_t *counts, int mem);
/* same with the points given as a POINT gpl_array (null points -> -1) */
int gpl_contains_join_array(gpl_ctx *ctx, const gpl_pip_index *idx, const gpl_array *points, int32_t *first_id,
                            int32_t *count, int mem);
/* the (lhs_index, rhs_index) pair list the reference emits (spatial_index.rs:139-157), sorted by
 * (point, polygon).  Call with lhs == NULL to get *n_pairs, then with buffers of that size. */
int gpl_contains_join_pairs(gpl_ctx *ctx, const gpl_pip_index *idx, const double *points_xy, int64_t n_points,
                            uint64_t *lhs, uint64_t *rhs, int64_t *n_pairs, int mem);
/* the same pair list for a POINT gpl_array already in HBM (null points match nothing), as a device-resident gpl_pairs
 * (gpl_pairs_count / gpl_pairs_copy / gpl_pairs_free): no host round trip of the point column */
int gpl_contains_join_pairs_array(gpl_ctx *ctx, const gpl_pip_index *idx, const gpl_array *points, gpl_pairs **out);
/* host-resident points streamed through HBM in chunks with H2D / kernel / D2H overlapped on three
 * streams (the end-to-end path: PCIe-bound).  chunk_points = 0 picks a default. */
int gpl_contains_join_host(gpl_ctx *ctx, const gpl_pip_index *idx, const double *points_xy_host, int64_t n_points,
                           int32_t *first_id_host, int64_t chunk_points);
/* per-polygon hit counts: counts[n_polygons] u64 += hits (config 4's all-reduce input) */
int gpl_join_histogram(gpl_ctx *ctx, const int32_t *first_id, int64_t n_points, uint64_t *counts, int64_t n_polygons,
                       int mem);

/* row-wise (Multi)Polygon.contains(Polygon) (the Predicate::Contains arms of spatial_index.rs:99-110; geo's
 * relate(..).is_contains(), DE-9IM [T*****FF*], for valid operands): Arrow bitmap, null rows -> false. */
int gpl_contains_polygon(gpl_ctx *ctx, const gpl_array *a, const gpl_array *b, uint8_t *out_bitmap, int mem);
/* spatial_join(lhs, rhs, predicate) for ANY two geometry columns (spatial_index.rs:37-157): candidates = pairs whose
 * envelopes intersect (closed intervals, :74-76), exact test by the reference's type-pair dispatch (:89-137: Point x
 * (Multi)Polygon / (Multi)LineString in either order -> contains(point) whatever the predicate; (Multi)Polygon x Polygon ->
 * contains or intersects; Polygon x MultiPolygon -> intersects only; every other pair of types -> no match).  The
 * result is the pair list the reference builds at :139-157; its order is unspecified there (tree traversal) and here. */
#define GPL_PREDICATE_INTERSECTS 0
#define GPL_PREDICATE_CONTAINS 1
int gpl_spatial_join(gpl_ctx *ctx, const gpl_array *lhs, const gpl_array *rhs, int predicate, gpl_pairs **out);
int64_t gpl_pairs_count(const gpl_pairs *pairs);
int gpl_pairs_copy(gpl_ctx *ctx, const gpl_pairs *pairs, uint64_t *lhs, uint64_t *rhs, int mem);
void gpl_pairs_free(gpl_pairs *pairs);

/* ---------------------------------------------------------------- synthetic data --------- */
/* device-side generators, bit-identical to geopolars_b200/synth.py (SURVEY.md §8d RNG) */
int gpl_gen_uniform_points(gpl_ctx *ctx, uint64_t stream_id, int64_t first, int64_t n, double scale, double *out_xy_dev);
int gpl_gen_walk_linestrings(gpl_ctx *ctx, uint64_t stream_id, int64_t other_of, int64_t first, int64_t n, int32_t k,
                             double *out_xy_dev, int64_t *out_geom_off_dev);
int gpl_gen_blob_polygons(gpl_ctx *ctx, uint64_t stream_id, int64_t first, int64_t n, int32_t nvert, double *out_xy_dev,
                          int64_t *out_ring_off_dev, int64_t *out_geom_off_dev);

#ifdef __cplusplus
}
#endif
#endif /* GEOPOLARS_B200_H */
