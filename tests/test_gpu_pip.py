"""Parity of the CUDA points-in-polygons join against the oracle (bit-exact: index outputs).
Reference semantics: geopolars/src/spatial_index.rs:89-96 (`poly.contains(point)`), golden vector
:432-484."""
import numpy as np
import pytest

from geopolars_b200 import GeoArrowArray, GeometryType, synth

pytestmark = pytest.mark.gpu


def test_golden_vector_square(ctx):
    """the reference's only numeric pin: 9 points x square -> exactly (1,1) and (10,1) are contained"""
    from geopolars_b200.engine import PipIndex

    sq = GeoArrowArray.from_shapes(GeometryType.POLYGON, [[[(0, 0), (20, 0), (20, 20), (0, 20), (0, 0)]]])
    pts = np.array([(0, 10), (1, 1), (10, 1), (1, -1), (0, -10), (-1, -1), (-10, 0), (-1, 1), (0, 10)], float)
    idx = PipIndex(ctx.upload(sq))
    first, cnt = idx.query(pts, with_count=True)
    assert first.tolist() == [-1, 0, 0, -1, -1, -1, -1, -1, -1]
    assert cnt.tolist() == [0, 1, 1, 0, 0, 0, 0, 0, 0]
    lhs, rhs = idx.pairs(pts)
    assert lhs.tolist() == [1, 2] and rhs.tolist() == [0, 0]  # inner join shape (2, ..) as in spatial_join_test


def test_unclosed_ring_is_closed_like_polygon_new(ctx):
    from geopolars_b200.engine import PipIndex

    sq = GeoArrowArray.from_shapes(GeometryType.POLYGON, [[[(0, 0), (20, 0), (20, 20), (0, 20)]]])
    pts = np.array([(0, 10), (1, 1), (10, 1), (19.5, 19.5), (20, 20), (0, 0), (-1, 5)], float)
    first = PipIndex(ctx.upload(sq)).query(pts)
    assert first.tolist() == [-1, 0, 0, 0, -1, -1, -1]


@pytest.mark.parametrize("m,grid,n", [(100, 10, 200_000), (2500, 50, 300_000)])
def test_star_polygons_vs_oracle(ctx, og, conv, m, grid, n):
    from geopolars_b200.engine import PipIndex

    xy, ro, go = synth.star_polygons(m, grid)
    polys = GeoArrowArray.polygons(xy, ro, go)
    pts = synth.uniform_points(n, scale=grid * 10.0)
    # adversarial additions: polygon vertices, edge midpoints, bbox corners, points far outside
    extra = np.concatenate([xy[:500], 0.5 * (xy[:500] + xy[1:501]), np.array([[-5.0, -5.0], [1e9, 1e9], [np.nan, 1.0]])])
    pts = np.concatenate([pts, extra])
    want_first, want_cnt = og.contains_join(conv(polys), pts, use_grid=True, threads=0)
    idx = PipIndex(ctx.upload(polys))
    first, cnt = idx.query(pts, with_count=True)
    assert np.array_equal(first, want_first)
    assert np.array_equal(cnt, want_cnt)
    lhs, rhs = idx.pairs(pts)
    hit = np.nonzero(want_first >= 0)[0]
    assert np.array_equal(lhs, hit.astype(np.uint64))
    assert np.array_equal(rhs, want_first[hit].astype(np.uint64))


def _holes_and_multis():
    # polygon with a hole, overlapping polygons, a multipolygon with two parts, a null row, an empty polygon
    outer = [(0, 0), (10, 0), (10, 10), (0, 10), (0, 0)]
    hole = [(4, 4), (4, 6), (6, 6), (6, 4), (4, 4)]
    tri = [(5, 5), (15, 5), (10, 15), (5, 5)]
    far1 = [(20, 20), (22, 20), (22, 22), (20, 22), (20, 20)]
    far2 = [(21, 21), (25, 21), (25, 25), (21, 25), (21, 21)]
    return [[[outer, hole]], [[tri]], [[far1], [far2]], None, []]


def test_holes_multipolygons_overlaps_nulls(ctx, og, conv):
    from geopolars_b200.engine import PipIndex

    polys = GeoArrowArray.from_shapes(GeometryType.MULTIPOLYGON, _holes_and_multis())
    g = np.linspace(-1, 26, 109)
    gx, gy = np.meshgrid(g, g)
    pts = np.stack([gx.ravel(), gy.ravel()], 1)  # lattice hits vertices, edges, hole borders exactly
    want_first, want_cnt = og.contains_join(conv(polys), pts, use_grid=False, threads=0)
    idx = PipIndex(ctx.upload(polys))
    first, cnt = idx.query(pts, with_count=True)
    assert np.array_equal(first, want_first)
    assert np.array_equal(cnt, want_cnt)
    assert cnt.max() == 2  # the overlap region really is exercised
    lhs, rhs = idx.pairs(pts)
    assert len(lhs) == int(want_cnt.sum())
    # pair list is sorted by (point, polygon) and consistent with per-point counts
    assert np.all(np.diff(lhs.astype(np.int64)) >= 0)
    assert np.array_equal(np.bincount(lhs.astype(np.int64), minlength=len(pts)), want_cnt)


def test_near_degenerate_points_use_exact_predicate(ctx, og, conv):
    """points a few ulps off long edges: the fast orient2d filter cannot decide, the adaptive stage must"""
    from geopolars_b200.engine import PipIndex

    big = [(1e6 + 0.1, 2e6 + 0.3), (1e6 + 1000.7, 2e6 + 500.9), (1e6 + 300.2, 2e6 + 900.4), (1e6 + 0.1, 2e6 + 0.3)]
    polys = GeoArrowArray.from_shapes(GeometryType.POLYGON, [[big]])
    a, b = np.array(big[0]), np.array(big[1])
    t = np.linspace(0.01, 0.99, 4000)
    on = a[None, :] + t[:, None] * (b - a)[None, :]
    pts = np.concatenate([on, np.nextafter(on, 1e9), np.nextafter(on, -1e9)])
    before = og.adapt_calls()
    want_first, want_cnt = og.contains_join(conv(polys), pts, use_grid=False, threads=1)
    assert og.adapt_calls() > before  # the oracle needed the adaptive stage, so the case is real
    first, cnt = PipIndex(ctx.upload(polys)).query(pts, with_count=True)
    assert np.array_equal(first, want_first)
    assert 0 < (want_first >= 0).sum() < len(pts)


def test_empty_inputs(ctx):
    from geopolars_b200.engine import PipIndex

    polys = GeoArrowArray.polygons(np.zeros((0, 2)), np.zeros(1, np.int64), np.zeros(1, np.int64))
    idx = PipIndex(ctx.upload(polys))
    assert idx.query(np.array([[1.0, 1.0]])).tolist() == [-1]
    xy, ro, go = synth.star_polygons(4, 2)
    idx2 = PipIndex(ctx.upload(GeoArrowArray.polygons(xy, ro, go)))
    assert idx2.query(np.zeros((0, 2))).shape == (0,)


def test_large_rings_overlapping_boxes_and_deferred_overflow(ctx, og, conv):
    """POLYGON rows that are not eligible for the FP32 fast table (buckets longer than 63 edges), cells with
    several candidates (overlapping boxes), and a point set made almost entirely of boundary points so that
    the deferred list overflows and the exact kernel falls back to scanning the id column."""
    from geopolars_b200.engine import PipIndex

    k = np.arange(3000)
    th = 2 * np.pi * k / 3000
    r = 10 + 3 * np.sin(40 * th)
    big = np.stack([r * np.cos(th), r * np.sin(th)], 1)
    big = np.concatenate([big, big[:1]])
    sq = lambda x, y, s: [(x, y), (x + s, y), (x + s, y + s), (x, y + s), (x, y)]
    shapes = [[big.tolist()], [sq(-3, -3, 6)], [sq(-1, -1, 9)], [sq(20, 20, 1)]]
    polys = GeoArrowArray.from_shapes(GeometryType.POLYGON, shapes)
    pts = np.concatenate([synth.uniform_points(150_000, scale=30.0) - 14.0, big[:-1], 0.5 * (big[:-1] + big[1:])])
    want_first, want_cnt = og.contains_join(conv(polys), pts, use_grid=True, threads=0)
    idx = PipIndex(ctx.upload(polys))
    first, cnt = idx.query(pts, with_count=True)
    assert np.array_equal(first, want_first) and np.array_equal(cnt, want_cnt)
    assert cnt.max() == 3
    # every point on a boundary: all deferred (list capacity is max(n/16, 65536) -> overflow -> scan path)
    xy, ro, go = synth.star_polygons(400, 20)
    stars = GeoArrowArray.polygons(xy, ro, go)
    t = np.linspace(0.0, 1.0, 41)[None, :, None]
    on_edges = (xy[:-1, None, :] * (1 - t) + xy[1:, None, :] * t).reshape(-1, 2)[:1_200_000]
    wf, wc = og.contains_join(conv(stars), on_edges, use_grid=True, threads=0)
    f2, c2 = PipIndex(ctx.upload(stars)).query(on_edges, with_count=True)
    assert np.array_equal(f2, wf) and np.array_equal(c2, wc)


def test_empty_polygon_next_to_polygon_with_hole(ctx, og, conv):
    """ring count == polygon count although a hole exists: the hole table must still be built"""
    from geopolars_b200.engine import PipIndex

    sq = [(0, 0), (10, 0), (10, 10), (0, 10), (0, 0)]
    hole = [(4, 4), (4, 6), (6, 6), (6, 4), (4, 4)]
    polys = GeoArrowArray.from_shapes(GeometryType.POLYGON, [[], [sq, hole]])
    assert polys.n_rings == len(polys) == 2
    g = np.linspace(-1, 11, 49)
    pts = np.stack(np.meshgrid(g, g), -1).reshape(-1, 2)
    want, wc = og.contains_join(conv(polys), pts, use_grid=False)
    first, cnt = PipIndex(ctx.upload(polys)).query(pts, with_count=True)
    assert np.array_equal(first, want) and np.array_equal(cnt, wc) and (want == 1).any() and (want == -1).any()


@pytest.mark.parametrize("scale,offset", [(1e-20, 0.0), (1e-3, 0.0), (1.0, 1e6), (1e19, 0.0), (1e-12, 7.0), (1e-25, 0.0), (1e25, 0.0)])
def test_part_extents_from_tiny_to_huge(ctx, og, conv, scale, offset):
    """FP32 filter scale guard (VERDICT r1): parts whose extent is far below / above the float range of R^2 must not
    be decided by the float filter; nybb-like parts (small extent at a 1e6 offset) must survive the float origin.
    Points: random, every vertex, edge midpoints, and the neighbours of both one ulp away."""
    from geopolars_b200.engine import PipIndex

    xy, ro, go = synth.star_polygons(100, 10)
    xy = xy * scale + offset
    polys = GeoArrowArray.polygons(xy, ro, go)
    pts = synth.uniform_points(20_000, scale=100.0) * scale + offset
    mid = 0.5 * (xy[:-1] + xy[1:])
    spec = np.concatenate([xy, mid])
    pts = np.concatenate([pts, spec, np.nextafter(spec, np.inf), np.nextafter(spec, -np.inf)])
    want_first, want_cnt = og.contains_join(conv(polys), pts, use_grid=False, threads=0)
    idx = PipIndex(ctx.upload(polys))
    first, cnt = idx.query(pts, with_count=True)
    assert np.array_equal(first, want_first) and np.array_equal(cnt, want_cnt)
    assert 0 < (want_first >= 0).sum() < len(pts)
    st = idx.stats()
    if scale in (1e-20, 1e-25, 1e19, 1e25):
        assert st["parts_not_fast"] == 100  # outside 2^-50 <= R <= 2^50: no FP32 lists, the f64 walk decides
    else:
        assert st["parts_not_fast"] == 0


def test_raster_cell_boundaries_and_census(ctx, og, conv):
    """the 2-bit raster: points ON the fine-cell lattice (and one ulp either side), its census on the config-2 shapes,
    and the deferred counter (exact re-evaluations) being small but non-zero on random points"""
    from geopolars_b200.engine import PipIndex

    xy, ro, go = synth.star_polygons(400, 20)
    polys = GeoArrowArray.polygons(xy, ro, go)
    idx = PipIndex(ctx.upload(polys))
    st = idx.stats()
    fg = st["fine_cells_per_axis"]
    assert fg == st["coarse_cells_per_axis"] << st["raster_log2"] and st["raster_log2"] >= 4
    total = fg * fg
    walk, inside = st["raster_walk_cells"], st["raster_inside_cells"]
    assert 0.03 < walk / total < 0.35, (walk, total)      # ring cells: the edge walk is the exception
    assert 0.15 < inside / total < 0.60, (inside, total)  # ~37 % of the plane is inside a star
    # lattice of fine-cell corners over a part of the grid, +- 1 ulp
    x0, y0 = xy[:, 0].min(), xy[:, 1].min()
    w, h = xy[:, 0].max() - x0, xy[:, 1].max() - y0
    k = np.arange(0, fg + 1, 7, dtype=np.float64)
    gx, gy = np.meshgrid(x0 + k / fg * w, y0 + (k[:200] + 3) / fg * h)
    lat = np.stack([gx.ravel(), gy.ravel()], 1)
    pts = np.concatenate([lat, np.nextafter(lat, np.inf), np.nextafter(lat, -np.inf), synth.uniform_points(400_000, scale=200.0)])
    want_first, want_cnt = og.contains_join(conv(polys), pts, use_grid=True, threads=0)
    first, cnt = idx.query(pts, with_count=True)
    assert np.array_equal(first, want_first) and np.array_equal(cnt, want_cnt)
    d = idx.stats()["deferred"]
    assert 0 < d < 0.01 * len(pts), d


def test_nested_and_covering_polygons(ctx, og, conv):
    """raster codes compose: a cell inside two candidates, inside a third-or-later candidate, or inside one polygon and
    on the ring of another must all take the walk; one giant polygon over many small ones exercises long candidate lists"""
    from geopolars_b200.engine import PipIndex

    sq = lambda x, y, s: [(x, y), (x + s, y), (x + s, y + s), (x, y + s), (x, y)]
    shapes = [[sq(0, 0, 100)], [sq(10, 10, 50)], [sq(20, 20, 20)], [sq(25, 25, 5)], [sq(70, 70, 10), sq(72, 72, 3)]]
    xy, ro, go = synth.star_polygons(64, 8, cell=12.5)
    stars = GeoArrowArray.polygons(xy, ro, go)
    for i in range(64):
        shapes.append([xy[ro[i]:ro[i + 1]].tolist()])
    polys = GeoArrowArray.from_shapes(GeometryType.POLYGON, shapes)
    g = np.linspace(-2, 102, 209)
    lat = np.stack(np.meshgrid(g, g), -1).reshape(-1, 2)
    pts = np.concatenate([lat, synth.uniform_points(300_000, scale=104.0) - 2.0])
    want_first, want_cnt = og.contains_join(conv(polys), pts, use_grid=False, threads=0)
    idx = PipIndex(ctx.upload(polys))
    first, cnt = idx.query(pts, with_count=True)
    assert np.array_equal(first, want_first) and np.array_equal(cnt, want_cnt)
    assert want_cnt.max() >= 4
    only_first = idx.query(pts)
    assert np.array_equal(only_first, want_first)
    lhs, rhs = idx.pairs(pts[:50_000])
    assert len(lhs) == int(want_cnt[:50_000].sum())
    # the same shapes as MULTIPOLYGON rows (parts of one row counted once)
    multi = GeoArrowArray.from_shapes(GeometryType.MULTIPOLYGON, [[s] for s in shapes[:5]] + [[shapes[5 + i], shapes[6 + i]] for i in range(0, 62, 2)])
    wf, wc = og.contains_join(conv(multi), pts, use_grid=False, threads=0)
    f2, c2 = PipIndex(ctx.upload(multi)).query(pts, with_count=True)
    assert np.array_equal(f2, wf) and np.array_equal(c2, wc)


def test_unaligned_point_and_id_columns(ctx, og, conv):
    """device columns that are only 16- / 4-byte aligned (slices) take the scalar load/store path of the streaming kernel"""
    import torch

    from geopolars_b200.engine import PipIndex

    xy, ro, go = synth.star_polygons(100, 10)
    polys = GeoArrowArray.polygons(xy, ro, go)
    n = 100_003
    pts = synth.uniform_points(n + 1, scale=100.0)
    want, _ = og.contains_join(conv(polys), pts[1:], use_grid=True, threads=0)
    idx = PipIndex(ctx.upload(polys))
    d_pts = torch.from_numpy(pts).cuda()
    d_ids = torch.full((n + 3,), -7, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    idx.query_device(d_pts.data_ptr() + 16, n, d_ids.data_ptr() + 4)  # points from row 1, ids from element 1
    ctx.synchronize()
    got = d_ids.cpu().numpy()
    assert got[0] == -7 and got[n + 1] == -7 and got[n + 2] == -7
    assert np.array_equal(got[1:n + 1], want)


def test_reference_golden_envelope_queries_gpu(ctx, og, conv):
    """spatial_index.rs:361-430 on the device: points -> rows {0,1,2,8}; the two squares -> row {0}; candidates -> {0,1}"""
    from geopolars_b200 import engine as E
    from test_oracle_cpu import AABB_POINTS, AABB_POLYS, AABB_QUERY

    pts = GeoArrowArray.from_shapes(GeometryType.POINT, AABB_POINTS)
    polys = GeoArrowArray.from_shapes(GeometryType.POLYGON, AABB_POLYS)
    d_pts, d_polys = ctx.upload(pts), ctx.upload(polys)
    assert np.nonzero(E.envelope_query(d_pts, AABB_QUERY))[0].tolist() == [0, 1, 2, 8]
    assert np.nonzero(E.envelope_query(d_polys, AABB_QUERY))[0].tolist() == [0]
    assert np.nonzero(E.envelope_query(d_polys, AABB_QUERY, intersecting=True))[0].tolist() == [0, 1]
    # the grid candidate stage of the join agrees with the AABB intersection test: every point whose degenerate box meets a
    # polygon's envelope reaches the exact test (here: candidates of square 0 are the points inside its closed envelope)
    idx = E.PipIndex(d_polys)
    first, cnt = idx.query(np.asarray(AABB_POINTS), with_count=True)
    assert first.tolist() == [-1, 0, -1, -1, -1, 1, -1, -1, -1]  # (1,1) inside square 0, (-1,-1) inside square 1; edges excluded
    # random columns against the oracle, both modes, incl. null and empty rows
    xy, ro, go = synth.star_polygons(400, 20)
    stars = GeoArrowArray.polygons(xy, ro, go)
    d = ctx.upload(stars)
    for box in [(0.0, 0.0, 200.0, 200.0), (33.0, 41.5, 120.25, 77.0), (1e3, 1e3, 2e3, 2e3)]:
        for mode in (0, 1):
            assert np.array_equal(E.envelope_query(d, box, intersecting=bool(mode)), og.envelope_query(conv(stars), box, mode))
    mixed = GeoArrowArray.from_shapes(GeometryType.MULTIPOLYGON, _holes_and_multis())
    for mode in (0, 1):
        assert np.array_equal(E.envelope_query(ctx.upload(mixed), (-1.0, -1.0, 16.0, 16.0), intersecting=bool(mode)),
                              og.envelope_query(conv(mixed), (-1.0, -1.0, 16.0, 16.0), mode))


def test_join_counts(ctx, og, conv):
    """gpl_contains_join_counts: ids + per-polygon hit counts, a histogram of the id column after the join (bins in shared
    memory up to 49152 polygon rows, global atomics beyond); boundary points (deferred to the exact kernel) must be counted
    exactly once"""
    from geopolars_b200.engine import PipIndex

    for m, grid in ((400, 20), (16_900, 130), (50_000, 224)):
        xy, ro, go = synth.star_polygons(m, grid)
        polys = GeoArrowArray.polygons(xy, ro, go)
        pts = np.concatenate([synth.uniform_points(300_000, scale=grid * 10.0), xy[:2000], 0.5 * (xy[:2000] + xy[1:2001])])
        want, _ = og.contains_join(conv(polys), pts, use_grid=True, threads=0)
        idx = PipIndex(ctx.upload(polys))
        first, counts = idx.query_counts(pts)
        assert np.array_equal(first, want)
        assert np.array_equal(counts.astype(np.int64), np.bincount(want[want >= 0], minlength=m))
        f2, c2 = idx.query_counts(pts)  # counts accumulate per call from a zeroed column: same result again
        assert np.array_equal(f2, want) and np.array_equal(c2, counts)


def test_kernel_timing_brackets_every_stream_launch(ctx):
    """gpl_ctx_kernel_timing (bench.py's roofline denominator): one event pair per k_pip_stream launch, read once"""
    from geopolars_b200.engine import PipIndex

    xy, ro, go = synth.star_polygons(100, 10)
    idx = PipIndex(ctx.upload(GeoArrowArray.polygons(xy, ro, go)))
    pts = synth.uniform_points(500_000, scale=100.0)
    base = idx.query(pts)
    assert ctx.kernel_timing_read() == (0.0, 0)  # off: nothing recorded
    ctx.kernel_timing(True)
    for _ in range(3):
        assert np.array_equal(idx.query(pts), base)
    ms, n = ctx.kernel_timing_read()
    assert n == 3 and 0.0 < ms < 100.0
    assert ctx.kernel_timing_read() == (0.0, 0)  # a read consumes the pairs
    ctx.kernel_timing(False)
    idx.query(pts)
    assert ctx.kernel_timing_read() == (0.0, 0)
