"""CPU tests of the oracle: pinned against the reference's golden vector, its bundled fixtures
(SURVEY.md Appendix A soft values) and the exact-rational referee.  No GPU needed."""
import os

import numpy as np
import pytest

from conftest import rel_close
from geopolars_b200 import GeoArrowArray, GeometryType, synth
from wkbutil import column_to_shapes

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def load(name):
    z = np.load(os.path.join(GOLD, name + ".npz"))
    code, shapes = column_to_shapes(z["offsets"], z["bytes"])
    return GeoArrowArray.from_shapes(GeometryType(code), shapes), z


def test_reference_golden_contains_vector(og, conv):
    """geopolars/src/spatial_index.rs:432-484: exactly rows 1 and 2 of the 9 points are contained;
    (0,10) lies on the boundary and is NOT contained; inner join (2,4), left join (9,4)."""
    z = np.load(os.path.join(GOLD, "contains_golden.npz"))
    sq = z["square"].tolist()
    poly = GeoArrowArray.from_shapes(GeometryType.POLYGON, [[sq + [sq[0]]]])  # polygon![] closes the ring
    first, cnt = og.contains_join(conv(poly), z["points"], use_grid=True)
    assert np.nonzero(first >= 0)[0].tolist() == z["inner_rows"].tolist()
    assert int(cnt.sum()) == int(z["inner_shape"][0]) and len(first) == int(z["left_shape"][0])
    pos = [og.coord_position(conv(poly), 0, *p) for p in z["points"]]
    assert pos == [1, 2, 2, 0, 0, 0, 0, 0, 1]  # B I I O O O O O B
    # unclosed ring given directly: geo's Polygon::new closes it, the oracle emulates that
    open_poly = GeoArrowArray.from_shapes(GeometryType.POLYGON, [[sq]])
    first2, _ = og.contains_join(conv(open_poly), z["points"], use_grid=False)
    assert np.array_equal(first, first2)


# The reference's two SpatialIndex tests (geopolars/src/spatial_index.rs:361-430), restated literally.
AABB_POINTS = [(0.0, 10.0), (1.0, 1.0), (10.0, 0.0), (1.0, -1.0), (0.0, -10.0), (-1.0, -1.0), (-10.0, 0.0), (-1.0, 1.0), (0.0, 10.0)]
AABB_POLYS = [[[(0.0, 0.0), (10.0, 0.0), (10.0, 10.0), (0.0, 10.0), (0.0, 0.0)]],
              [[(0.0, 0.0), (-10.0, 0.0), (-10.0, -10.0), (0.0, -10.0), (0.0, 0.0)]]]
AABB_QUERY = (0.0, 0.0, 20.0, 20.0)


def test_reference_golden_envelope_queries(og, conv):
    """spatial_index_points (:361-393): `locate_in_envelope(AABB [0,0]-[20,20])` over 9 points returns exactly rows
    {0, 1, 2, 8} (closed intervals: (10,0) and (0,10) lie on the box's edge and count).
    spatial_index_polygons (:395-430): over the two squares it returns exactly row 0 — the second square touches the
    query box at the corner (0,0) only and its envelope [-10,-10]-[0,0] is not INSIDE the box (rstar's
    locate_in_envelope is containment, not intersection)."""
    pts = GeoArrowArray.from_shapes(GeometryType.POINT, AABB_POINTS)
    assert np.nonzero(og.envelope_query(conv(pts), AABB_QUERY))[0].tolist() == [0, 1, 2, 8]
    polys = GeoArrowArray.from_shapes(GeometryType.POLYGON, AABB_POLYS)
    assert np.nonzero(og.envelope_query(conv(polys), AABB_QUERY))[0].tolist() == [0]
    # the join's candidate test is intersection with closed intervals (:74-76): the corner-touching square IS a candidate
    assert np.nonzero(og.envelope_query(conv(polys), AABB_QUERY, mode=1))[0].tolist() == [0, 1]
    # NodeEnvelope of a point is the degenerate box (:289); of a polygon its exterior's bounding_rect (:218-226)
    b, v = og.envelope(conv(polys))
    assert v.all() and b.tolist() == [[0.0, 0.0, 10.0, 10.0], [-10.0, -10.0, 0.0, 0.0]]


def test_config1_cities_points(og, conv):
    """BASELINE config 1: centroid(points) == points bit-exactly, area == 0, 202 rows"""
    arr, _ = load("cities")
    assert len(arr) == 202 and arr.type == GeometryType.POINT
    c, v = og.centroid(conv(arr))
    assert v.all() and np.array_equal(c, arr.xy)
    assert np.array_equal(og.area(conv(arr)), np.zeros(202))
    arr2, _ = load("naturalearth_cities")
    assert len(arr2) == 243  # py-geopolars/tests/unit/internals/test_geoseries.py:4-5


def test_fixture_soft_known_values(og, conv):
    """SURVEY.md Appendix A (derived, not reference assertions): areas/centroids/envelopes to 1e-9"""
    nybb, z = load("nybb")
    assert nybb.type == GeometryType.MULTIPOLYGON and len(nybb) == 5
    area = og.area(conv(nybb))
    want_area = [1623821996.706837, 3045213694.3233314, 1937478349.33195, 636471237.9668642, 1186926294.336624]
    assert rel_close(area, want_area, 1e-9)
    assert np.all(np.abs(area / z["Shape_Area"] - 1) < 2e-6)  # the attribute column was computed upstream at lower precision
    cen, v = og.centroid(conv(nybb))
    want_cen = [(941639.4503875433, 150931.9911411282), (1034578.0784064498, 197116.6042299129), (998769.1146889547, 174169.76072686614),
                (993336.964938482, 222451.43672456007), (1021174.7897672353, 249937.9800696837)]
    assert v.all() and rel_close(cen, want_cen, 1e-9)
    env, _ = og.envelope(conv(nybb))
    assert env[0].tolist() == [913175.1090087891, 120121.8812543372, 970570.1481933594, 175708.9620361328]
    low, _ = load("naturalearth_lowres")
    assert len(low) == 177
    a = og.area(conv(low))
    assert rel_close(a[:4], [1.639510995900778, 76.30196359087157, 8.603984207472145, 1712.9952276493766], 1e-9)
    c, _ = og.centroid(conv(low))
    assert rel_close(c[1], (34.752989854755945, -6.25773242850609), 1e-9)


def test_orient2d_sign_against_exact_rational(og):
    from oracle import exact

    rng = np.random.default_rng(1)
    before = og.adapt_calls()
    bad = 0
    for k in range(4000):
        a = rng.uniform(-1e3, 1e3, 2)
        b = a + rng.uniform(-1, 1, 2) * 10.0 ** rng.integers(-6, 4)
        t = rng.uniform(-2, 3)
        c = a + t * (b - a)  # nearly collinear: the fast filter cannot decide
        if k % 3 == 0:
            c = np.nextafter(c, c + rng.normal(size=2))
        if k % 50 == 0:
            c = a.copy()  # exactly degenerate
        got = og.orient2d(a, b, c)
        want = exact.orient_sign(tuple(a), tuple(b), tuple(c))
        bad += ((got > 0) - (got < 0)) != want
    assert bad == 0
    assert og.adapt_calls() > before + 200  # the adaptive stages really ran


def test_contains_and_intersects_against_exact_rational(og, conv):
    from oracle import exact

    xy, ro, go = synth.star_polygons(9, 3)
    polys = GeoArrowArray.polygons(xy, ro, go)
    pts = np.concatenate([synth.uniform_points(1500, scale=30.0), xy[:40], 0.5 * (xy[:40] + xy[1:41])])
    first, cnt = og.contains_join(conv(polys), pts, use_grid=True)
    for i, p in enumerate(pts):
        want = [j for j in range(9) if exact.polygon_contains(tuple(p), [xy[ro[j] : ro[j + 1]].tolist()])]
        assert cnt[i] == len(want) and first[i] == (want[0] if want else -1)
    axy, aoff = synth.walk_linestrings(300, 8, stream=3)
    bxy, boff = synth.walk_linestrings(300, 8, stream=4, other_of=3)
    A, B = GeoArrowArray.linestrings(axy, aoff), GeoArrowArray.linestrings(bxy, boff)
    got = og.intersects_rowwise(conv(A), conv(B))
    want = [exact.linestrings_intersect(axy[aoff[i] : aoff[i + 1]].tolist(), bxy[boff[i] : boff[i + 1]].tolist()) for i in range(300)]
    assert got.tolist() == want and 50 < sum(want) < 250
    d = og.distance_rowwise(conv(A), conv(B))
    assert np.array_equal(d == 0.0, got)


def test_convex_hull_against_exact_rational_and_scipy(og, conv):
    from oracle import exact

    xy, ro, go = synth.blob_polygons(60, 48)
    arr = GeoArrowArray.polygons(xy, ro, go)
    off, hxy = og.convex_hull(conv(arr))
    from scipy.spatial import ConvexHull

    for i in range(60):
        ring = hxy[off[i] : off[i + 1]]
        pts = xy[ro[i] : ro[i + 1]]
        want = exact.convex_hull_vertices(pts.tolist())
        assert np.array_equal(ring[0], ring[-1])
        assert sorted(map(tuple, ring[:-1].tolist())) == sorted(want)
        sp = ConvexHull(pts[:-1])
        assert sorted(map(tuple, pts[:-1][sp.vertices].tolist())) == sorted(want)
    # geo's documented vertex order on the 9-point example (SURVEY.md §8a a4)
    ex = GeoArrowArray.from_shapes(GeometryType.POLYGON, [[[(0, 0), (2, -1), (4, 0), (5, 2), (4, 4), (2, 5), (0, 4), (-1, 2), (0, 0)]]])
    off, hxy = og.convex_hull(conv(ex))
    assert hxy.tolist() == [[0, 0], [2, -1], [4, 0], [5, 2], [4, 4], [2, 5], [0, 4], [-1, 2], [0, 0]]


def test_area_centroid_analytic_shapes(og, conv):
    n = np.arange(3, 40)
    shapes = []
    for k in n:
        th = 2 * np.pi * np.arange(k) / k
        ring = [(3 + 2 * np.cos(t), -1 + 2 * np.sin(t)) for t in th]
        shapes.append([ring + [ring[0]]])
    arr = GeoArrowArray.from_shapes(GeometryType.POLYGON, shapes)
    want = 0.5 * n * 4.0 * np.sin(2 * np.pi / n)
    assert rel_close(og.area(conv(arr)), want, 1e-12)
    c, v = og.centroid(conv(arr))
    assert v.all() and np.allclose(c, [3, -1], atol=1e-12)
    sq, hole = [(0, 0), (4, 0), (4, 4), (0, 4), (0, 0)], [(1, 1), (1, 2), (2, 2), (2, 1), (1, 1)]
    p = GeoArrowArray.from_shapes(GeometryType.POLYGON, [[sq, hole], [sq, sq], [[(0, 0), (2, 2), (4, 4), (0, 0)]], []])
    assert og.area(conv(p)).tolist() == [15.0, 0.0, 0.0, 0.0]
    c, v = og.centroid(conv(p))
    assert v.tolist() == [True, True, True, False]
    assert np.allclose(c[0], [(32 - 1.5) / 15, (32 - 1.5) / 15])
    assert np.allclose(c[1], [2, 2]) and np.allclose(c[2], [2, 2])  # linestring fallbacks


def test_synth_generators_are_bit_reproducible(og):
    p = synth.uniform_points(5000, first=123)
    assert np.array_equal(p, og.gen_uniform_points(2, 123, 5000, 1000.0))
    xy, ro, go = synth.star_polygons(50, 10)
    assert xy.shape == (50 * 65, 2) and np.array_equal(xy[ro[:-1]], xy[ro[1:] - 1])
    a = og.area(og.OGArray(og.POLYGON, xy, geom_off=go, ring_off=ro))
    assert (a > 10).all() and (a < 80).all()


def test_generic_intersects_against_exact_referee_and_symmetry(og, conv):
    """the all-type-pairs restatement of geo's Intersects: polygon pairs and linestring x polygon agree with
    the exact-rational set definition, every type pair is symmetric in its arguments"""
    import shapes
    from oracle import exact
    from geopolars_b200 import GeoArrowArray, GeometryType

    T = dict(zip(shapes.KINDS, [GeometryType.POINT, GeometryType.MULTIPOINT, GeometryType.LINESTRING,
                                GeometryType.MULTILINESTRING, GeometryType.POLYGON, GeometryType.MULTIPOLYGON]))
    rng = np.random.default_rng(1)
    A, B = shapes.random_rows(rng, "polygon", 400), shapes.random_rows(rng, "polygon", 400)
    L = shapes.random_rows(rng, "linestring", 400)
    ga, gb, gl = (GeoArrowArray.from_shapes(T[k], r) for k, r in (("polygon", A), ("polygon", B), ("linestring", L)))
    got = og.intersects_rowwise(conv(ga), conv(gb))
    assert np.array_equal(got, [exact.polygons_intersect(a, b) for a, b in zip(A, B)]) and got.any() and not got.all()
    got = og.intersects_rowwise(conv(gl), conv(gb))
    assert np.array_equal(got, [exact.linestring_intersects_polygon(l, b) for l, b in zip(L, B)]) and got.any()
    for ka in shapes.KINDS:
        for kb in shapes.KINDS:
            rb = shapes.random_rows(rng, kb, 120)
            ra = shapes.plant_touching(rng, ka, shapes.random_rows(rng, ka, 120), kb, rb)
            x, y = GeoArrowArray.from_shapes(T[ka], ra), GeoArrowArray.from_shapes(T[kb], rb)
            ab, ba = og.intersects_rowwise(conv(x), conv(y)), og.intersects_rowwise(conv(y), conv(x))
            assert np.array_equal(ab, ba), (ka, kb)
            assert ab.any(), (ka, kb)


def test_linestring_contains_point_known_answers(og, conv):
    from geopolars_b200 import GeoArrowArray, GeometryType

    L = [[(0, 0), (2, 0), (2, 2), (0, 0)], [(0, 0), (2, 0), (2, 2)], [(0, 0), (2, 0), (2, 2)], [(0, 0), (2, 0), (2, 2)],
         [(1, 1), (1, 1)], [], [(0, 0), (4, 4)], [(0, 0), (4, 4)]]
    P = [(0, 0), (0, 0), (2, 0), (1, 0), (1, 1), (1, 1), (1, 1), (1, 1.5)]
    got = og.contains_rowwise(conv(GeoArrowArray.from_shapes(GeometryType.LINESTRING, L)), np.array(P, float))
    #      closed end  open end  vertex  on segment  degenerate (is_closed)  empty  interior  off
    assert got.tolist() == [True, False, True, True, True, False, True, False]


def test_polygon_linestring_distance_known_answers(og, conv):
    from geopolars_b200 import GeoArrowArray, GeometryType

    sq = [(0, 0), (10, 0), (10, 10), (0, 10), (0, 0)]
    hole = [(2, 2), (2, 8), (8, 8), (8, 2), (2, 2)]
    inner = [(4, 4), (6, 4), (6, 6), (4, 6), (4, 4)]
    right = [(13, 0), (15, 0), (15, 10), (13, 10), (13, 0)]
    diag = [(13, 14), (20, 14), (20, 20), (13, 14)]
    A = GeoArrowArray.from_shapes(GeometryType.POLYGON, [[sq], [sq], [sq, hole], [sq, hole], [sq]])
    B = GeoArrowArray.from_shapes(GeometryType.POLYGON, [[right], [diag], [inner], [right], [inner]])
    d = og.distance_rowwise(conv(A), conv(B))
    assert d.tolist() == [3.0, 5.0, 2.0, 3.0, 0.0]
    assert og.distance_rowwise(conv(B), conv(A)).tolist() == d.tolist()
    L = GeoArrowArray.from_shapes(GeometryType.LINESTRING, [[(13, 5), (20, 5)], [(13, 14), (20, 20)], [(4, 5), (6, 5)], [(5, 5), (12, 5)], [(1, 1), (2, 1)]])
    assert og.distance_rowwise(conv(A), conv(L)).tolist() == [3.0, 5.0, 2.0, 0.0, 0.0]
    assert og.distance_rowwise(conv(L), conv(A)).tolist() == [3.0, 5.0, 2.0, 0.0, 0.0]


def test_simplify_known_answers(og, conv):
    """geo's own documentation / unit-test examples for Simplify (recalled), plus the minimum-size guard"""
    from geopolars_b200 import GeoArrowArray, GeometryType

    ls = [(0.0, 0.0), (5.0, 4.0), (11.0, 5.5), (17.3, 3.2), (27.8, 0.1)]
    arr = GeoArrowArray.from_shapes(GeometryType.LINESTRING, [ls, ls[:2], [], [(1, 1)], [(0, 0), (1, 0.1), (2, 0)]])
    keep = og.simplify_mask(conv(arr), 1.0)
    assert keep[:5].tolist() == [True, True, True, False, True]  # -> (0,0),(5,4),(11,5.5),(27.8,0.1)
    assert keep[5:8].tolist() == [True, True, True] and keep[8:].tolist() == [True, False, True]
    assert og.simplify_mask(conv(arr), 0.0).all() and og.simplify_mask(conv(arr), -1.0).all()
    poly = [(0.0, 0.0), (0.0, 10.0), (5.0, 11.0), (10.0, 10.0), (10.0, 0.0), (0.0, 0.0)]
    tri = [(0.0, 0.0), (4.0, 0.1), (8.0, 0.0), (4.0, 5.0), (0.0, 0.0)]  # 5 coords: culling (4,0.1) leaves 4 -> allowed
    sliver = [(0.0, 0.0), (4.0, 0.1), (8.0, 0.0), (0.0, 0.0)]  # 4 coords: any cull would leave < 4 -> untouched
    parr = GeoArrowArray.from_shapes(GeometryType.POLYGON, [[poly], [tri], [sliver]])
    keep = og.simplify_mask(conv(parr), 2.0)
    assert keep[:6].tolist() == [True, True, False, True, True, True]  # -> (0,0),(0,10),(10,10),(10,0),(0,0)
    assert keep[6:11].tolist() == [True, False, True, True, True]
    assert keep[11:].all()
    with pytest.raises(TypeError):
        og.simplify_mask(conv(GeoArrowArray.points(np.zeros((2, 2)))), 1.0)


def test_geodesic_known_answers(og):
    """pins the oracle's Karney / Vincenty / haversine restatement on published values: the WGS84 quarter
    meridian, a quarter of the equator, Karney (2013) section 7's near-antipodal example and the inverse of
    his direct example; Vincenty agrees with Karney where it converges"""
    g = lambda *a: og.geodesic_distance("geodesic", *a)
    assert abs(g(0, 0, 0, 90) - 10001965.729) < 1e-3
    assert abs(g(0, 0, 90, 0) - 6378137.0 * np.pi / 2) < 1e-8
    assert abs(g(0, 0, 180, 0) - 2 * g(0, 0, 0, 90)) < 1e-8
    assert abs(g(0, -30, 179.8, 29.9) - 19989832.82761) < 1e-5
    assert abs(g(0, 40, 137.84490004377, 41.79331020506) - 1e7) < 1e-5
    assert g(10, 20, 10, 20) == 0.0
    rng = np.random.default_rng(0)
    worst = 0.0
    for _ in range(3000):
        lo1, lo2 = rng.uniform(-180, 180, 2)
        la1, la2 = rng.uniform(-89, 89, 2)
        k, v = g(lo1, la1, lo2, la2), og.geodesic_distance("vincenty", lo1, la1, lo2, la2)
        if not np.isnan(v):
            worst = max(worst, abs(k - v) / k)
        assert abs(k - g(lo2, la2, lo1, la1)) <= 1e-9 * k
    assert worst < 1e-9
    assert np.isnan(og.geodesic_distance("vincenty", 0, 0, 180, 0))  # antipodal: FailedToConvergeError
    # haversine on the mean sphere: a quarter great circle
    assert abs(og.geodesic_distance("haversine", 0, 0, 90, 0) - 6371008.8 * np.pi / 2) < 1e-6


def test_oracle_properties_distance_hull_simplify(og, conv):
    """size-independent properties the domain offers, on the oracle itself: distance is symmetric and zero exactly
    where intersects holds; the hull of a hull is the hull; simplify keeps end points, keeps everything at
    epsilon <= 0 and never keeps MORE points at a larger epsilon on a plain linestring"""
    import shapes
    from geopolars_b200 import GeoArrowArray, GeometryType

    T = dict(zip(shapes.KINDS, [GeometryType.POINT, GeometryType.MULTIPOINT, GeometryType.LINESTRING,
                                GeometryType.MULTILINESTRING, GeometryType.POLYGON, GeometryType.MULTIPOLYGON]))
    rng = np.random.default_rng(21)
    for ka, kb in [("linestring", "linestring"), ("linestring", "polygon"), ("polygon", "polygon"), ("point", "polygon"), ("point", "linestring")]:
        ra, rb = shapes.random_rows(rng, ka, 300, span=14.0), shapes.random_rows(rng, kb, 300, span=14.0)
        a, b = GeoArrowArray.from_shapes(T[ka], ra), GeoArrowArray.from_shapes(T[kb], rb)
        dab, dba = og.distance_rowwise(conv(a), conv(b)), og.distance_rowwise(conv(b), conv(a))
        ok = ~np.isnan(dab)
        assert np.array_equal(np.isnan(dab), np.isnan(dba)) and rel_close(dab[ok], dba[ok], 1e-12)
        assert (dab[ok] >= 0).all()
        if ka != "point":  # Point x LineString distance uses geo-types' epsilon-based containment, not Intersects
            hit = og.intersects_rowwise(conv(a), conv(b))
            assert np.array_equal(dab[ok] == 0.0, hit[ok])
    # hull idempotence (vertex order included)
    polys = GeoArrowArray.from_shapes(GeometryType.POLYGON, shapes.random_rows(rng, "polygon", 300))
    off1, xy1 = og.convex_hull(conv(polys))
    hulls = GeoArrowArray.polygons(xy1, off1, np.arange(len(polys) + 1))
    off2, xy2 = og.convex_hull(conv(hulls))
    assert np.array_equal(off1, off2) and np.array_equal(xy1, xy2)
    # simplify
    lens = rng.integers(2, 60, 400)
    off = np.concatenate([[0], np.cumsum(lens)])
    xy = np.cumsum(rng.normal(0, 1, (off[-1], 2)), axis=0)
    ls = GeoArrowArray.linestrings(xy, off)
    prev = og.simplify_mask(conv(ls), 0.0)
    assert prev.all()
    for eps in (0.1, 0.5, 2.0, 10.0):
        keep = og.simplify_mask(conv(ls), eps)
        assert keep[off[:-1]].all() and keep[off[1:] - 1].all()  # end points always survive
        assert keep.sum() <= prev.sum()
        prev = keep


def test_polygon_contains_polygon_oracle_vs_exact_referee(og, conv):
    """(Multi)Polygon.contains(Polygon) (spatial_index.rs:99-110; geo relate().is_contains(), recalled — parity unpinned by
    the reference): the oracle's orientation-sign procedure against the exact-rational arrangement form of the same
    definition (closure(A) contains B, interiors meet), on crafted touching / equal / hole / notch cases and random valid
    lattice polygons"""
    import shapes
    from oracle import exact

    rng = np.random.default_rng(5)
    A, B = shapes.contains_cases(rng, 250)
    ga, gb = GeoArrowArray.from_shapes(GeometryType.POLYGON, A), GeoArrowArray.from_shapes(GeometryType.POLYGON, B)
    got = og.contains_polygon_rowwise(conv(ga), conv(gb), threads=0)
    ref = np.array([exact.region_contains_polygon([a], b) for a, b in zip(A, B)])
    assert np.array_equal(got, ref)
    assert got[:18].tolist() == [True, True, True, False, False, False, True, True, True, True, True, True, False, False, False, True, True, True]
    assert 40 < got.sum() < len(got) - 40
    MA, MB = shapes.multi_contains_cases()
    ma, mb = GeoArrowArray.from_shapes(GeometryType.MULTIPOLYGON, MA), GeoArrowArray.from_shapes(GeometryType.POLYGON, MB)
    gm = og.contains_polygon_rowwise(conv(ma), conv(mb))
    assert gm.tolist() == [exact.region_contains_polygon(a, b) for a, b in zip(MA, MB)] == [True, True, False, True, True, False, False]


def test_multi_distance_is_the_minimum_over_members(og, conv):
    """GeoSeries::distance with Multi* operands (geo's impl for iterable geometries, recalled): the minimum over the
    members, f64::MAX for an empty collection; checked against a brute-force segment scan on the reference's nybb rows"""
    arr, _ = load("nybb")
    cw, cv = og.centroid(conv(arr))
    pts = GeoArrowArray.points(np.roll(cw, 1, axis=0))
    d = og.distance_rowwise(conv(arr), conv(pts), threads=0)
    for i in range(len(arr)):
        p, best = pts.xy[i], np.inf
        for part in range(arr.geom_off[i], arr.geom_off[i + 1]):
            for r in range(arr.part_off[part], arr.part_off[part + 1]):
                c = arr.xy[arr.ring_off[r] : arr.ring_off[r + 1]]
                a, ab = c[:-1], c[1:] - c[:-1]
                L = (ab * ab).sum(1)
                t = np.clip(((p - a) * ab).sum(1) / np.where(L > 0, L, 1), 0, 1)
                best = min(best, np.hypot(*(p - (a + t[:, None] * ab)).T).min())
        assert abs(best - d[i]) <= 1e-9 * best
    empty = GeoArrowArray.from_shapes(GeometryType.MULTIPOINT, [[], [(1.0, 1.0), (4.0, 5.0)]])
    q = GeoArrowArray.points(np.array([[0.0, 0.0], [1.0, 1.0]]))
    assert og.distance_rowwise(conv(empty), conv(q)).tolist() == [1.7976931348623157e308, 0.0]


def test_area_centroid_length_envelope_against_exact_rational(og, conv):
    """random polygons with holes and MultiPolygons at three magnitudes: the shoelace area, the area-weighted centroid, the ring
    length and the envelope evaluated in exact rational arithmetic on the SAME doubles, against the oracle's f64 loops
    (geo's `Area`, `Centroid`, `EuclideanLength`, `BoundingRect` restated) — an independent formulation, 1e-12 relative"""
    from fractions import Fraction as F

    rng = np.random.default_rng(21)

    def ring(cx, cy, r0, r1, n, sc):
        th = np.sort(rng.uniform(0, 2 * np.pi, n))
        rr = rng.uniform(r0, r1, n)
        pts = [(float(sc * (cx + rr[i] * np.cos(th[i]))), float(sc * (cy + rr[i] * np.sin(th[i])))) for i in range(n)]
        return pts + [pts[0]]

    def shoelace(r):  # signed area (exact) and first moments of a closed ring
        a = mx = my = F(0)
        for (x0, y0), (x1, y1) in zip(r[:-1], r[1:]):
            x0, y0, x1, y1 = F(x0), F(y0), F(x1), F(y1)
            c = x0 * y1 - x1 * y0
            a += c
            mx += (x0 + x1) * c
            my += (y0 + y1) * c
        return a / 2, mx / 6, my / 6

    polys, multis = [], []
    for k in range(60):
        sc, off = [(1.0, 0.0), (1e-3, 5.0), (250.0, 4000.0)][k % 3]
        ext = ring(off, -off, 4.0, 9.0, int(rng.integers(5, 40)), sc)
        holes = [ring(off + dx, -off + dy, 0.3, 0.9, int(rng.integers(3, 9)), sc) for dx, dy in [(-1.5, 0.0), (1.5, 0.5)][: k % 3]]
        polys.append([ext] + holes)
    for k in range(20):
        multis.append([[ring(10.0 * j, 3.0 * k, 1.0, 2.5, int(rng.integers(4, 20)), 1.0)] + ([ring(10.0 * j, 3.0 * k, 0.2, 0.6, 5, 1.0)] if j % 2 else []) for j in range(1 + k % 3)])

    def exact_poly(rings):
        A = MX = MY = F(0)
        for i, r in enumerate(rings):
            a, mx, my = shoelace(r)
            s = 1 if a >= 0 else -1  # orientation-independent: |exterior| - sum |holes|
            w = 1 if i == 0 else -1
            A += w * s * a
            MX += w * s * mx
            MY += w * s * my
        return A, MX, MY

    for typ, shapes in ((GeometryType.POLYGON, polys), (GeometryType.MULTIPOLYGON, multis)):
        arr = GeoArrowArray.from_shapes(typ, shapes)
        area = og.area(conv(arr))
        cen, valid = og.centroid(conv(arr))
        length = og.euclidean_length(conv(arr))
        env, ev = og.envelope(conv(arr))
        assert valid.all() and ev.all()
        for i, shp in enumerate(shapes):
            parts = [shp] if typ == GeometryType.POLYGON else shp
            A = MX = MY = F(0)
            for rings in parts:
                a, mx, my = exact_poly(rings)
                A, MX, MY = A + a, MX + mx, MY + my
            assert abs(area[i] - float(A)) <= 1e-12 * abs(float(A))
            cx, cy = float(MX / A), float(MY / A)
            scale = max(abs(cx), abs(cy), 1e-300)
            assert abs(cen[i, 0] - cx) <= 1e-9 * scale and abs(cen[i, 1] - cy) <= 1e-9 * scale
            coords = [c for rings in parts for r in rings for c in r]
            xs, ys = [c[0] for c in coords], [c[1] for c in coords]
            ext_coords = [c for rings in parts for c in rings[0]]
            assert env[i].tolist() == [min(c[0] for c in ext_coords), min(c[1] for c in ext_coords), max(c[0] for c in ext_coords), max(c[1] for c in ext_coords)] \
                or env[i].tolist() == [min(xs), min(ys), max(xs), max(ys)]
            # euclidean_length of an areal row = the length of its exterior ring(s) (the reference maps polygons to their exterior,
            # geoseries.rs:35-41); correctly rounded sum of hypots as the yardstick
            import math

            want_len = math.fsum(math.hypot(b[0] - a[0], b[1] - a[1]) for rings in parts for a, b in zip(rings[0][:-1], rings[0][1:]))
            assert abs(length[i] - want_len) <= 1e-12 * want_len


def test_native_oracle_cache_is_private(tmp_path, monkeypatch):
    """the -march=native oracle is cached under the shared temporary directory: a cache directory that is a link, or that
    others can enter, is refused instead of loading a library planted there; a private one is built once and reused"""
    import tempfile

    from oracle import oracle

    monkeypatch.setattr(tempfile, "tempdir", str(tmp_path))
    base = tmp_path / f"geo_oracle-{os.getuid()}"
    planted = tmp_path / "planted"
    (planted / "sig").mkdir(parents=True)
    (planted / "sig" / "flags.txt").write_text("planted")
    planted.chmod(0o700)
    base.symlink_to(planted)
    with pytest.raises(PermissionError):
        oracle._build_native("sig")
    base.unlink()
    planted.chmod(0o755)
    planted.rename(base)
    with pytest.raises(PermissionError):
        oracle._build_native("sig")
    base.chmod(0o700)
    built = oracle._build_native("fresh")
    assert built == str(base / "fresh") and (base / "fresh" / "libgeo_oracle.so").is_file()
    assert "-march=native" in (base / "fresh" / "flags.txt").read_text()
    assert sorted(p.name for p in base.iterdir()) == ["fresh", "sig"]  # no half-built directory left behind
    assert oracle._build_native("fresh") == built
