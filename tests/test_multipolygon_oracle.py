"""CPU tests of the contract for outlines with holes and several parts (oracle/multipolygon_ref.py) and of the host
side of the polygon layout: known answers, the XOR of the single-ring decisions, bit-exact reduction to one ring,
``pack_polygons`` on nested lists and on shapely-like stand-ins, malformed offsets and the C-ABI argument checks."""
from types import SimpleNamespace

import numpy as np
import pytest

from oracle.buffered_geometry_ref import points_in_buffered_polygons_ref, polygon_props_ref
from oracle.geometry_ref import points_in_polygons_ref
from oracle.multipolygon_ref import check_layout, multipolygon_props_ref, points_in_multipolygons_ref
from segger_b200.geometry import Outlines, PackedPolygons, pack_polygons, pack_rings


def _sq(x0, y0, x1, y1):
    return np.array([[x0, y0], [x1, y0], [x1, y1], [x0, y1]], dtype=np.float64)


def _ngon(c, r, n, phase=0.0):
    ang = np.linspace(0, 2 * np.pi, n, endpoint=False) + phase
    return np.stack([c[0] + r * np.cos(ang), c[1] + r * np.sin(ang)], 1)


def _pairs(pts, geoms, dist=None):
    layout = pack_polygons(geoms)
    return set(map(tuple, points_in_multipolygons_ref(pts, *layout, dist=dist).T))


HOLED = [[_sq(0, 0, 4, 4), _sq(1, 1, 3, 3)]]                   # one part: a square with a square hole


def test_square_with_square_hole():
    pts = np.array([[0.5, 0.5], [2.0, 2.0], [2.0, 1.2], [3.5, 2.0], [4.2, 2.0], [2.0, 1.35]])
    assert _pairs(pts, [HOLED]) == {(0, 0), (3, 0)}            # the hole is out
    # grown by 0.3: points of the hole within 0.3 of its rim come in, and so does the rim's outside within 0.3
    assert _pairs(pts, [HOLED], [0.3]) == {(0, 0), (2, 0), (3, 0), (4, 0)}
    # shrunk by 0.4: (3.5, 2) is 0.5 from both rims and stays; (0.5, 0.5) is 0.5 from the outer rim and stays
    assert _pairs(pts, [HOLED], [-0.4]) == {(0, 0), (3, 0)}
    assert _pairs(pts, [HOLED], [-0.5]) == set()               # exactly |d| from a rim: out (strict)


def test_two_disjoint_squares_are_one_geometry():
    geom = [[_sq(0, 0, 1, 1)], [_sq(5, 5, 6, 6)]]              # two parts
    pts = np.array([[0.5, 0.5], [5.5, 5.5], [3.0, 3.0], [5.5, 0.5]])
    got = points_in_multipolygons_ref(pts, *pack_polygons([geom, [[_sq(0, 0, 6, 6)]]]))
    assert got.T.tolist() == [[0, 0], [0, 1], [1, 0], [1, 1], [2, 1], [3, 1]]   # each point once per geometry
    # buffered: the gap between the parts closes once 2 d exceeds it
    assert _pairs(np.array([[3.0, 3.0]]), [geom], [2.9]) == {(0, 0)}
    assert _pairs(np.array([[3.0, 3.0]]), [geom], [2.8]) == set()


def test_annulus_area_and_centroid():
    c = (10.0, -3.0)
    outer, inner = _ngon(c, 5.0, 96, 0.1), _ngon(c, 2.0, 48, 0.3)
    verts, ring_off, part_off, geom_off = pack_polygons([[[outer, inner]]])
    area, cen, box, dist = multipolygon_props_ref(verts, ring_off, part_off, geom_off, ratio=0.5)
    a_out, a_in = polygon_props_ref(*pack_rings([outer, inner]))[0]
    assert area[0] == abs(a_out) - abs(a_in)
    assert np.allclose(cen[0], c, rtol=0, atol=1e-13)
    assert box[0].tolist() == [outer[:, 0].min(), outer[:, 1].min(), outer[:, 0].max(), outer[:, 1].max()]
    assert dist[0] == np.sqrt(area[0] / np.pi) * 0.5
    # a clockwise hole and a closing vertex change nothing
    verts2, *off2 = pack_polygons([[[np.concatenate([outer, outer[:1]]), inner[::-1]]]])
    a2 = multipolygon_props_ref(verts2, *off2)[0]
    assert abs(a2[0] - area[0]) <= 1e-12 * area[0]


def test_plain_join_is_the_xor_of_the_single_ring_decisions():
    rng = np.random.default_rng(3)
    geoms = []
    for i in range(25):
        parts = []
        for _ in range(1 + i % 3):
            c = rng.uniform(5, 55, 2)
            rings = [_ngon(c, rng.uniform(3, 6), int(rng.integers(5, 20)), rng.uniform(0, 1))]
            for _ in range(int(rng.integers(0, 3))):            # holes, overlapping each other and the rim at times
                rings.append(_ngon(c + rng.uniform(-3, 3, 2), rng.uniform(0.5, 2.5), int(rng.integers(3, 12))))
            parts.append(rings)
        geoms.append(parts)
    verts, ring_off, part_off, geom_off = pack_polygons(geoms)
    pts = rng.uniform(-2, 62, (20000, 2))
    got = points_in_multipolygons_ref(pts, verts, ring_off, part_off, geom_off)
    per_ring = points_in_polygons_ref(pts, verts, ring_off)
    geom_of_ring = np.repeat(np.arange(len(geoms)), np.diff(part_off[geom_off]))
    keys = per_ring[0].astype(np.int64) * len(geoms) + geom_of_ring[per_ring[1]]
    uniq, cnt = np.unique(keys, return_counts=True)
    odd = uniq[cnt % 2 == 1]
    assert np.array_equal(got[0].astype(np.int64) * len(geoms) + got[1], odd)
    assert got.shape[1] > 1000 and (cnt % 2 == 0).any()        # holes actually removed points


def test_single_ring_geometries_reproduce_the_ring_oracle_bit_for_bit():
    rng = np.random.default_rng(5)
    rings = [_ngon(rng.uniform(5, 45, 2), rng.uniform(1, 5), int(rng.integers(3, 30)), rng.uniform(0, 1))
             for _ in range(40)]
    rings[3] = rings[3][::-1]                                   # clockwise
    rings[4] = np.concatenate([rings[4], rings[4][:1]])         # closed
    rings[5] = np.array([[1.0, 2.0], [3.0, 4.0]])               # two vertices: zero area, first vertex
    rings[6] = np.array([[0.0, 0.0], [1.0, 1.0], [2.0, 2.0]])   # collinear
    verts, ring_off = pack_rings(rings)
    one = np.arange(len(rings) + 1)
    area, cen, box, dist = polygon_props_ref(verts, ring_off, ratio=0.3)
    m_area, m_cen, m_box, m_dist = multipolygon_props_ref(verts, ring_off, one, one, ratio=0.3)
    assert np.array_equal(m_area, np.abs(area)) and np.array_equal(m_cen, cen)
    assert np.array_equal(m_box, box) and np.array_equal(m_dist, dist)
    pts = rng.uniform(-2, 52, (20000, 2))
    d = np.sqrt(np.abs(area) / np.pi) * np.array([0.3, 0.0, -0.2])[np.arange(len(rings)) % 3]
    assert np.array_equal(points_in_multipolygons_ref(pts, verts, ring_off, one, one, d),
                          points_in_buffered_polygons_ref(pts, verts, ring_off, d))
    assert np.array_equal(points_in_multipolygons_ref(pts, verts, ring_off, one, one),
                          points_in_polygons_ref(pts, verts, ring_off))


def test_empty_rings_parts_and_geometries_match_nothing():
    geoms = [[], [[]], [[np.zeros((0, 2))]], [[np.zeros((0, 2)), _sq(0, 0, 1, 1)]], [[_sq(0, 0, 2, 2)]]]
    verts, ring_off, part_off, geom_off = pack_polygons(geoms)
    assert part_off.tolist() == [0, 0, 1, 3, 4] and geom_off.tolist() == [0, 0, 1, 2, 3, 4]
    got = points_in_multipolygons_ref(np.array([[0.5, 0.5]]), verts, ring_off, part_off, geom_off, [0.1] * 5)
    assert got.T.tolist() == [[0, 3], [0, 4]]                  # an empty exterior leaves its hole alone
    area, cen, box, _ = multipolygon_props_ref(verts, ring_off, part_off, geom_off)
    assert area[:3].tolist() == [0.0, 0.0, 0.0] and np.isnan(cen[:3]).all() and np.isinf(box[:3]).all()
    assert area[3] == -1.0 and cen[3].tolist() == [0.5, 0.5]    # the lone hole counts negative
    # net area 0 with vertices: the first ring's centroid
    a, c, _, _ = multipolygon_props_ref(*pack_polygons([[[_sq(0, 0, 2, 2), _sq(0, 0, 2, 2)]]]))
    assert a[0] == 0.0 and c[0].tolist() == [1.0, 1.0]


def _polygon(ext, holes=()):
    return SimpleNamespace(geom_type="Polygon", exterior=SimpleNamespace(coords=[tuple(p) for p in ext]),
                           interiors=[SimpleNamespace(coords=[tuple(p) for p in h]) for h in holes])


def test_pack_polygons_nested_and_duck_typed():
    a, h, b = _sq(0, 0, 4, 4), _sq(1, 1, 2, 2), _sq(6, 6, 7, 7)
    nested = pack_polygons([[[a, h]], [[b], [a + 10]]])
    ducks = pack_polygons([_polygon(a, [h]), SimpleNamespace(geom_type="MultiPolygon", geoms=[_polygon(b), _polygon(a + 10)])])
    for x, y in zip(nested, ducks):
        assert np.array_equal(x, y)
    verts, ring_off, part_off, geom_off = nested
    assert ring_off.tolist() == [0, 4, 8, 12, 16] and part_off.tolist() == [0, 2, 3, 4] and geom_off.tolist() == [0, 1, 3]
    assert verts.dtype == np.float64 and np.array_equal(verts[4:8], h)
    assert pack_polygons([None])[3].tolist() == [0, 0]
    with pytest.raises(TypeError):
        pack_polygons([SimpleNamespace(geom_type="LineString")])
    # Outlines keep the layout; of_type keeps parts and holes and renumbers
    o = Outlines(*nested[:2], ["nucleus", "cell"], *nested[2:])
    assert o.multi and o.n_poly == 2
    c = o.of_type("cell")
    assert c.n_poly == 1 and c.part_off.tolist() == [0, 1, 2] and c.geom_off.tolist() == [0, 2]
    assert np.array_equal(c.verts, np.concatenate([b, a + 10])) and c.boundary_type.tolist() == ["cell"]
    assert o.of_type("none").n_poly == 0


def test_malformed_offsets_raise():
    verts, ring_off, part_off, geom_off = pack_polygons([[[_sq(0, 0, 1, 1), _sq(0, 0, 1, 1)]], [[_sq(0, 0, 1, 1)]]])
    bad = [
        (ring_off[:-1], part_off, geom_off),                   # rings do not cover the vertices
        (ring_off, np.array([0, 2, 1, 3]), geom_off),          # decreasing
        (ring_off, part_off, np.array([1, 2])),                # does not start at 0
        (ring_off, part_off, np.array([0, 1, 3])),             # past the parts
        (ring_off, np.array([0, 2]), np.array([0, 1])),        # leaves a ring out
        (np.array([], dtype=np.int64), part_off, geom_off),
    ]
    for args in bad:
        with pytest.raises(ValueError):
            check_layout(len(verts), *args)
        with pytest.raises(ValueError):
            PackedPolygons(verts, *args)
        with pytest.raises(ValueError):
            Outlines(verts, args[0], None, *args[1:])
    with pytest.raises(ValueError):
        PackedPolygons(verts, ring_off, part_off)              # the two offsets go together
    with pytest.raises(ValueError):
        Outlines(verts, ring_off, ["cell"] * 3, part_off, geom_off)   # one label per geometry
    check_layout(len(verts), ring_off, part_off, geom_off)


def test_multi_abi_argument_validation_without_gpu(lib):
    assert lib.sgb_polygon_props_multi(None, None, None, None, -1, 0.0, None, None, None, None, None) == -3
    assert lib.sgb_polygon_props_multi(None, None, None, None, 0, 0.0, None, None, None, None, None) == 0
    assert lib.sgb_polygon_props_multi(None, None, None, None, 3, 0.0, None, None, None, None, None) == -1
    assert lib.sgb_pip_multi_count(None, 0, 10, None, None, None, None, None, 4, 0.0, 0.0, 1.0, 1, 1, None, None, 0,
                                   None) == -1
    assert b"null offsets" in lib.sgb_last_error()
    assert lib.sgb_pip_multi_fill(None, None, None, None, None, 10, 4, 0.0, 0.0, 1.0, 1, 1, 5, None, 5, None, 0, None, 0,
                                  None) == -1
    assert lib.sgb_pip_multi_fill(None, None, None, None, None, 10, 4, 0.0, 0.0, 1.0, 1, 1, 0, None, 0, None, 0, None, 0,
                                  None) == 0
