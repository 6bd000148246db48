"""CPU tests of the buffered point-in-polygon contract (oracle/buffered_geometry_ref.py) and of the host side of
``geometry.Outlines``: known answers, strictness at the rim, monotonicity in the distance, an independent brute-force
distance, boundary-type selection and the C-ABI argument checks."""
import numpy as np
import pytest

from oracle.buffered_geometry_ref import points_in_buffered_polygons_ref, polygon_props_ref
from oracle.geometry_ref import points_in_polygons_ref
from segger_b200.geometry import Outlines, pack_rings

SQ2 = np.array([[0.0, 0.0], [2.0, 0.0], [2.0, 2.0], [0.0, 2.0]])


def _pairs(pts, rings, dist):
    verts, off = pack_rings(rings)
    return set(map(tuple, points_in_buffered_polygons_ref(pts, verts, off, np.asarray(dist, dtype=np.float64)).T))


def _stars(rng, n, n_arms=7, r_in=2.0, r_out=5.0, side=60.0):
    rings = []
    for c in rng.uniform(8, side - 8, (n, 2)):
        ang = np.linspace(0, 2 * np.pi, 2 * n_arms, endpoint=False) + rng.uniform(0, np.pi)
        r = np.where(np.arange(2 * n_arms) % 2 == 0, r_out, r_in) * rng.uniform(0.8, 1.2, 2 * n_arms)
        rings.append(np.stack([c[0] + r * np.cos(ang), c[1] + r * np.sin(ang)], 1))
    return rings


def test_area_centroid_box_known_answers():
    unit = np.array([[0.0, 0.0], [1.0, 0.0], [1.0, 1.0], [0.0, 1.0]])
    ccw = np.array([[0.0, 0.0], [4.0, 0.0], [0.0, 3.0]])
    rings = [unit, np.concatenate([unit, unit[:1]]), ccw, ccw[::-1], np.concatenate([ccw[::-1], ccw[-1:]]),
             np.zeros((0, 2)), np.array([[5.0, 6.0], [7.0, 8.0]])]
    verts, off = pack_rings(rings)
    area, cen, box, dist = polygon_props_ref(verts, off, ratio=0.5)
    assert area.tolist() == [1.0, 1.0, 6.0, -6.0, -6.0, 0.0, 0.0]          # open == closed; CW < 0
    assert np.allclose(cen[:5], [[0.5, 0.5], [0.5, 0.5], [4 / 3, 1.0], [4 / 3, 1.0], [4 / 3, 1.0]], rtol=0, atol=1e-15)
    assert np.isnan(cen[5]).all() and cen[6].tolist() == [5.0, 6.0]        # empty: NaN; zero area: first vertex
    assert box[2].tolist() == [0.0, 0.0, 4.0, 3.0] and box[5].tolist() == [np.inf, np.inf, -np.inf, -np.inf]
    assert dist[3] == np.sqrt(6.0 / np.pi) * 0.5 and dist[5] == 0.0


def test_square_corner_and_exact_rim():
    c = 2.0 + np.array([0.99, 1.02]) / np.sqrt(2.0)
    pts = np.array([[c[0], c[0]], [c[1], c[1]], [3.0, 1.0], [-1.0, 1.0], [1.0, 2.999], [0.5, 1.0], [1.0, 1.0]])
    got = _pairs(pts, [SQ2], [1.0])
    assert (0, 0) in got and (1, 0) not in got          # 0.99 from the corner in, 1.02 out
    assert (2, 0) not in got and (3, 0) not in got      # exactly at distance d: out (strict)
    assert (4, 0) in got and (6, 0) in got
    ero = _pairs(pts, [SQ2], [-0.5])
    assert ero == {(6, 0)}                               # (0.5, 1) is exactly |d| from the edge: out


def test_notch_narrower_than_2d_fills_in():
    u = np.array([[0.0, 0.0], [3.0, 0.0], [3.0, 4.0], [1.7, 4.0], [1.7, 1.0], [1.3, 1.0], [1.3, 4.0], [0.0, 4.0]])
    pts = np.array([[1.5, 3.0], [1.5, 1.5], [1.5, 4.1]])            # 4.1: 0.224 from the notch's lips
    assert _pairs(pts, [u], [0.0]) == set()
    assert _pairs(pts, [u], [0.25]) == {(0, 0), (1, 0), (2, 0)}           # notch 0.4 wide < 2 d
    assert _pairs(pts, [u], [0.15]) == set()                              # 0.4 > 2 d: the notch stays open


def test_zero_distance_equals_plain_join_and_nesting_in_d():
    rng = np.random.default_rng(4)
    rings = _stars(rng, 30)
    rings[3] = np.concatenate([rings[3], rings[3][:1]])                    # a closed ring
    verts, off = pack_rings(rings)
    pts = rng.uniform(-2, 62, (20000, 2))
    area = polygon_props_ref(verts, off)[0]
    scale = np.sqrt(np.abs(area) / np.pi)
    zero = points_in_buffered_polygons_ref(pts, verts, off, np.zeros(len(rings)))
    assert np.array_equal(zero, points_in_polygons_ref(pts, verts, off))
    sets = [set(map(tuple, points_in_buffered_polygons_ref(pts, verts, off, scale * r).T))
            for r in (-0.3, -0.1, 0.0, 0.05, 0.2, 0.6)]
    for a, b in zip(sets, sets[1:]):
        assert a < b                                                       # strictly growing regions
    # mixed signs per ring: each ring behaves as it does alone
    mixed = scale * np.where(np.arange(len(rings)) % 3 == 0, -0.2, np.where(np.arange(len(rings)) % 3 == 1, 0.0, 0.3))
    got = points_in_buffered_polygons_ref(pts, verts, off, mixed)
    for g in range(len(rings)):
        alone = points_in_buffered_polygons_ref(pts, verts[off[g]:off[g + 1]], np.array([0, off[g + 1] - off[g]]),
                                                mixed[g:g + 1])
        assert np.array_equal(got[0, got[1] == g], alone[0])


def test_against_brute_force_hypot_distance():
    """Independent restatement: the distance to every edge at once by projection with np.hypot; membership must agree
    wherever the point is not within 1e-9 of the rim (the two formulas round differently there)."""
    rng = np.random.default_rng(11)
    rings = _stars(rng, 6, side=30.0)
    verts, off = pack_rings(rings)
    pts = rng.uniform(-4, 34, (40000, 2))
    dist = np.array([0.8, -0.7, 1.5, 0.0, 2.5, -0.3])
    got = set(map(tuple, points_in_buffered_polygons_ref(pts, verts, off, dist).T))
    plain = set(map(tuple, points_in_polygons_ref(pts, verts, off).T))
    for g, ring in enumerate(rings):
        a, b = ring, np.roll(ring, -1, axis=0)
        ab = b - a
        t = np.clip(((pts[:, None, :] - a[None]) * ab[None]).sum(-1) / (ab * ab).sum(-1)[None], 0.0, 1.0)
        q = a[None] + t[..., None] * ab[None]
        dmin = np.hypot(pts[:, None, 0] - q[..., 0], pts[:, None, 1] - q[..., 1]).min(1)
        inside = np.array([(i, g) in plain for i in range(len(pts))])
        d = dist[g]
        want = (inside | (dmin < d)) if d > 0 else ((inside & (dmin > -d)) if d < 0 else inside)
        clear = np.abs(dmin - abs(d)) > 1e-9
        have = np.array([(i, g) in got for i in range(len(pts))])
        assert np.array_equal(have[clear], want[clear])
        assert want.sum() > 0


def test_grown_box_reaches_outside_the_raw_union():
    pts = np.array([[2.9, 1.0], [-0.9, 1.0], [1.0, -0.9], [1.0, 2.9], [3.1, 1.0]])
    assert _pairs(pts, [SQ2], [1.0]) == {(0, 0), (1, 0), (2, 0), (3, 0)}


def test_outlines_type_selection_renumbers_on_the_host():
    rings = [SQ2 + 10 * i for i in range(5)]
    rings[2] = np.concatenate([rings[2], rings[2][:1]])
    verts, off = pack_rings(rings)
    o = Outlines(verts, off, np.array(["cell", "nucleus", "cell", "nucleus", "cell"]))
    c = o.of_type("cell")
    assert c.n_poly == 3 and c.of_type("cell").n_poly == 3 and o.of_type("cell") is c
    assert c.ring_off.tolist() == [0, 4, 9, 13]
    assert np.array_equal(c.verts[4:9], rings[2]) and np.array_equal(c.verts[9:], rings[4])
    assert o.of_type("nucleus").n_poly == 2 and o.of_type("other").n_poly == 0
    with pytest.raises(ValueError):
        Outlines(verts, off, ["cell"])
    with pytest.raises(ValueError):
        Outlines(verts, off[:-1])
    with pytest.raises(ValueError):
        Outlines(verts, off).of_type("cell")


def test_buffered_abi_argument_validation_without_gpu(lib):
    assert lib.sgb_polygon_props(None, None, -1, 0.0, None, None, None, None, None) == -3
    assert lib.sgb_polygon_props(None, None, 0, 0.0, None, None, None, None, None) == 0
    assert lib.sgb_pip_buffered_count(None, 0, 10, None, None, None, 4, 0.0, 0.0, 1.0, 1, 1, None, None, 0, None) == -1
    assert b"null dist" in lib.sgb_last_error()
    assert lib.sgb_pip_buffered_fill(None, None, None, 10, 4, 0.0, 0.0, 1.0, 1, 1, 5, None, 5, None, 0, None, 0, None) == -1
