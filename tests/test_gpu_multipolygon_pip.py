"""GPU parity of the join and the properties for outlines with holes and several parts (sgb_polygon_props_multi,
sgb_pip_multi_count / _fill): bit-exact against the numpy oracle, against the XOR of the existing single-ring join, and
against the existing entry points on one-ring geometries; the prediction graph from such outlines."""
import os
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle.multipolygon_ref import multipolygon_props_ref, points_in_multipolygons_ref
from segger_b200 import neighbors as nb
from segger_b200.geometry import BufferedOutlines, Outlines, PackedPolygons, pack_polygons, pack_rings, points_in_polygons
from segger_b200.synth import synth
from tests.test_gpu_buffered_pip import _mixed_rings, _ngon, _star

pytestmark = pytest.mark.gpu


def _mixed_geoms(rng):
    """Annuli, holed stars, two- and three-part geometries, one with 80 holes (over the 64-ring cap), one whose rings
    total over 1,024 vertices, empty rings, parts and geometries, closed rings and rings of 2 vertices; 120 x 120."""
    geoms = []
    for i, c in enumerate(rng.uniform(10, 110, (48, 2))):
        kind = i % 8
        if kind == 0:                                                           # annulus
            geoms.append([[_ngon(c, rng.uniform(4, 7), 16, rng.uniform(0, 1)), _ngon(c + rng.uniform(-1, 1, 2), 2.0, 12)]])
        elif kind == 1:                                                         # star with two holes, one closed
            h = _ngon(c + 0.9, 0.6, 9)
            geoms.append([[_star(c, 2.5, 6.0, 7, rng), _ngon(c - 0.5, 1.0, 7), np.concatenate([h, h[:1]])]])
        elif kind == 2:                                                         # two parts, the second holed
            geoms.append([[_ngon(c, 3.0, 14)], [_ngon(c + 7.0, 2.5, 10), _ngon(c + 7.0, 1.0, 6)]])
        elif kind == 3:                                                         # 80 holes in a square
            sq = np.array([[-6.0, -6.0], [6.0, -6.0], [6.0, 6.0], [-6.0, 6.0]]) + c
            holes = [_ngon(c + np.array([-5.0 + 1.25 * (k % 9), -5.0 + 1.25 * (k // 9)]), 0.4, 5) for k in range(80)]
            geoms.append([[sq] + holes])
        elif kind == 4:                                                         # rings total 1,300 vertices
            geoms.append([[_ngon(c, 6.0, 1000, 0.2), _ngon(c, 2.0, 300)]])
        elif kind == 5:                                                         # empties and a 2-vertex ring
            geoms.append([[], [np.zeros((0, 2))], [_ngon(c, 3.0, 8), np.array([[c[0], c[1]], [c[0] + 1, c[1]]])]])
        elif kind == 6:                                                         # one ring over the 1,024 cap
            geoms.append([[_ngon(c, 4.5, 1100, 0.3)]])
        else:                                                                   # three parts
            geoms.append([[_ngon(c + 3.0 * np.array([np.cos(k), np.sin(k)]), 1.2, 6)] for k in range(3)])
    geoms[13] = []                                                              # no parts
    geoms[21] = [[np.zeros((0, 2))]]                                            # one empty ring
    return geoms


def _buffered(layout, dist):
    o = Outlines(layout[0], layout[1], None, layout[2], layout[3])
    return BufferedOutlines(o, torch.as_tensor(np.asarray(dist, dtype=np.float64)).cuda())


def _xor_reduce(pairs, geom_of_ring, n_geom):
    keys = pairs[0].astype(np.int64) * n_geom + geom_of_ring[pairs[1]]
    uniq, cnt = np.unique(keys, return_counts=True)
    odd = uniq[cnt % 2 == 1]
    return np.stack([odd // n_geom, odd % n_geom]).astype(np.int32)


def test_multipolygon_props_bit_exact():
    layout = pack_polygons(_mixed_geoms(np.random.default_rng(1)))
    area, cen, box, dist = multipolygon_props_ref(*layout, ratio=0.37)
    o = Outlines(layout[0], layout[1], None, layout[2], layout[3])
    assert np.array_equal(o.areas(), area) and np.array_equal(o.centroids(), cen, equal_nan=True)
    d_area, d_cen, d_box, d_dist = o._device_props("cuda", 0.37)
    assert np.array_equal(d_area.cpu().numpy(), area) and np.array_equal(d_box.cpu().numpy(), box)
    assert np.array_equal(d_dist.cpu().numpy(), dist)
    assert np.array_equal(d_cen.cpu().numpy(), cen, equal_nan=True)
    assert (area[np.isfinite(box[:, 0])] >= 0).all() and np.isnan(cen[[13, 21]]).all()


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_multi_join_bit_exact_mixed_signs(dtype):
    rng = np.random.default_rng(2 if dtype == np.float32 else 3)
    geoms = _mixed_geoms(rng)
    layout = pack_polygons(geoms)
    area = multipolygon_props_ref(*layout)[0]
    dist = np.sqrt(np.abs(area) / np.pi) * np.array([0.3, 0.0, -0.05])[np.arange(len(geoms)) % 3]
    pts = rng.uniform(-5, 125, (300_000, 2)).astype(dtype)
    ref = points_in_multipolygons_ref(pts, *layout, dist=dist)
    got = points_in_polygons(pts, _buffered(layout, dist))
    assert got.dtype == torch.int32 and not got.is_cuda
    assert np.array_equal(got.numpy(), ref)
    live = [g for g in range(len(geoms)) if g not in (13, 21)]
    assert all((ref[1] == g).any() for g in live)                           # every real geometry is exercised
    plain = points_in_polygons(pts, PackedPolygons(*layout))
    assert np.array_equal(plain.numpy(), points_in_multipolygons_ref(pts, *layout))
    again = points_in_polygons(torch.from_numpy(pts).cuda(), PackedPolygons(*layout), device_output=True)
    assert again.is_cuda and torch.equal(again.cpu(), plain)


def test_plain_multi_join_is_the_xor_of_the_existing_single_ring_join():
    """Oracle-independent: the same rings as separate polygons through sgb_pip_count / _fill, reduced by XOR."""
    rng = np.random.default_rng(4)
    geoms = _mixed_geoms(rng)
    verts, ring_off, part_off, geom_off = pack_polygons(geoms)
    pts = rng.uniform(-5, 125, (400_000, 2))
    per_ring = points_in_polygons(pts, verts, ring_off).numpy()
    geom_of_ring = np.repeat(np.arange(len(geoms)), np.diff(part_off[geom_off]))
    want = _xor_reduce(per_ring, geom_of_ring, len(geoms))
    got = points_in_polygons(pts, PackedPolygons(verts, ring_off, part_off, geom_off)).numpy()
    assert np.array_equal(got, want)
    assert got.shape[1] < per_ring.shape[1]                                 # holes removed points


def test_one_ring_layout_equals_the_existing_entry_points():
    rng = np.random.default_rng(6)
    rings = _mixed_rings(rng)
    verts, off = pack_rings(rings)
    one = np.arange(len(rings) + 1)
    pts = rng.uniform(-10, 130, (300_000, 2))
    assert np.array_equal(points_in_polygons(pts, PackedPolygons(verts, off, one, one)).numpy(),
                          points_in_polygons(pts, verts, off).numpy())
    single, multi = Outlines(verts, off), Outlines(verts, off, None, one, one)
    area, cen, box, dist = single._device_props("cuda", 0.25)
    m_area, m_cen, m_box, m_dist = multi._device_props("cuda", 0.25)
    assert torch.equal(m_area, area.abs()) and torch.equal(m_box, box) and torch.equal(m_dist, dist)
    assert np.array_equal(m_cen.cpu().numpy(), cen.cpu().numpy(), equal_nan=True)
    d = dist * torch.tensor([1.0, 0.0, -1.0], dtype=torch.float64, device="cuda").repeat(len(rings))[:len(rings)]
    assert torch.equal(points_in_polygons(pts, BufferedOutlines(multi, d)),
                       points_in_polygons(pts, BufferedOutlines(single, d)))
    gd = np.load(os.path.join(os.path.dirname(__file__), "golden", "pip_small.npz"))
    one = np.arange(len(gd["ring_off"]))
    got = points_in_polygons(gd["points"], PackedPolygons(gd["verts"], gd["ring_off"], one, one))
    assert np.array_equal(got.numpy(), gd["pairs"])


def _synth_cells(ts, rng):
    """Per synthetic cell: a 'cell' geometry (a 16-gon with its nucleus as a hole, every third one split into two
    parts) and a 'nucleus' geometry (the nucleus 12-gon), interleaved."""
    geoms, types = [], []
    for i, c in enumerate(ts.bd_pos.astype(np.float64)):
        nuc = _ngon(c + rng.uniform(-1, 1, 2), 2.5, 12)
        cell = _ngon(c, 6.5 * rng.uniform(0.8, 1.1), 16, rng.uniform(0, 1))
        geoms.append([[cell, nuc]] + ([[_ngon(c + 9.0, 1.5, 8)]] if i % 3 == 0 else []))
        types.append("cell")
        geoms.append([[nuc]])
        types.append("nucleus")
    return geoms, np.array(types)


def test_setup_prediction_graph_from_multipart_outlines_all_modes(monkeypatch):
    for mod in ("geopandas", "shapely"):
        monkeypatch.setitem(sys.modules, mod, None)                          # importing either now fails
    ts = synth(50_000, 500, seed=5)
    rng = np.random.default_rng(5)
    geoms, types = _synth_cells(ts, rng)
    verts, ring_off, part_off, geom_off = pack_polygons(geoms)
    bd = Outlines(verts, ring_off, types, part_off, geom_off)
    for mode, ratio in (("cell", 0.5), ("nucleus", 1.2), ("cell", -0.2)):
        sel = pack_polygons([g for g, t in zip(geoms, types) if t == mode])
        dist = multipolygon_props_ref(*sel, ratio=ratio)[3]
        ref = points_in_multipolygons_ref(ts.tx_pos, *sel, dist=dist)
        got = nb.setup_prediction_graph(ts.tx_pos, bd, 5, ratio, mode)
        assert got.dtype == torch.int32 and not got.is_cuda
        assert np.array_equal(got.numpy(), ref), mode
        assert ref.shape[1] > 0 and ref[1].max() < (types == mode).sum()
    # 'cell' excludes the nucleus it surrounds: no transcript is a candidate of both a cell and its own nucleus
    cell = nb.setup_prediction_graph(ts.tx_pos, bd, 5, 0.0, "cell")
    nuc = nb.setup_prediction_graph(ts.tx_pos, bd, 5, 0.0, "nucleus")
    assert not (set(map(tuple, cell.T.tolist())) & set(map(tuple, nuc.T.tolist())))
    # uniform: k nearest transcripts of every geometry centroid, centroids from the device
    cen = multipolygon_props_ref(verts, ring_off, part_off, geom_off)[1]
    assert np.array_equal(bd.centroids(), cen)
    got = nb.setup_prediction_graph(ts.tx_pos, bd, 5, 0.5, "uniform")
    assert torch.equal(got, nb.setup_prediction_graph(ts.tx_pos, cen, 5, 0.5, "uniform"))
    assert got.shape[1] == 5 * len(types)


class _Series(list):
    """The few GeoSeries members setup_prediction_graph reads; ``buffer`` returns the geometries given as buffered."""

    def __init__(self, geoms, buffered=None):
        super().__init__(geoms)
        self.buffered = buffered

    @property
    def area(self):
        return np.ones(len(self))

    def buffer(self, dists):
        assert len(dists) == len(self)
        return _Series(self.buffered)

    def reset_index(self, drop=False):
        return self


class _Frame:
    def __init__(self, geoms, buffered, types):
        self.geoms, self.buffered, self.types = geoms, buffered, np.asarray(types)

    def __getitem__(self, key):
        if isinstance(key, str):
            return self.types
        keep = np.nonzero(key)[0]
        return SimpleNamespace(geometry=_Series([self.geoms[i] for i in keep], [self.buffered[i] for i in keep]))

    @property
    def geometry(self):
        return _Series(self.geoms, self.buffered)


def _shp_polygon(ext, holes=()):
    return SimpleNamespace(geom_type="Polygon", exterior=SimpleNamespace(coords=ext),
                           interiors=[SimpleNamespace(coords=h) for h in holes])


def test_geodataframe_path_keeps_holes_and_parts():
    """Buffered geometries that are a holed Polygon and a MultiPolygon: before, the hole was dropped and the
    MultiPolygon raised AttributeError."""
    ring = np.array([[0.0, 0.0], [10.0, 0.0], [10.0, 10.0], [0.0, 10.0], [0.0, 0.0]])
    hole = np.array([[3.0, 3.0], [7.0, 3.0], [7.0, 7.0], [3.0, 7.0], [3.0, 3.0]])
    holed = _shp_polygon(ring, [hole])
    multi = SimpleNamespace(geom_type="MultiPolygon", geoms=[_shp_polygon(ring + 20.0), _shp_polygon(ring + [40.0, 20.0])])
    plain = _shp_polygon(ring + [0.0, 40.0])
    buffered = [holed, plain, multi]
    bd = _Frame([None] * 3, buffered, ["cell", "nucleus", "cell"])
    pts = np.array([[5.0, 5.0], [1.0, 1.0], [25.0, 25.0], [45.0, 25.0], [35.0, 25.0], [5.0, 45.0]])
    got = nb.setup_prediction_graph(pts, bd, 5, 0.1, "cell")
    ref = points_in_multipolygons_ref(pts, *pack_polygons([holed, multi]))
    assert np.array_equal(got.numpy(), ref)
    assert got.T.tolist() == [[1, 0], [2, 1], [3, 1]]                      # not the hole, both parts, one id
    # a frame of plain hole-free polygons takes the one-ring layout and gives what it gave before
    got = nb.setup_prediction_graph(pts, bd, 5, 0.1, "nucleus")
    assert got.T.tolist() == [[5, 0]]


def test_one_million_transcripts_ten_thousand_annuli_sampled():
    rng = np.random.default_rng(7)
    n_geom, side = 10_000, 1_400.0
    centers = rng.uniform(10, side - 10, (n_geom, 2))
    geoms = [[[_ngon(c, 6.8 * (1 + 0.3 * rng.uniform(-1, 1, 16)), 16), _ngon(c + rng.uniform(-1, 1, 2), 2.5, 12)]]
             for c in centers]
    layout = pack_polygons(geoms)
    pts = rng.uniform(0, side, (1_000_000, 2)).astype(np.float32)
    bd = Outlines(layout[0], layout[1], None, layout[2], layout[3])
    got = points_in_polygons(pts, bd.buffered(0.4)).numpy()
    dist = multipolygon_props_ref(*layout, ratio=0.4)[3]
    sample = np.sort(rng.choice(n_geom, 300, replace=False))
    ref = points_in_multipolygons_ref(pts, *pack_polygons([geoms[g] for g in sample]), dist=dist[sample])
    ref[1] = sample[ref[1]]
    keep = np.isin(got[1], sample)
    assert np.array_equal(got[:, keep], ref)
    assert ref.shape[1] > 10_000
