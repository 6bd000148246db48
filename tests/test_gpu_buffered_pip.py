"""GPU parity of the buffered point-in-polygon join and of the ring properties (sgb_polygon_props,
sgb_pip_buffered_count / _fill) against the numpy oracle: bit-exact pair lists and bit-exact areas / centroids."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle.buffered_geometry_ref import points_in_buffered_polygons_ref, polygon_props_ref
from segger_b200 import neighbors as nb
from segger_b200.geometry import BufferedOutlines, Outlines, pack_rings, points_in_polygons
from segger_b200.synth import synth

pytestmark = pytest.mark.gpu


def _ngon(c, r, n=16, phase=0.0):
    ang = np.linspace(0, 2 * np.pi, n, endpoint=False) + phase
    return np.stack([c[0] + r * np.cos(ang), c[1] + r * np.sin(ang)], 1)


def _star(c, r_in, r_out, arms, rng):
    ang = np.linspace(0, 2 * np.pi, 2 * arms, endpoint=False) + rng.uniform(0, np.pi)
    r = np.where(np.arange(2 * arms) % 2 == 0, r_out, r_in) * rng.uniform(0.85, 1.15, 2 * arms)
    return np.stack([c[0] + r * np.cos(ang), c[1] + r * np.sin(ang)], 1)


def _mixed_rings(rng):
    """Convex 16-gons, non-convex stars, rings over 1,024 vertices, zero-length and collinear edges, closed rings and
    degenerate ones, spread over a 120 x 120 square."""
    rings = []
    for i, c in enumerate(rng.uniform(8, 112, (60, 2))):
        kind = i % 6
        if kind == 0:
            rings.append(_ngon(c, rng.uniform(3, 6), 16, rng.uniform(0, 1)))
        elif kind == 1:
            rings.append(_star(c, 1.5, 5.5, 6, rng))
        elif kind == 2:
            rings.append(_star(c, 3.0, 6.0, 700, rng))                          # 1,400 vertices: global-memory path
        elif kind == 3:                                                         # zero-length + collinear edges
            sq = np.array([[0, 0], [2, 0], [4, 0], [4, 0], [4, 3], [4, 6], [0, 6], [0, 6], [0, 3]], dtype=np.float64)
            rings.append(sq + c - 2.0)
        elif kind == 4:
            r = _ngon(c, rng.uniform(2, 5), 11)
            rings.append(np.concatenate([r, r[:1]]))                            # closed ring
        else:
            rings.append(_ngon(c, 4.0, 1024 + 3, 0.1))                          # just over the shared-memory ring
    rings[5] = np.array([[1.0, 1.0], [2.0, 2.0]])                              # < 3 vertices: matches nothing
    rings[11] = np.zeros((0, 2))                                                # empty
    return rings


def _join(pts, verts, off, dist, **kw):
    o = Outlines(verts, off)
    return points_in_polygons(pts, BufferedOutlines(o, torch.from_numpy(np.asarray(dist, dtype=np.float64)).cuda()), **kw)


def test_polygon_props_bit_exact():
    rng = np.random.default_rng(1)
    rings = _mixed_rings(rng)
    verts, off = pack_rings(rings)
    area, cen, box, dist = polygon_props_ref(verts, off, ratio=0.37)
    o = Outlines(verts, off)
    assert np.array_equal(o.areas(), area)
    assert np.array_equal(o.centroids(), cen, equal_nan=True)
    d_area, d_cen, d_box, d_dist = o._device_props("cuda", 0.37)
    assert np.array_equal(d_area.cpu().numpy(), area) and np.array_equal(d_box.cpu().numpy(), box)
    assert np.array_equal(d_dist.cpu().numpy(), dist)
    assert np.array_equal(d_cen.cpu().numpy(), cen, equal_nan=True)
    assert np.array_equal(o.buffered(0.37).dist.cpu().numpy(), dist)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_buffered_join_bit_exact_mixed_signs(dtype):
    rng = np.random.default_rng(2 if dtype == np.float32 else 3)
    rings = _mixed_rings(rng)
    verts, off = pack_rings(rings)
    area = polygon_props_ref(verts, off)[0]
    scale = np.sqrt(np.abs(area) / np.pi)
    sign = np.array([0.4, 0.0, -0.25])[np.arange(len(rings)) % 3]
    dist = scale * sign
    pts = rng.uniform(-10, 130, (300_000, 2)).astype(dtype)
    ref = points_in_buffered_polygons_ref(pts, verts, off, dist)
    got = _join(pts, verts, off, dist)
    assert got.dtype == torch.int32 and not got.is_cuda
    assert np.array_equal(got.numpy(), ref)
    assert all((ref[1] == g).any() for g in range(len(rings)) if g not in (5, 11))    # every real ring is exercised
    # deterministic, and device_output keeps the same list on the device
    again = _join(torch.from_numpy(pts).cuda(), verts, off, dist, device_output=True)
    assert again.is_cuda and torch.equal(again.cpu(), got)


def test_grown_boxes_leave_the_raw_union():
    """Rings at the edge of the union box: the grid must cover the grown boxes, or these points are never binned."""
    sq = np.array([[0.0, 0.0], [2.0, 0.0], [2.0, 2.0], [0.0, 2.0]])
    verts, off = pack_rings([sq, sq + 10.0])
    pts = np.array([[2.9, 1.0], [-0.9, 1.0], [1.0, -0.9], [12.9, 11.0], [11.0, 12.9], [12.95, 12.2], [3.1, 1.0], [1.0, 1.0]])
    dist = np.array([1.0, 1.0])
    ref = points_in_buffered_polygons_ref(pts, verts, off, dist)
    got = _join(pts, verts, off, dist).numpy()
    assert np.array_equal(got, ref)
    assert set(map(tuple, got.T)) == {(0, 0), (1, 0), (2, 0), (3, 1), (4, 1), (5, 1), (7, 0)}


def test_zero_distance_reproduces_the_plain_golden_fixture():
    gd = np.load(os.path.join(os.path.dirname(__file__), "golden", "pip_small.npz"))
    o = Outlines(gd["verts"], gd["ring_off"])
    got = points_in_polygons(gd["points"], o.buffered(0.0))
    assert np.array_equal(got.numpy(), gd["pairs"])


def _synth_outlines(ts, rng):
    """A 16-gon cell outline and a smaller nucleus outline per synthetic cell, interleaved."""
    rings, types = [], []
    for c in ts.bd_pos.astype(np.float64):
        rings.append(_ngon(c, 6.5 * rng.uniform(0.8, 1.1), 16, rng.uniform(0, 1)))
        types.append("cell")
        rings.append(_ngon(c + rng.uniform(-1, 1, 2), 3.0, 12))
        types.append("nucleus")
    verts, off = pack_rings(rings)
    return verts, off, np.array(types)


def test_setup_prediction_graph_from_outlines_all_modes(monkeypatch):
    for mod in ("geopandas", "shapely"):
        monkeypatch.setitem(sys.modules, mod, None)                          # importing either now fails
    ts = synth(50_000, 500, seed=5)
    rng = np.random.default_rng(5)
    verts, off, types = _synth_outlines(ts, rng)
    bd = Outlines(verts, off, types)
    for mode, ratio in (("cell", 0.5), ("nucleus", 1.2), ("cell", -0.2)):
        sel = np.nonzero(types == mode)[0]
        s_verts, s_off = pack_rings([verts[off[g]:off[g + 1]] for g in sel])
        dist = polygon_props_ref(s_verts, s_off, ratio)[3]
        ref = points_in_buffered_polygons_ref(ts.tx_pos, s_verts, s_off, dist)
        got = nb.setup_prediction_graph(ts.tx_pos, bd, 5, ratio, mode)
        assert got.dtype == torch.int32 and not got.is_cuda
        assert np.array_equal(got.numpy(), ref), mode
        assert ref.shape[1] > 0 and ref[1].max() < sel.size                  # ids count within the selection
    # the buffered outlines are built once and reused by the next tile
    assert bd.of_type("cell").buffered(0.5) is bd.of_type("cell").buffered(0.5)
    # no boundary_type: every ring takes part
    plain = Outlines(verts, off)
    dist = polygon_props_ref(verts, off, 0.3)[3]
    assert np.array_equal(nb.setup_prediction_graph(ts.tx_pos, plain, 5, 0.3, "cell").numpy(),
                          points_in_buffered_polygons_ref(ts.tx_pos, verts, off, dist))
    # uniform: k nearest transcripts of every outline centroid, centroids from the device
    cen = polygon_props_ref(verts, off)[1]
    assert np.array_equal(bd.centroids(), cen)
    got = nb.setup_prediction_graph(ts.tx_pos, bd, 5, 0.5, "uniform")
    assert torch.equal(got, nb.setup_prediction_graph(ts.tx_pos, cen, 5, 0.5, "uniform"))
    assert got.shape[1] == 5 * len(types)


def test_one_million_transcripts_ten_thousand_outlines_sampled():
    rng = np.random.default_rng(7)
    n_poly, side = 10_000, 1_400.0
    centers = rng.uniform(10, side - 10, (n_poly, 2))
    rings = [_ngon(c, 6.8 * (1 + 0.3 * rng.uniform(-1, 1, 16)), 16) for c in centers]
    verts, off = pack_rings(rings)
    pts = rng.uniform(0, side, (1_000_000, 2)).astype(np.float32)
    bd = Outlines(verts, off)
    got = points_in_polygons(pts, bd.buffered(0.4)).numpy()
    dist = polygon_props_ref(verts, off, 0.4)[3]
    sample = np.sort(rng.choice(n_poly, 300, replace=False))
    s_verts, s_off = pack_rings([rings[g] for g in sample])
    ref = points_in_buffered_polygons_ref(pts, s_verts, s_off, dist[sample])
    ref[1] = sample[ref[1]]
    keep = np.isin(got[1], sample)
    assert np.array_equal(got[:, keep], ref)
    assert ref.shape[1] > 10_000
