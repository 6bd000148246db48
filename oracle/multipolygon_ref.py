"""CPU restatement of the point-in-polygon join and polygon properties for outlines with holes and several parts --
TEST INFRASTRUCTURE ONLY.

The reference's cuSpatial join takes a GeoSeries in the GeoArrow polygon layout, so a boundary row may be a Polygon
with holes or a MultiPolygon.  This file states the contract the B200 kernels (sgb_polygon_props_multi,
sgb_pip_multi_count / _fill) implement for that layout, in numpy float64 with the kernels' operation order, so
decisions agree bit for bit.  Layout: ``verts`` [V, 2]; ``ring_off`` [R+1] vertices of ring r; ``part_off`` [Q+1]
rings of part q, the first its exterior and the rest its holes; ``geom_off`` [P+1] parts of geometry g.  A ring is
read as in ``buffered_geometry_ref`` (a repeated closing vertex dropped); rings of fewer than 3 vertices, and so
empty rings, parts and geometries, match nothing.

- plain join (strict): p is in geometry g iff the even-odd rule over all rings of g says "inside", i.e. the XOR over
  the rings of the single-ring decision (inside the ring's box, then ``_even_odd``) of ``points_in_polygons_ref``.  For
  valid geometry (disjoint parts, holes inside their exterior) this is the union of the parts minus their holes.  A
  point is listed at most once per geometry;
- buffered join with distance d: d > 0: inside, or squared distance (``ring_dist2_ref``) to the nearest edge of any
  ring of g ``< d^2``; d < 0: inside and squared distance to every ring ``> d^2``; d == 0: inside -- the exact
  Minkowski sum (erosion) of the whole geometry with a disc; candidates: the union of the ring boxes grown by
  ``|d| (1 + 2^-20)``;
- properties: each non-empty ring r has the area A_r, fan centroid c_r and box of ``polygon_props_ref``, and the
  weight w_r = +|A_r| for an exterior, -|A_r| for a hole.  With c_f the centroid of the first non-empty ring,
  accumulated left to right from 0 in ring order:
  ``area W = sum w_r`` (shapely's ``.area`` for valid geometry), ``centroid = c_f + (sum w_r (c_r - c_f)) / W``
  (the area-weighted mean of the ring centroids, written relative to c_f so that one ring reproduces its own centroid
  exactly), ``c_f`` when W == 0 (for a degenerate first ring that is its first vertex); ``box`` = union of the ring
  boxes; ``dist = sqrt(|W| / pi) * ratio`` (what ``polygons.buffer(sqrt(polygons.area / pi) * ratio)`` uses).  A
  geometry with one non-empty ring gives |A|, the centroid, box and dist of ``polygon_props_ref`` bit for bit; one
  without vertices has area 0, a NaN centroid and the empty box.

PARITY UNPINNED against shapely (not installed): beyond the buffering differences stated in
``buffered_geometry_ref`` (16-chord round joins, GEOS's ring simplifier), shapely's buffer of a holed or multi-part
geometry merges what overlaps after growing; the Minkowski sum here is the same set, but a point within about
``0.01 |d|`` of the exact rim can be judged differently.
"""
from __future__ import annotations

import numpy as np

from .buffered_geometry_ref import GROW, _even_odd, _ring, polygon_props_ref, ring_dist2_ref


def check_layout(n_verts: int, ring_off, part_off, geom_off):
    """-> (ring_off, part_off, geom_off) as int64 arrays; ValueError unless each starts at 0, never decreases and ends
    at the length of the array it indexes."""
    arrs = []
    for name, off, n in (("ring_off", ring_off, n_verts), ("part_off", part_off, None), ("geom_off", geom_off, None)):
        off = np.asarray(off, dtype=np.int64).reshape(-1)
        if n is None:
            n = len(arrs[-1]) - 1
        if off.size == 0 or off[0] != 0 or off[-1] != n or np.any(np.diff(off) < 0):
            raise ValueError(f"{name} must run from 0 to {n} without decreasing")
        arrs.append(off)
    return tuple(arrs)


def _geom_rings(ring_off, part_off, geom_off, g):
    """-> [(ring index, is_hole)] of geometry g in layout order."""
    out = []
    for q in range(geom_off[g], geom_off[g + 1]):
        for r in range(part_off[q], part_off[q + 1]):
            out.append((r, r != part_off[q]))
    return out


def multipolygon_props_ref(verts, ring_off, part_off, geom_off, ratio: float = 0.0):
    """-> (area [P], centroid [P, 2], box [P, 4] = (xmin, ymin, xmax, ymax), dist [P]), all float64."""
    verts = np.asarray(verts, dtype=np.float64).reshape(-1, 2)
    ring_off, part_off, geom_off = check_layout(verts.shape[0], ring_off, part_off, geom_off)
    r_area, r_cen, r_box, _ = polygon_props_ref(verts, ring_off)
    P = len(geom_off) - 1
    area = np.zeros(P)
    cen = np.full((P, 2), np.nan)
    box = np.tile(np.array([np.inf, np.inf, -np.inf, -np.inf]), (P, 1))
    for g in range(P):
        W = nx = ny = 0.0
        cf = None
        for r, hole in _geom_rings(ring_off, part_off, geom_off, g):
            if len(_ring(verts, ring_off, r)) == 0:
                continue
            cx, cy = float(r_cen[r, 0]), float(r_cen[r, 1])
            if cf is None:
                cf = (cx, cy)
            w = -abs(float(r_area[r])) if hole else abs(float(r_area[r]))
            box[g, :2] = np.minimum(box[g, :2], r_box[r, :2])
            box[g, 2:] = np.maximum(box[g, 2:], r_box[r, 2:])
            W = W + w
            nx = nx + w * (cx - cf[0])
            ny = ny + w * (cy - cf[1])
        area[g] = W
        if cf is not None:
            cen[g] = [cf[0] + nx / W, cf[1] + ny / W] if W != 0.0 else cf
    dist = np.sqrt(np.abs(area) / np.pi) * ratio
    return area, cen, box, dist


def points_in_multipolygons_ref(points, verts, ring_off, part_off, geom_off, dist=None) -> np.ndarray:
    """-> int32 [2, E] (row 0 = point, row 1 = geometry; point-major, geometries ascending); ``dist`` [P] or None for
    the plain join."""
    pts = np.asarray(points, dtype=np.float64)
    verts = np.asarray(verts, dtype=np.float64).reshape(-1, 2)
    ring_off, part_off, geom_off = check_layout(verts.shape[0], ring_off, part_off, geom_off)
    P = len(geom_off) - 1
    dist = np.zeros(P) if dist is None else np.asarray(dist, dtype=np.float64)
    out_p, out_g = [], []
    for g in range(P):
        rings = [_ring(verts, ring_off, r) for r, _ in _geom_rings(ring_off, part_off, geom_off, g)]
        rings = [ring for ring in rings if len(ring) >= 3]
        if not rings:
            continue
        d = float(dist[g])
        grow = abs(d) * GROW
        lo = np.min([ring.min(0) for ring in rings], axis=0)
        hi = np.max([ring.max(0) for ring in rings], axis=0)
        cand = np.nonzero((pts[:, 0] >= lo[0] - grow) & (pts[:, 0] <= hi[0] + grow)
                          & (pts[:, 1] >= lo[1] - grow) & (pts[:, 1] <= hi[1] + grow))[0]
        if cand.size == 0:
            continue
        px, py = pts[cand, 0], pts[cand, 1]
        inside = np.zeros(cand.size, dtype=bool)
        for ring in rings:
            rlo, rhi = ring.min(0), ring.max(0)
            in_box = (px >= rlo[0]) & (px <= rhi[0]) & (py >= rlo[1]) & (py <= rhi[1])
            inside ^= in_box & _even_odd(ring, px, py)
        if d != 0.0:
            d2 = np.min([ring_dist2_ref(ring, px, py) for ring in rings], axis=0)
            inside = (inside | (d2 < d * d)) if d > 0.0 else (inside & (d2 > d * d))
        hit = cand[inside]
        out_p.append(hit)
        out_g.append(np.full(hit.size, g, dtype=np.int64))
    if not out_p:
        return np.zeros((2, 0), dtype=np.int32)
    p, g = np.concatenate(out_p), np.concatenate(out_g)
    order = np.lexsort((g, p))
    return np.stack([p[order], g[order]]).astype(np.int32)
