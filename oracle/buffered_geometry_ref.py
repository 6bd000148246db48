"""CPU restatement of the buffered prediction-graph join -- TEST INFRASTRUCTURE ONLY.

The reference grows every cell / nucleus outline by ``sqrt(area / pi) * buffer_ratio`` with geopandas
(/root/reference/src/segger/data/utils/neighbors.py:229-231) and then keeps the transcripts strictly inside the grown
outline.  This file states the contract the B200 kernels (sgb_polygon_props, sgb_pip_buffered_count / _fill) implement
instead, in numpy float64 with the kernels' operation order, so decisions agree bit for bit:

- ring: the exterior ring as ``points_in_polygons_ref`` reads it (a repeated closing vertex is dropped; fewer than 3
  vertices match nothing);
- area: signed shoelace with x relative to the first vertex (GEOS's ring-area order),
  ``A = 0.5 * sum_{i=1..n-1} (x_i - x_0) * (y_{i+1} - y_{i-1})`` accumulated left to right, counter-clockwise > 0;
- centroid: triangle fan from the first vertex, ``p_0 + sum c_i (a_i + b_i) / (3 sum c_i)`` with ``a_i = p_i - p_0``,
  ``b_i = p_{i+1} - p_0``, ``c_i = a_i x b_i``; the first vertex when the fan area is 0, NaN for an empty ring;
- distance: ``d = sqrt(|A| / pi) * ratio``;
- membership (strict): ``d > 0``: inside the ring (the plain test, box prefilter included) or squared distance to the
  ring ``< d^2`` -- the exact Minkowski sum with a disc of radius d; ``d < 0``: inside and squared distance ``> d^2``;
  ``d == 0``: inside;
- squared distance to the ring: minimum over the edges a -> b of ``(ex - t dx)^2 + (ey - t dy)^2`` with
  ``dx, dy = b - a``, ``ex, ey = p - a``, ``L = dx^2 + dy^2``, ``t = clamp((ex dx + ey dy) / L, 0, 1)`` if L > 0 else 0;
- candidates: the ring's box grown by ``|d| (1 + 2^-20)``.

PARITY UNPINNED against shapely (not installed): shapely approximates round joins by 16 chords per quarter circle,
which lie inside the exact arc, and GEOS simplifies the input ring by about 1 % of d, so a point within about
``0.01 |d|`` of the exact buffered rim can be judged differently by geopandas.  Out of scope: GEOS's fillets and ring
simplifier, holes, multipolygons.
"""
from __future__ import annotations

import numpy as np

GROW = 1.0 + 2.0 ** -20


def _ring(verts: np.ndarray, ring_off: np.ndarray, g: int) -> np.ndarray:
    ring = verts[ring_off[g]:ring_off[g + 1]]
    if len(ring) >= 2 and ring[0, 0] == ring[-1, 0] and ring[0, 1] == ring[-1, 1]:
        ring = ring[:-1]
    return ring


def polygon_props_ref(verts: np.ndarray, ring_off: np.ndarray, ratio: float = 0.0):
    """-> (area [M], centroid [M, 2], box [M, 4] = (xmin, ymin, xmax, ymax), dist [M]), all float64."""
    verts = np.asarray(verts, dtype=np.float64).reshape(-1, 2)
    ring_off = np.asarray(ring_off, dtype=np.int64)
    M = len(ring_off) - 1
    area = np.zeros(M)
    cen = np.full((M, 2), np.nan)
    box = np.tile(np.array([np.inf, np.inf, -np.inf, -np.inf]), (M, 1))
    for g in range(M):
        v = _ring(verts, ring_off, g)
        n = len(v)
        if n == 0:
            continue
        box[g] = [v[:, 0].min(), v[:, 1].min(), v[:, 0].max(), v[:, 1].max()]
        cen[g] = v[0]
        if n < 3:
            continue
        x0, y0 = v[0]
        # sequential accumulation in float64 scalars: the kernel's order, not numpy's pairwise sum
        xs = (v[1:, 0] - x0).tolist()
        dy = (v[np.r_[2:n, 0], 1] - v[0:n - 1, 1]).tolist()
        s = 0.0
        for a, b in zip(xs, dy):
            s = s + a * b
        area[g] = s * 0.5
        ax, ay = v[1:n - 1, 0] - x0, v[1:n - 1, 1] - y0
        bx, by = v[2:n, 0] - x0, v[2:n, 1] - y0
        c = (ax * by - ay * bx).tolist()
        tx, ty = (ax + bx).tolist(), (ay + by).tolist()
        a2 = sx = sy = 0.0
        for ci, txi, tyi in zip(c, tx, ty):
            a2 = a2 + ci
            sx = sx + ci * txi
            sy = sy + ci * tyi
        if a2 != 0.0:
            den = 3.0 * a2
            cen[g] = [x0 + sx / den, y0 + sy / den]
    dist = np.sqrt(np.abs(area) / np.pi) * ratio
    return area, cen, box, dist


def _even_odd(ring: np.ndarray, px: np.ndarray, py: np.ndarray) -> np.ndarray:
    inside = np.zeros(px.size, dtype=bool)
    a = ring[-1]
    for b in ring:
        straddle = (a[1] > py) != (b[1] > py)
        with np.errstate(divide="ignore", invalid="ignore"):
            t = ((py - a[1]) * (b[0] - a[0])) / (b[1] - a[1])
            inside ^= straddle & (px < a[0] + t)
        a = b
    return inside


def ring_dist2_ref(ring: np.ndarray, px: np.ndarray, py: np.ndarray) -> np.ndarray:
    """Squared distance of every point to the ring, operation by operation as the kernel evaluates it."""
    best = np.full(px.size, np.inf)
    a = ring[-1]
    for b in ring:
        dx, dy = b[0] - a[0], b[1] - a[1]
        ex, ey = px - a[0], py - a[1]
        L = dx * dx + dy * dy
        if L > 0.0:
            t = np.minimum(np.maximum((ex * dx + ey * dy) / L, 0.0), 1.0)
        else:
            t = np.zeros(px.size)
        qx, qy = ex - t * dx, ey - t * dy
        best = np.minimum(best, qx * qx + qy * qy)
        a = b
    return best


def points_in_buffered_polygons_ref(points: np.ndarray, verts: np.ndarray, ring_off: np.ndarray,
                                    dist: np.ndarray) -> np.ndarray:
    """-> int32 [2, E] (row 0 = point, row 1 = polygon; point-major, polygons ascending) of the buffered join."""
    pts = np.asarray(points, dtype=np.float64)
    verts = np.asarray(verts, dtype=np.float64).reshape(-1, 2)
    dist = np.asarray(dist, dtype=np.float64)
    out_p, out_g = [], []
    for g in range(len(ring_off) - 1):
        ring = _ring(verts, ring_off, g)
        if len(ring) < 3:
            continue
        d = float(dist[g])
        grow = abs(d) * GROW
        lo, hi = ring.min(0), ring.max(0)
        cand = np.nonzero((pts[:, 0] >= lo[0] - grow) & (pts[:, 0] <= hi[0] + grow)
                          & (pts[:, 1] >= lo[1] - grow) & (pts[:, 1] <= hi[1] + grow))[0]
        if cand.size == 0:
            continue
        px, py = pts[cand, 0], pts[cand, 1]
        in_box = (px >= lo[0]) & (px <= hi[0]) & (py >= lo[1]) & (py <= hi[1])
        inside = in_box & _even_odd(ring, px, py)
        if d != 0.0:
            d2 = ring_dist2_ref(ring, px, py)
            inside = (inside | (d2 < d * d)) if d > 0.0 else (inside & (d2 > d * d))
        hit = cand[inside]
        out_p.append(hit)
        out_g.append(np.full(hit.size, g, dtype=np.int64))
    if not out_p:
        return np.zeros((2, 0), dtype=np.int32)
    p, g = np.concatenate(out_p), np.concatenate(out_g)
    order = np.lexsort((g, p))
    return np.stack([p[order], g[order]]).astype(np.int32)
