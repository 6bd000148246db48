"""numpy restatement of quadtree tiling -- TEST INFRASTRUCTURE ONLY.  PARITY UNPINNED.

The reference tiles with ``QuadTreeTiling`` (data/tiling.py:198-235): cuSpatial quadtree leaves of <= 50,000 nodes over
all node positions (data_module.py:155,248-252), and ``TileFitDataset`` (data/tile_dataset.py:13-153) labels every node
with its tile and marks the nodes inside their tile shrunk by the margin, halving the margin for a tile that would vanish
(data/tiling.py:103-127).  Those modules import cuSpatial / geopandas and cannot run here, so the rules below are the
contract (segger_b200.tiles.QuadTreeTiling and sgb_quadtree.cu implement them, the tests compare bit for bit):

* Root and cells.  ``xmin, ymin`` = minimum over the points; ``side = max(xmax - xmin, ymax - ymin)`` (1.0 if 0);
  ``scale = side / 2**D`` with ``D = max_depth`` in 1..15.  Every cell edge is ``edge(c) = xmin + c * scale`` in fp64
  with integer ``c`` -- one formula for all levels, so neighbouring leaves share bit-identical edges.  A point's cell is
  ``floor((x - xmin) / scale)`` (inputs widened exactly to fp64), corrected by +-1 so that
  ``edge(ix) <= x < edge(ix + 1)``, clamped to ``[0, 2**D - 1]``.  A point lies in the closed box of its leaf.
* Leaves.  A quadrant at level ``L`` (root = 0) is split iff it holds more than ``max_tile_size`` points and ``L < D``.
  Tiles are the non-empty unsplit quadrants in Morton order (x in the even key bits).  A leaf at depth ``D`` may hold
  more than ``max_tile_size`` points (duplicates), as with cuSpatial.  The reference's retry loop on an invalid cuSpatial
  tree (geometry/quadtree.py:181-202) has no counterpart.
* Tile box = ``[edge(qx * 2**(D-L)), edge((qx + 1) * 2**(D-L))] x [same in y]``.
* Fit mask.  A node is in the mask iff it lies in its own tile's box shrunk by ``m_t`` on every side (closed), with
  ``m_t = margin / 2**j`` for the smallest ``j >= 0`` that leaves the shrunk box non-empty in both axes.
* Other points (e.g. ``bd`` nodes when the tree is built over transcripts): the same cell rule, then the leaf containing
  that cell; points outside the root clamp to the rim cells; a cell of an empty quadrant has no tile (-1).

Written as a plain recursive top-down split counting points per quadrant from integer cell coordinates -- independently of
the kernel's frontier-over-sorted-keys algorithm.
"""
from __future__ import annotations

from typing import List, Tuple

import numpy as np


def root_of(points: np.ndarray, max_depth: int) -> Tuple[float, float, float]:
    """-> (xmin, ymin, scale)."""
    p = np.asarray(points, dtype=np.float64).reshape(-1, 2)
    if p.shape[0] == 0:
        return 0.0, 0.0, 1.0 / float(2 ** max_depth)
    xmin, ymin = float(p[:, 0].min()), float(p[:, 1].min())
    side = max(float(p[:, 0].max()) - xmin, float(p[:, 1].max()) - ymin)
    if not side > 0.0:
        side = 1.0
    return xmin, ymin, side / float(2 ** max_depth)


def cells(v: np.ndarray, lo: float, scale: float, max_depth: int) -> np.ndarray:
    """Cell index along one axis (fp64; the +-1 correction makes edge(c) <= v < edge(c + 1) exact)."""
    nc = 2 ** max_depth
    v = np.asarray(v, dtype=np.float64)
    f = np.clip(np.floor((v - lo) / scale), -1.0, float(nc))
    c = f.astype(np.int64)
    below = v < lo + c.astype(np.float64) * scale
    above = v >= lo + (c + 1).astype(np.float64) * scale
    c = np.where(below, c - 1, np.where(above, c + 1, c))
    return np.clip(c, 0, nc - 1)


def build(points: np.ndarray, max_tile_size: int = 50_000, max_depth: int = 15):
    """-> dict(labels int32 [N], boxes fp64 [P, 4], counts [P], levels [P], qx [P], qy [P], root (xmin, ymin, scale))."""
    if not 1 <= max_depth <= 15:
        raise ValueError("max_depth must be in 1..15")
    p = np.asarray(points, dtype=np.float64).reshape(-1, 2)
    D = max_depth
    xmin, ymin, scale = root_of(p, D)
    ix, iy = cells(p[:, 0], xmin, scale, D), cells(p[:, 1], ymin, scale, D)
    labels = np.full(p.shape[0], -1, dtype=np.int32)
    leaves: List[Tuple[int, int, int, int]] = []          # (level, qx, qy, count)

    def visit(level: int, qx: int, qy: int, idx: np.ndarray) -> None:
        if idx.size == 0:
            return
        if idx.size > max_tile_size and level < D:
            sh = D - level - 1
            bx, by = (ix[idx] >> sh) & 1, (iy[idx] >> sh) & 1
            for cy in (0, 1):                               # Morton order: (0,0), (1,0), (0,1), (1,1)
                for cx in (0, 1):
                    visit(level + 1, 2 * qx + cx, 2 * qy + cy, idx[(bx == cx) & (by == cy)])
            return
        labels[idx] = len(leaves)
        leaves.append((level, qx, qy, idx.size))

    visit(0, 0, 0, np.arange(p.shape[0]))
    lv = np.array([l[0] for l in leaves], dtype=np.int64)
    qx = np.array([l[1] for l in leaves], dtype=np.int64)
    qy = np.array([l[2] for l in leaves], dtype=np.int64)
    span = np.left_shift(np.int64(1), D - lv) if len(leaves) else np.zeros(0, np.int64)
    edge = lambda lo, c: lo + c.astype(np.float64) * scale      # noqa: E731
    boxes = np.stack([edge(xmin, qx * span), edge(ymin, qy * span), edge(xmin, (qx + 1) * span),
                      edge(ymin, (qy + 1) * span)], 1) if len(leaves) else np.zeros((0, 4))
    return dict(labels=labels, boxes=boxes, counts=np.array([l[3] for l in leaves], dtype=np.int64), levels=lv, qx=qx, qy=qy,
                root=(xmin, ymin, scale), max_depth=D)


def label(tree: dict, points: np.ndarray) -> np.ndarray:
    """Leaf containing each point's cell (-1: an empty quadrant), by descending level by level."""
    p = np.asarray(points, dtype=np.float64).reshape(-1, 2)
    D = tree["max_depth"]
    xmin, ymin, scale = tree["root"]
    ix, iy = cells(p[:, 0], xmin, scale, D), cells(p[:, 1], ymin, scale, D)
    out = np.full(p.shape[0], -1, dtype=np.int32)
    for L in range(D + 1):
        at = np.nonzero(tree["levels"] == L)[0]
        if at.size == 0:
            continue
        table = {(int(tree["qx"][i]), int(tree["qy"][i])): i for i in at}
        sh = D - L
        for j in np.nonzero(out < 0)[0]:
            hit = table.get((int(ix[j] >> sh), int(iy[j] >> sh)))
            if hit is not None:
                out[j] = hit
    return out


def margins(boxes: np.ndarray, margin: float) -> np.ndarray:
    """Per-tile margin: ``margin / 2**j``, smallest j >= 0 with the shrunk box non-empty in both axes."""
    out = []
    for x0, y0, x1, y1 in np.asarray(boxes, dtype=np.float64).reshape(-1, 4).tolist():
        m = float(margin)
        while m > 0.0 and not (x0 + m <= x1 - m and y0 + m <= y1 - m):
            m = m / 2.0
        out.append(m)
    return np.array(out, dtype=np.float64)


def fit_mask(tree: dict, points: np.ndarray, labels: np.ndarray, margin: float) -> np.ndarray:
    """Inside the own tile's box shrunk by that tile's margin (closed); False without a tile."""
    p = np.asarray(points, dtype=np.float64).reshape(-1, 2)
    m = margins(tree["boxes"], margin)
    out = np.zeros(p.shape[0], dtype=bool)
    ok = labels >= 0
    b, mm = tree["boxes"][labels[ok]], m[labels[ok]]
    x, y = p[ok, 0], p[ok, 1]
    out[ok] = (x >= b[:, 0] + mm) & (x <= b[:, 2] - mm) & (y >= b[:, 1] + mm) & (y <= b[:, 3] - mm)
    return out
