"""B200-native point-in-polygon join for the prediction graph (SURVEY 8f row N2):
``points_in_polygons(points, polygons, predicate='contains')`` of /root/reference/src/segger/geometry/query.py:21-100
and the shape modes of ``setup_prediction_graph`` (/root/reference/src/segger/data/utils/neighbors.py:226-238), on
``sgb_pip_count`` / ``sgb_pip_fill`` instead of cuSpatial's quadtree join.  Polygons are passed as packed rings
(``verts`` [V,2] float64 + ``ring_off`` [M+1]).  Raw outlines (``Outlines``) are buffered on the device instead of
with geopandas (neighbors.py:229-231): ``sgb_polygon_props`` gives each ring's area and so its buffer distance, and
``sgb_pip_buffered_count`` / ``_fill`` join against the exact grown ring."""
from __future__ import annotations

import ctypes as C
from typing import Tuple

import numpy as np
import torch
from torch import Tensor

from . import _lib, ops
from ._lib import check, ptr, stream_ptr


def pack_rings(rings) -> Tuple[np.ndarray, np.ndarray]:
    """list of [n_i, 2] arrays -> (verts [V,2] float64, ring_off [M+1] int64)."""
    off = np.zeros(len(rings) + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(r) for r in rings])
    verts = np.concatenate([np.asarray(r, dtype=np.float64).reshape(-1, 2) for r in rings]) if rings else np.zeros((0, 2))
    return np.ascontiguousarray(verts, dtype=np.float64), off


def _grid(verts: np.ndarray, ring_off: np.ndarray):
    """Uniform grid over the polygons' bounding box, cell ~ the median polygon extent (host side: the rings come from
    host geometry anyway); capped at 2^26 cells."""
    sizes = np.diff(ring_off)
    starts = ring_off[:-1][sizes > 0]
    # per-ring boxes with reduceat (rings are contiguous runs; empty rings are skipped), then the union box
    mx = np.maximum.reduceat(verts, starts, axis=0)
    mn = np.minimum.reduceat(verts, starts, axis=0)
    return _grid_from_boxes(mn, mx)


def _grid_from_boxes(mn: np.ndarray, mx: np.ndarray):
    """The grid of ``_grid`` from per-ring box corners [k, 2] (non-empty rings only)."""
    ext = mx - mn
    lo = np.array([mn[:, 0].min(), mn[:, 1].min()])
    hi = np.array([mx[:, 0].max(), mx[:, 1].max()])
    cell = float(max(np.median(ext.max(1)), 1e-9))
    span = np.maximum(hi - lo, cell)
    while (np.floor(span[0] / cell) + 1) * (np.floor(span[1] / cell) + 1) >= 2 ** 26:
        cell *= 2.0
    nx, ny = int(np.floor(span[0] / cell)) + 1, int(np.floor(span[1] / cell)) + 1
    return float(lo[0]), float(lo[1]), cell, nx, ny


class PackedPolygons:
    """Rings + their grid + device copies, built once per boundary set (the outlines of a dataset do not change
    between prediction tiles)."""

    def __init__(self, verts: np.ndarray, ring_off: np.ndarray):
        self.verts = np.ascontiguousarray(verts, dtype=np.float64).reshape(-1, 2)
        self.ring_off = np.ascontiguousarray(ring_off, dtype=np.int64)
        self.n_poly = len(self.ring_off) - 1
        self.grid = _grid(self.verts, self.ring_off) if self.n_poly > 0 and self.verts.shape[0] > 0 else None
        self._dev = {}

    def on(self, device):
        key = str(device)
        if key not in self._dev:
            self._dev[key] = (torch.from_numpy(self.verts).to(device), torch.from_numpy(self.ring_off).to(device))
        return self._dev[key]


class Outlines:
    """Raw, unbuffered cell / nucleus outlines, one ring each (``verts`` [V,2] float64, ``ring_off`` [M+1] int64, a
    closing duplicate of the first vertex tolerated), packed once per dataset.  ``boundary_type``: optional [M] array
    of per-ring labels ('cell' / 'nucleus', the reference's ``boundary_type`` column).

    ``areas()`` / ``centroids()`` are computed on the device (``sgb_polygon_props``); ``buffered(ratio)`` grows every
    ring by ``sqrt(|area| / pi) * ratio`` as the reference's geopandas buffer does (neighbors.py:229-231), exactly
    (a disc, not shapely's 16-chord approximation) -- pass its result to ``points_in_polygons``."""

    def __init__(self, verts: np.ndarray, ring_off: np.ndarray, boundary_type=None):
        self.verts = np.ascontiguousarray(verts, dtype=np.float64).reshape(-1, 2)
        self.ring_off = np.ascontiguousarray(ring_off, dtype=np.int64)
        self.n_poly = len(self.ring_off) - 1
        if self.n_poly < 0 or (self.n_poly > 0 and (self.ring_off[0] != 0 or self.ring_off[-1] != self.verts.shape[0]
                                                    or np.any(np.diff(self.ring_off) < 0))):
            raise ValueError("Outlines: ring_off must run from 0 to len(verts) without decreasing")
        self.boundary_type = None if boundary_type is None else np.asarray(boundary_type)
        if self.boundary_type is not None and self.boundary_type.shape != (self.n_poly,):
            raise ValueError(f"Outlines: boundary_type must have one entry per ring ({self.n_poly}), "
                             f"got shape {self.boundary_type.shape}")
        self._dev, self._props, self._buffered, self._types = {}, {}, {}, {}

    def on(self, device):
        key = str(device)
        if key not in self._dev:
            self._dev[key] = (torch.from_numpy(self.verts).to(device), torch.from_numpy(self.ring_off).to(device))
        return self._dev[key]

    def _device_props(self, device, ratio: float | None):
        """(area [M], centroid [M,2], box [M,4], dist [M] or None) device float64 tensors."""
        device = torch.device(device if device is not None else "cuda")
        d_verts, d_off = self.on(device)
        M = self.n_poly
        area = torch.empty(M, dtype=torch.float64, device=device)
        cen = torch.empty(M, 2, dtype=torch.float64, device=device)
        box = torch.empty(M, 4, dtype=torch.float64, device=device)
        dist = torch.empty(M, dtype=torch.float64, device=device) if ratio is not None else None
        check(_lib.load().sgb_polygon_props(ptr(d_verts), ptr(d_off), M, float(ratio or 0.0), ptr(area), ptr(cen), ptr(box),
                                            ptr(dist), stream_ptr(device)), "polygon_props")
        ops._count(1)
        return area, cen, box, dist

    def _host_props(self, device=None):
        key = str(device)
        if key not in self._props:
            area, cen, _, _ = self._device_props(device, None)
            self._props[key] = (area.cpu().numpy(), cen.cpu().numpy())
        return self._props[key]

    def areas(self, device=None) -> np.ndarray:
        """[M] float64 signed ring areas (counter-clockwise > 0), computed on ``device``."""
        return self._host_props(device)[0]

    def centroids(self, device=None) -> np.ndarray:
        """[M, 2] float64 area-weighted centroids (a ring of zero area: its first vertex; an empty ring: NaN)."""
        return self._host_props(device)[1]

    def of_type(self, boundary_type: str) -> "Outlines":
        """The rings labelled ``boundary_type``, renumbered from 0 in their original order (the reference's
        ``bd[bd.boundary_type == t].reset_index(drop=True)``); cached."""
        if self.boundary_type is None:
            raise ValueError("Outlines.of_type: these outlines carry no boundary_type")
        if boundary_type not in self._types:
            keep = np.nonzero(self.boundary_type == boundary_type)[0]
            sizes = np.diff(self.ring_off)[keep]
            off = np.zeros(keep.size + 1, dtype=np.int64)
            off[1:] = np.cumsum(sizes)
            idx = np.repeat(self.ring_off[keep] - off[:-1], sizes) + np.arange(off[-1], dtype=np.int64)
            self._types[boundary_type] = Outlines(self.verts[idx], off, self.boundary_type[keep])
        return self._types[boundary_type]

    def buffered(self, ratio: float, device=None) -> "BufferedOutlines":
        """Every ring grown by ``sqrt(|area| / pi) * ratio`` (shrunk for ratio < 0), ready for ``points_in_polygons``;
        built once per (ratio, device) and reused across prediction tiles."""
        device = torch.device(device if device is not None else "cuda")
        key = (float(ratio), str(device))
        if key not in self._buffered:
            self._buffered[key] = BufferedOutlines(self, self._device_props(device, float(ratio))[3])
        return self._buffered[key]


class BufferedOutlines:
    """``Outlines`` + one buffer distance per ring (``dist`` [M] float64; d > 0 grows the ring by d, d < 0 shrinks
    it, d == 0 keeps it) + a grid over the grown boxes.  ``Outlines.buffered(ratio)`` builds the reference's
    distances ``sqrt(|area| / pi) * ratio``."""

    GROW = 1.0 + 2.0 ** -20          # boxes grow by |d| (1 + 2^-20): conservative under the rounding of the rim test

    def __init__(self, outlines: Outlines, dist):
        self.outlines, self.n_poly = outlines, outlines.n_poly
        dist = torch.as_tensor(dist, dtype=torch.float64)
        if dist.shape != (self.n_poly,):
            raise ValueError(f"BufferedOutlines: dist must have one entry per ring ({self.n_poly}), got {tuple(dist.shape)}")
        device = dist.device if dist.is_cuda else torch.device("cuda")
        self.dist = dist.to(device).contiguous()
        self._dist = {str(device): self.dist}
        self.grid = None
        if self.n_poly == 0 or outlines.verts.shape[0] == 0:
            return
        box = outlines._device_props(device, None)[2].cpu().numpy()
        d = self.dist.cpu().numpy()
        keep = np.isfinite(box[:, 0])                     # empty rings have the empty box
        g = (np.abs(d) * self.GROW)[keep, None]
        self.grid = _grid_from_boxes(box[keep, :2] - g, box[keep, 2:] + g)

    def on(self, device):
        """(verts, ring_off, dist) on ``device``."""
        key = str(device)
        if key not in self._dist:
            self._dist[key] = self.dist.to(device)
        return (*self.outlines.on(device), self._dist[key])


def points_in_polygons(points, verts, ring_off=None, device=None, device_output: bool = False) -> Tensor:
    """-> int32 [2, E] (index_query = point, index_match = polygon), strict containment, point-major order.
    ``points``: [N, 2] numpy / tensor (float32 or float64; device tensors are used in place); polygons either as
    (``verts``, ``ring_off``) arrays or as a ``PackedPolygons`` (pass it as ``verts``) -- both taken as already buffered
    -- or as the ``BufferedOutlines`` of ``Outlines.buffered`` (grown on the device)."""
    device = torch.device(device if device is not None else "cuda")
    buffered = isinstance(verts, BufferedOutlines)
    polys = verts if isinstance(verts, (PackedPolygons, BufferedOutlines)) else PackedPolygons(verts, ring_off)
    n_poly = polys.n_poly
    if isinstance(points, np.ndarray):
        pts = torch.from_numpy(np.ascontiguousarray(points if points.dtype in (np.float32, np.float64)
                                                    else points.astype(np.float64)))
    else:
        pts = points if points.dtype in (torch.float32, torch.float64) else points.double()
    pts = pts.to(device).contiguous()
    n = pts.size(0)
    empty = torch.zeros(2, 0, dtype=torch.int32, device=device if device_output else "cpu")
    if n == 0 or polys.grid is None:
        return empty
    xmin, ymin, cell, nx, ny = polys.grid
    lib = _lib.load()
    if buffered:
        d_verts, d_off, d_dist = polys.on(device)
    else:
        d_verts, d_off = polys.on(device)
    ws = torch.empty(max(int(lib.sgb_pip_workspace_bytes(n, n_poly, nx, ny)), 16), dtype=torch.uint8, device=device)
    total = torch.zeros(1, dtype=torch.int32, device=device)
    f64 = int(pts.dtype == torch.float64)
    if buffered:
        check(lib.sgb_pip_buffered_count(ptr(pts), f64, n, ptr(d_verts), ptr(d_off), ptr(d_dist), n_poly, xmin, ymin, cell, nx,
                                         ny, ptr(total), ptr(ws), ws.numel(), stream_ptr(device)), "pip_buffered_count")
    else:
        check(lib.sgb_pip_count(ptr(pts), f64, n, ptr(d_verts), ptr(d_off), n_poly, xmin, ymin, cell, nx, ny, ptr(total),
                                ptr(ws), ws.numel(), stream_ptr(device)), "pip_count")
    E = int(total.item())
    ops._count(12)
    if E == 0:
        return empty
    out = torch.empty(2, E, dtype=torch.int32, device=device)
    scratch = torch.empty(int(lib.sgb_pip_fill_scratch_bytes(E)), dtype=torch.uint8, device=device)
    if buffered:
        check(lib.sgb_pip_buffered_fill(ptr(d_verts), ptr(d_off), ptr(d_dist), n, n_poly, xmin, ymin, cell, nx, ny, E, ptr(out),
                                        E, ptr(ws), ws.numel(), ptr(scratch), scratch.numel(), stream_ptr(device)),
              "pip_buffered_fill")
    else:
        check(lib.sgb_pip_fill(ptr(d_verts), ptr(d_off), n, n_poly, xmin, ymin, cell, nx, ny, E, ptr(out), E, ptr(ws),
                               ws.numel(), ptr(scratch), scratch.numel(), stream_ptr(device)), "pip_fill")
    ops._count(12)
    return out if device_output else out.cpu()


def setup_prediction_graph(points, verts, ring_off=None, device=None) -> Tensor:
    """Round-1 entry point for already-buffered outlines; the drop-in with the reference's signature is
    ``segger_b200.neighbors.setup_prediction_graph(tx, bd, max_k, buffer_ratio, mode)``."""
    return points_in_polygons(points, verts, ring_off, device=device, device_output=False)
