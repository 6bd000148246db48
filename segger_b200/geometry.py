"""B200-native point-in-polygon join for the prediction graph (SURVEY 8f row N2):
``points_in_polygons(points, polygons, predicate='contains')`` of /root/reference/src/segger/geometry/query.py:21-100
and the shape modes of ``setup_prediction_graph`` (/root/reference/src/segger/data/utils/neighbors.py:226-238), on
``sgb_pip_count`` / ``sgb_pip_fill`` instead of cuSpatial's quadtree join.  Polygons are passed as packed rings
(``verts`` [V,2] float64 + ``ring_off`` [M+1]).  Raw outlines (``Outlines``) are buffered on the device instead of
with geopandas (neighbors.py:229-231): ``sgb_polygon_props`` gives each ring's area and so its buffer distance, and
``sgb_pip_buffered_count`` / ``_fill`` join against the exact grown ring.  Outlines with holes or several parts use
the GeoArrow / cuSpatial polygon layout (``pack_polygons``: ``ring_off``, ``part_off``, ``geom_off``), joined by
``sgb_pip_multi_count`` / ``_fill`` and measured by ``sgb_polygon_props_multi``."""
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


def _part_rings(part) -> list:
    """The rings of one polygon part, exterior first: a shapely-like Polygon (``exterior.coords``, ``interiors``) or
    a sequence of [n, 2] rings."""
    if hasattr(part, "exterior"):
        if part.exterior is None:
            return []
        return [part.exterior.coords] + [ring.coords for ring in part.interiors]
    return list(part)


def _geom_parts(geom) -> list:
    """The parts of one geometry: a shapely-like Polygon / MultiPolygon (read through ``geom_type`` and ``geoms``), or
    a sequence of parts; None is a geometry with no parts."""
    if geom is None:
        return []
    kind = getattr(geom, "geom_type", None)
    if kind == "Polygon":
        return [geom]
    if kind == "MultiPolygon":
        return list(geom.geoms)
    if kind is not None:
        raise TypeError(f"pack_polygons: cannot pack a {kind}; expected a Polygon or a MultiPolygon")
    return list(geom)


def pack_polygons(geoms) -> Tuple[np.ndarray, np.ndarray, np.ndarray, np.ndarray]:
    """Geometries -> (verts [V,2] float64, ring_off [R+1], part_off [Q+1], geom_off [P+1] int64), the GeoArrow /
    cuSpatial polygon layout: ring r owns verts[ring_off[r]:ring_off[r+1]], part q rings part_off[q]:part_off[q+1]
    (its exterior, then its holes), geometry g parts geom_off[g]:geom_off[g+1].  Each geometry is either a
    shapely-like Polygon or MultiPolygon (only ``geom_type``, ``exterior.coords``, ``interiors`` and ``geoms`` are
    read; shapely is not imported) or nested sequences: parts -> rings -> [n, 2] vertices, exterior first."""
    rings, part_sizes, geom_sizes = [], [], []
    for geom in geoms:
        parts = _geom_parts(geom)
        geom_sizes.append(len(parts))
        for part in parts:
            pr = _part_rings(part)
            part_sizes.append(len(pr))
            rings.extend(np.asarray(r, dtype=np.float64).reshape(-1, 2) for r in pr)
    verts, ring_off = pack_rings(rings)
    part_off = np.zeros(len(part_sizes) + 1, dtype=np.int64)
    part_off[1:] = np.cumsum(part_sizes)
    geom_off = np.zeros(len(geom_sizes) + 1, dtype=np.int64)
    geom_off[1:] = np.cumsum(geom_sizes)
    return verts, ring_off, part_off, geom_off


def _check_layout(n_verts: int, ring_off, part_off, geom_off):
    """-> the three offset arrays as int64; ValueError unless each starts at 0, never decreases and ends at the length
    of the array it indexes (verts, rings, parts)."""
    out, n = [], n_verts
    for name, off in (("ring_off", ring_off), ("part_off", part_off), ("geom_off", geom_off)):
        off = np.ascontiguousarray(off, dtype=np.int64).reshape(-1)
        if off.size == 0 or off[0] != 0 or off[-1] != n or np.any(np.diff(off) < 0):
            raise ValueError(f"{name} must run from 0 to {n} without decreasing")
        out.append(off)
        n = off.size - 1
    return tuple(out)


def _ranges(starts: np.ndarray, counts: np.ndarray) -> np.ndarray:
    """Concatenation of arange(s, s + c) over (starts, counts)."""
    off = np.zeros(counts.size + 1, dtype=np.int64)
    off[1:] = np.cumsum(counts)
    return np.repeat(starts - off[:-1], counts) + np.arange(off[-1], dtype=np.int64)


def _take_geoms(verts, ring_off, part_off, geom_off, keep):
    """The geometries ``keep`` of a polygon layout, their parts and rings kept, renumbered from 0."""
    parts = _ranges(geom_off[keep], np.diff(geom_off)[keep])
    rings = _ranges(part_off[parts], np.diff(part_off)[parts])
    out = []
    for counts in (np.diff(ring_off)[rings], np.diff(part_off)[parts], np.diff(geom_off)[keep]):
        off = np.zeros(counts.size + 1, dtype=np.int64)
        off[1:] = np.cumsum(counts)
        out.append(off)
    return (verts[_ranges(ring_off[rings], np.diff(ring_off)[rings])], *out)


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
    between prediction tiles).  With ``part_off`` and ``geom_off`` (``pack_polygons``) the rings form geometries
    with holes and parts, one polygon id per geometry; without them every ring is one polygon."""

    def __init__(self, verts: np.ndarray, ring_off: np.ndarray, part_off=None, geom_off=None):
        self.verts = np.ascontiguousarray(verts, dtype=np.float64).reshape(-1, 2)
        self.multi = part_off is not None or geom_off is not None
        if self.multi:
            if part_off is None or geom_off is None:
                raise ValueError("PackedPolygons: part_off and geom_off go together")
            self.ring_off, self.part_off, self.geom_off = _check_layout(self.verts.shape[0], ring_off, part_off, geom_off)
            self.n_poly = len(self.geom_off) - 1
        else:
            self.ring_off = np.ascontiguousarray(ring_off, dtype=np.int64)
            self.n_poly = len(self.ring_off) - 1
        self.grid = _grid(self.verts, self.ring_off) if self.n_poly > 0 and self.verts.shape[0] > 0 else None
        self._dev = {}

    def on(self, device):
        """(verts, ring_off) on ``device``, and (part_off, geom_off) after them for a multi-part layout."""
        key = str(device)
        if key not in self._dev:
            arrs = (self.verts, self.ring_off) + ((self.part_off, self.geom_off) if self.multi else ())
            self._dev[key] = tuple(torch.from_numpy(a).to(device) for a in arrs)
        return self._dev[key]


class Outlines:
    """Raw, unbuffered cell / nucleus outlines, one ring each (``verts`` [V,2] float64, ``ring_off`` [M+1] int64, a
    closing duplicate of the first vertex tolerated), packed once per dataset.  ``boundary_type``: optional [M] array
    of per-ring labels ('cell' / 'nucleus', the reference's ``boundary_type`` column).  Outlines with holes or several
    parts pass ``part_off`` and ``geom_off`` as well (the layout of ``pack_polygons``); M is then the number of
    geometries, and ``boundary_type`` and every per-outline result are per geometry.

    ``areas()`` / ``centroids()`` are computed on the device (``sgb_polygon_props``, ``sgb_polygon_props_multi``);
    ``buffered(ratio)`` grows every outline by ``sqrt(|area| / pi) * ratio`` as the reference's geopandas buffer does
    (neighbors.py:229-231), exactly (a disc, not shapely's 16-chord approximation) -- pass its result to
    ``points_in_polygons``."""

    def __init__(self, verts: np.ndarray, ring_off: np.ndarray, boundary_type=None, part_off=None, geom_off=None):
        self.verts = np.ascontiguousarray(verts, dtype=np.float64).reshape(-1, 2)
        self.multi = part_off is not None or geom_off is not None
        if self.multi:
            if part_off is None or geom_off is None:
                raise ValueError("Outlines: part_off and geom_off go together")
            self.ring_off, self.part_off, self.geom_off = _check_layout(self.verts.shape[0], ring_off, part_off, geom_off)
            self.n_poly = len(self.geom_off) - 1
        else:
            self.ring_off = np.ascontiguousarray(ring_off, dtype=np.int64)
            self.n_poly = len(self.ring_off) - 1
            if self.n_poly < 0 or (self.n_poly > 0 and (self.ring_off[0] != 0 or self.ring_off[-1] != self.verts.shape[0]
                                                        or np.any(np.diff(self.ring_off) < 0))):
                raise ValueError("Outlines: ring_off must run from 0 to len(verts) without decreasing")
        self.boundary_type = None if boundary_type is None else np.asarray(boundary_type)
        if self.boundary_type is not None and self.boundary_type.shape != (self.n_poly,):
            raise ValueError(f"Outlines: boundary_type must have one entry per {'geometry' if self.multi else 'ring'} "
                             f"({self.n_poly}), got shape {self.boundary_type.shape}")
        self._dev, self._props, self._buffered, self._types = {}, {}, {}, {}

    def on(self, device):
        """(verts, ring_off) on ``device``, and (part_off, geom_off) after them for a multi-part layout."""
        key = str(device)
        if key not in self._dev:
            arrs = (self.verts, self.ring_off) + ((self.part_off, self.geom_off) if self.multi else ())
            self._dev[key] = tuple(torch.from_numpy(a).to(device) for a in arrs)
        return self._dev[key]

    def _device_props(self, device, ratio: float | None):
        """(area [M], centroid [M,2], box [M,4], dist [M] or None) device float64 tensors."""
        device = torch.device(device if device is not None else "cuda")
        d = self.on(device)
        M = self.n_poly
        area = torch.empty(M, dtype=torch.float64, device=device)
        cen = torch.empty(M, 2, dtype=torch.float64, device=device)
        box = torch.empty(M, 4, dtype=torch.float64, device=device)
        dist = torch.empty(M, dtype=torch.float64, device=device) if ratio is not None else None
        if self.multi:
            check(_lib.load().sgb_polygon_props_multi(*map(ptr, d), M, float(ratio or 0.0), ptr(area), ptr(cen), ptr(box),
                                                      ptr(dist), stream_ptr(device)), "polygon_props_multi")
        else:
            check(_lib.load().sgb_polygon_props(ptr(d[0]), ptr(d[1]), M, float(ratio or 0.0), ptr(area), ptr(cen), ptr(box),
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
        """[M] float64 signed ring areas (counter-clockwise > 0), computed on ``device``; for a multi-part layout the
        net area of each geometry (exteriors minus holes, >= 0)."""
        return self._host_props(device)[0]

    def centroids(self, device=None) -> np.ndarray:
        """[M, 2] float64 area-weighted centroids (a ring of zero area: its first vertex; an empty ring: NaN); for a
        multi-part layout the centroid of each geometry, holes subtracted."""
        return self._host_props(device)[1]

    def of_type(self, boundary_type: str) -> "Outlines":
        """The outlines labelled ``boundary_type``, renumbered from 0 in their original order (the reference's
        ``bd[bd.boundary_type == t].reset_index(drop=True)``), parts and holes kept; cached."""
        if self.boundary_type is None:
            raise ValueError("Outlines.of_type: these outlines carry no boundary_type")
        if boundary_type not in self._types and self.multi:
            keep = np.nonzero(self.boundary_type == boundary_type)[0]
            verts, ring_off, part_off, geom_off = _take_geoms(self.verts, self.ring_off, self.part_off, self.geom_off, keep)
            self._types[boundary_type] = Outlines(verts, ring_off, self.boundary_type[keep], part_off, geom_off)
        if boundary_type not in self._types:
            keep = np.nonzero(self.boundary_type == boundary_type)[0]
            sizes = np.diff(self.ring_off)[keep]
            off = np.zeros(keep.size + 1, dtype=np.int64)
            off[1:] = np.cumsum(sizes)
            idx = np.repeat(self.ring_off[keep] - off[:-1], sizes) + np.arange(off[-1], dtype=np.int64)
            self._types[boundary_type] = Outlines(self.verts[idx], off, self.boundary_type[keep])
        return self._types[boundary_type]

    def buffered(self, ratio: float, device=None) -> "BufferedOutlines":
        """Every outline grown by ``sqrt(|area| / pi) * ratio`` (shrunk for ratio < 0), ready for ``points_in_polygons``;
        built once per (ratio, device) and reused across prediction tiles."""
        device = torch.device(device if device is not None else "cuda")
        key = (float(ratio), str(device))
        if key not in self._buffered:
            self._buffered[key] = BufferedOutlines(self, self._device_props(device, float(ratio))[3])
        return self._buffered[key]


class BufferedOutlines:
    """``Outlines`` + one buffer distance per outline (``dist`` [M] float64; d > 0 grows the outline by d, d < 0
    shrinks it, d == 0 keeps it) + a grid over the grown boxes.  ``Outlines.buffered(ratio)`` builds the reference's
    distances ``sqrt(|area| / pi) * ratio``."""

    GROW = 1.0 + 2.0 ** -20          # boxes grow by |d| (1 + 2^-20): conservative under the rounding of the rim test

    def __init__(self, outlines: Outlines, dist):
        self.outlines, self.n_poly, self.multi = outlines, outlines.n_poly, outlines.multi
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
        keep = np.isfinite(box[:, 0])                     # empty outlines have the empty box
        g = (np.abs(d) * self.GROW)[keep, None]
        self.grid = _grid_from_boxes(box[keep, :2] - g, box[keep, 2:] + g)

    def on(self, device):
        """(verts, ring_off, dist) on ``device``; (verts, ring_off, part_off, geom_off, dist) for a multi-part layout."""
        key = str(device)
        if key not in self._dist:
            self._dist[key] = self.dist.to(device)
        return (*self.outlines.on(device), self._dist[key])


def points_in_polygons(points, verts, ring_off=None, device=None, device_output: bool = False) -> Tensor:
    """-> int32 [2, E] (index_query = point, index_match = polygon), strict containment, point-major order.
    ``points``: [N, 2] numpy / tensor (float32 or float64; device tensors are used in place); polygons either as
    (``verts``, ``ring_off``) arrays or as a ``PackedPolygons`` (pass it as ``verts``) -- both taken as already buffered
    -- or as the ``BufferedOutlines`` of ``Outlines.buffered`` (grown on the device).  A multi-part ``PackedPolygons``
    or ``BufferedOutlines`` (holes and parts, ``pack_polygons``) is joined per geometry: the even-odd rule over all of
    its rings, each point listed at most once per geometry."""
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
    dev = polys.on(device)
    d_dist = dev[-1] if buffered else None
    d_verts, d_off = dev[0], dev[1]
    ws = torch.empty(max(int(lib.sgb_pip_workspace_bytes(n, n_poly, nx, ny)), 16), dtype=torch.uint8, device=device)
    total = torch.zeros(1, dtype=torch.int32, device=device)
    f64 = int(pts.dtype == torch.float64)
    if polys.multi:
        d_part, d_geom = dev[2], dev[3]
        check(lib.sgb_pip_multi_count(ptr(pts), f64, n, ptr(d_verts), ptr(d_off), ptr(d_part), ptr(d_geom), ptr(d_dist), n_poly,
                                      xmin, ymin, cell, nx, ny, ptr(total), ptr(ws), ws.numel(), stream_ptr(device)),
              "pip_multi_count")
    elif buffered:
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
    if polys.multi:
        check(lib.sgb_pip_multi_fill(ptr(d_verts), ptr(d_off), ptr(d_part), ptr(d_geom), ptr(d_dist), n, n_poly, xmin, ymin,
                                     cell, nx, ny, E, ptr(out), E, ptr(ws), ws.numel(), ptr(scratch), scratch.numel(),
                                     stream_ptr(device)), "pip_multi_fill")
    elif buffered:
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
