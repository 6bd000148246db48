"""Device-side tiling of a heterogeneous graph (SURVEY.md 8f rows N2 second half and N3).

What the reference does on the host, per tile and per attribute, between the kernels of the hot path:

* ``PartitionDataset`` (/root/reference/src/segger/data/partition/dataset.py:375-579): permute nodes so that every
  tile is contiguous, renumber / sort the edges by tile and DROP edges between tiles (:483-494), slice a tile out
  (``__getitem__``, :512-579); the PyG ``DataLoader`` then collates the tiles of a batch;
* ``PartitionSampler`` (data/partition/sampler.py:11-82,186-282,292-405): best-fit-decreasing (or shuffled first-fit)
  packing of tiles into batches of <= ``max_num`` edges;
* ``TilePredictDataset._subset`` (data/tile_dataset.py:218-246): nodes inside the tile grown by ``margin`` +
  ``HeteroData.subgraph`` + ``predict_mask`` = inside the tile itself.

Here the graph stays on the GPU as a ``HeteroBatch`` and every step is a kernel of ``sgb_tiles.cu`` (stable radix
sort, flag / scan / scatter selections, range gathers): a batch is assembled with a handful of launches and at most
one small device->host read (the selection counts of a prediction tile).  Batches produced here carry tagged
``batch`` vectors (``ist_encoder.set_num_graphs``) and pre-validated edges, so the forward runs without any stream
synchronisation and can be captured in a CUDA graph.
"""
from __future__ import annotations

import bisect
import ctypes as C
import random
from typing import Dict, List, Optional, Sequence, Tuple

import torch
from torch import Tensor

from . import _lib, ops
from ._lib import check, ptr, require_cuda, stream_ptr
from .hetero import HeteroBatch
from .ist_encoder import set_num_graphs

EdgeType = Tuple[str, str, str]


# ---------------------------------------------------------------------------------------------------------------------
# bin packing (host; a few hundred tiles)
# ---------------------------------------------------------------------------------------------------------------------
def _check_items(items: Sequence[float], capacity: float, skip_too_big: bool) -> List[Tuple[float, int]]:
    if skip_too_big:
        return [(v, i) for i, v in enumerate(items) if 0 < v <= capacity]
    if not all(0 < v <= capacity for v in items):
        raise ValueError("All items must be > 0 and <= bin_capacity.")
    return [(v, i) for i, v in enumerate(items)]


def best_fit_decreasing(items: Sequence[float], bin_capacity: float, skip_too_big: bool = False) -> List[List[int]]:
    """sampler.py:11-82: items in decreasing size, each into the open bin it fills most tightly (lowest bin index among
    equals), a new bin when none fits.  Returns bins of original item indices."""
    todo = sorted(_check_items(items, bin_capacity, skip_too_big), key=lambda t: t[0], reverse=True)   # stable, like list.sort
    bins: List[List[int]] = []
    free: List[Tuple[float, int]] = []          # (remaining capacity, bin index), kept sorted
    for size, idx in todo:
        k = bisect.bisect_left(free, (size, -1))
        if k == len(free):
            bins.append([idx])
            bisect.insort(free, (bin_capacity - size, len(bins) - 1))
        else:
            rem, b = free.pop(k)                 # smallest remaining capacity that still fits; ties -> lowest bin index
            bins[b].append(idx)
            bisect.insort(free, (rem - size, b))
    return bins


def first_fit_shuffled(items: Sequence[float], bin_capacity: float, skip_too_big: bool = False,
                       rng: Optional[random.Random] = None) -> List[List[int]]:
    """sampler.py:186-282 as ``PartitionSampler`` calls it for ``shuffle=True`` (``n_buckets=1``): sort decreasing,
    shuffle everything with ``rng`` (the global ``random`` by default), then first fit."""
    rng = rng or random
    todo = sorted(_check_items(items, bin_capacity, skip_too_big), key=lambda t: t[0], reverse=True)
    if len(todo) > 1:
        rng.shuffle(todo)
    bins: List[List[int]] = []
    left: List[float] = []
    for size, idx in todo:
        for b, cap in enumerate(left):
            if cap >= size:
                bins[b].append(idx)
                left[b] -= size
                break
        else:
            bins.append([idx])
            left.append(bin_capacity - size)
    return bins


# ---------------------------------------------------------------------------------------------------------------------
# thin kernel wrappers
# ---------------------------------------------------------------------------------------------------------------------
def _i32(n: int, device) -> Tensor:
    return torch.empty(n, dtype=torch.int32, device=device)


def stable_argsort(labels: Tensor, n_values: int) -> Tuple[Tensor, Tensor, Tensor]:
    """-> (perm int32 [n], indptr int32 [n_values + 1], status int32 [1]) of ``PartitionDataset._get_permutation``."""
    require_cuda(labels)
    if labels.dtype not in (torch.int32, torch.int64):
        labels = labels.long()
    labels = labels.contiguous()
    n, dev = labels.numel(), labels.device
    lib = _lib.load()
    perm, indptr = _i32(n, dev), _i32(n_values + 1, dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    ws = ops._ws(lib.sgb_argsort_workspace_bytes(n), dev)
    check(lib.sgb_argsort_stable(ptr(labels), labels.element_size(), n, n_values, ptr(perm), ptr(indptr), ptr(status), ptr(ws),
                                 ws.numel(), stream_ptr(dev)), "argsort_stable")
    ops._count(8)
    return perm, indptr, status


def gather_rows(attr: Tensor, sel: Tensor, count: Optional[Tensor] = None, m: Optional[int] = None) -> Tensor:
    """attr[sel[:m]] along dim 0 for any dtype / trailing shape (rows of the worst-case size ``m`` are allocated; with a
    device ``count`` only the first ``count`` are written)."""
    attr = attr.contiguous()
    m = sel.numel() if m is None else m
    out = torch.empty((m,) + tuple(attr.shape[1:]), dtype=attr.dtype, device=attr.device)
    row_elems = 1
    for d in attr.shape[1:]:
        row_elems *= int(d)
    row_bytes = attr.element_size() * row_elems
    if m > 0 and attr.size(0) > 0:
        a = attr.view(torch.uint8) if attr.dtype == torch.bool else attr
        o = out.view(torch.uint8) if out.dtype == torch.bool else out
        check(_lib.load().sgb_gather_rows_bytes(ptr(a), row_bytes, ptr(sel), ptr(count), m, ptr(o), stream_ptr(attr.device)),
              "gather_rows_bytes")
        ops._count(1)
    return out


def _dev_i64(values: Sequence[int], device) -> Tensor:
    return torch.tensor(list(values), dtype=torch.int64).to(device, non_blocking=True)


# ---------------------------------------------------------------------------------------------------------------------
# quadtree tiles (QuadTreeTiling + TileFitDataset labels / masks)
# ---------------------------------------------------------------------------------------------------------------------
def _pos_arg(pos: Tensor) -> Tensor:
    require_cuda(pos)
    if pos.dim() != 2 or pos.size(1) != 2:
        raise ValueError(f"positions must be [N, 2], got {tuple(pos.shape)}")
    return (pos if pos.dtype in (torch.float32, torch.float64) else pos.float()).contiguous()


def fit_margins(boxes: Tensor, margin: float) -> Tensor:
    """Per-tile training margin (data/tiling.py:103-127): ``margin / 2**j`` with the smallest ``j >= 0`` that leaves the
    box shrunk by it non-empty in both axes.  fp64 on the host, once per tiling; returned on the boxes' device."""
    b = boxes.detach().to("cpu", torch.float64)
    m = torch.full((b.size(0),), float(margin), dtype=torch.float64)
    while True:
        bad = (m > 0) & ~((b[:, 0] + m <= b[:, 2] - m) & (b[:, 1] + m <= b[:, 3] - m))
        if not bool(bad.any()):
            return m.to(boxes.device)
        m = torch.where(bad, m / 2, m)


class QuadTreeTiling:
    """``QuadTreeTiling`` (data/tiling.py:198-235) without cuSpatial: quadtree leaves holding <= ``max_tile_size`` points
    over ``positions`` -- an [N, 2] fp32 / fp64 CUDA tensor, or a dict of them per node type (all node positions, as
    the reference builds it).  Rules in oracle/quadtree_ref.py; built by sgb_quadtree.cu with one device->host read
    (the tile count).

    ``tiles``: [P, 4] fp64 boxes (xmin, ymin, xmax, ymax) in Morton order; ``labels``: int32 tile of every input point
    (a dict when ``positions`` is); ``counts``: int32 points per tile; ``label(points)``: the tile of other points."""

    def __init__(self, positions, max_tile_size: int = 50_000, max_depth: int = 15):
        if not 1 <= int(max_depth) <= 15:
            raise ValueError(f"max_depth must be in 1..15, got {max_depth}")
        if int(max_tile_size) < 1:
            raise ValueError(f"max_tile_size must be >= 1, got {max_tile_size}")
        self.max_tile_size, self.max_depth = int(max_tile_size), int(max_depth)
        named = isinstance(positions, dict)
        parts = {k: _pos_arg(v) for k, v in positions.items()} if named else {None: _pos_arg(positions)}
        if not parts:
            raise ValueError("QuadTreeTiling: no positions")
        dtypes = {p.dtype for p in parts.values()}
        dt = torch.float64 if len(dtypes) > 1 else dtypes.pop()               # widening to fp64 is exact
        pos = torch.cat([p.to(dt) for p in parts.values()]) if len(parts) > 1 else next(iter(parts.values()))
        n, dev = pos.size(0), pos.device
        lib = _lib.load()
        cap = max(1, int(lib.sgb_quadtree_max_leaves(n, self.max_tile_size, self.max_depth)))
        labels = _i32(n, dev)
        self.root = torch.empty(3, dtype=torch.float64, device=dev)           # (xmin, ymin, scale)
        meta = torch.empty(cap, 3, dtype=torch.int32, device=dev)
        boxes = torch.empty(cap, 4, dtype=torch.float64, device=dev)
        n_leaves = torch.zeros(1, dtype=torch.int32, device=dev)
        ws = ops._ws(lib.sgb_quadtree_workspace_bytes(n, self.max_tile_size, self.max_depth), dev)
        check(lib.sgb_quadtree_build(ptr(pos), int(pos.dtype == torch.float64), n, self.max_tile_size, self.max_depth,
                                     ptr(labels), ptr(self.root), ptr(meta), ptr(boxes), cap, ptr(n_leaves), ptr(ws), ws.numel(),
                                     stream_ptr(dev)), "quadtree_build")
        ops._count(6 + self.max_depth + 12)                                   # + the radix sort's and the scan's launches
        P = int(n_leaves.item())                                              # the one read-back
        self._meta = meta[:P]
        self.tiles = boxes[:P]
        self.counts = self._meta[:, 2]
        if named:
            self.labels, o = {}, 0
            for k, p in parts.items():
                self.labels[k] = labels[o:o + p.size(0)]
                o += p.size(0)
        else:
            self.labels = labels

    def __len__(self) -> int:
        return self.tiles.size(0)

    @property
    def levels(self) -> Tensor:
        return self._meta[:, 1]

    def label(self, points: Tensor) -> Tensor:
        """int32 tile of each point: the leaf containing its cell (points outside the root clamp to the rim cells);
        -1 for a cell of an empty quadrant."""
        pts = _pos_arg(points)
        out = _i32(pts.size(0), pts.device)
        check(_lib.load().sgb_quadtree_label(ptr(pts), int(pts.dtype == torch.float64), pts.size(0), ptr(self.root), self.max_depth,
                                             ptr(self._meta), len(self), ptr(out), stream_ptr(pts.device)), "quadtree_label")
        ops._count(1)
        return out

    def fit_labels_and_masks(self, data: HeteroBatch, margin: float) -> Tuple[Dict[str, Tensor], Dict[str, Tensor]]:
        """``TileFitDataset``: per node type the tile label (``TilePartition(data, labels, len(self))``) and the training
        ``mask`` ``LitISTEncoder.get_losses`` reads = inside the own tile shrunk by the tile's margin (halved until the
        shrunk tile is non-empty).  Nodes whose cell lies in an empty quadrant get label -1 and mask False."""
        lib = _lib.load()
        margins = fit_margins(self.tiles, margin)
        labels, masks = {}, {}
        for nt in data.node_types:
            pos = _pos_arg(data[nt]["pos"])
            lab = self.label(pos)
            mask = torch.empty(pos.size(0), dtype=torch.bool, device=pos.device)
            check(lib.sgb_quadtree_fit_mask(ptr(pos), int(pos.dtype == torch.float64), pos.size(0), ptr(lab), ptr(self.tiles),
                                            ptr(margins), len(self), ptr(mask.view(torch.uint8)), stream_ptr(pos.device)),
                  "quadtree_fit_mask")
            ops._count(1)
            labels[nt], masks[nt] = lab, mask
        return labels, masks


# ---------------------------------------------------------------------------------------------------------------------
# training tiles: partition once, slice / collate per batch
# ---------------------------------------------------------------------------------------------------------------------
class TilePartition:
    """``PartitionDataset`` for a ``HeteroBatch`` that lives on the GPU.

    ``labels[node_type]`` assigns every node to a tile in ``[0, n_tiles)``.  After construction ``self.data`` holds
    the permuted graph (tile-contiguous nodes, edges sorted by tile, inter-tile edges dropped) and
    ``node_indptr[type]`` / ``edge_indptr[edge_type]`` (host lists) delimit the tiles.  The reference's
    ``torch.argsort`` is not stable; here members of a tile keep their original relative order.
    """

    def __init__(self, data: HeteroBatch, labels: Dict[str, Tensor], n_tiles: int):
        self.n_tiles = int(n_tiles)
        self.node_perm: Dict[str, Tensor] = {}
        self.node_indptr: Dict[str, List[int]] = {}
        self.edge_indptr: Dict[EdgeType, List[int]] = {}
        lib = _lib.load()
        out = HeteroBatch()
        inv, lab = {}, {}
        statuses, ptrs = [], []
        for nt in data.node_types:
            store = data[nt]
            l = labels[nt]
            require_cuda(l)
            l = (l if l.dtype in (torch.int32, torch.int64) else l.long()).contiguous()
            perm, indptr, status = stable_argsort(l, self.n_tiles)
            n = l.numel()
            iv = _i32(n, l.device)
            check(lib.sgb_invert_permutation(ptr(perm), n, ptr(iv), stream_ptr(l.device)), "invert_permutation")
            ops._count(1)
            self.node_perm[nt], inv[nt], lab[nt] = perm, iv, l
            statuses.append(status)
            ptrs.append(indptr)
            for name, attr in store.items():
                out[nt][name] = gather_rows(attr, perm) if isinstance(attr, Tensor) and attr.dim() >= 1 and attr.size(0) == n else attr
        edge_ptrs = []
        for et in data.edge_types:
            src, _, dst = et
            ei = data[et]["edge_index"]
            require_cuda(ei)
            E = ei.size(1)
            dev = ei.device
            new_ei = torch.empty(2, E, dtype=ei.dtype, device=dev)
            kept = _i32(E, dev)
            rowptr = _i32(self.n_tiles + 2, dev)
            status = torch.zeros(1, dtype=torch.int32, device=dev)
            ws = ops._ws(lib.sgb_argsort_workspace_bytes(E) + 4 * max(E, 1) + 256, dev)
            ls, ld = lab[src], lab[dst]
            if ls.dtype != ld.dtype:
                ls, ld = ls.long(), ld.long()
            check(lib.sgb_partition_edges(ptr(ei), ei.element_size(), ei.stride(0), ei.stride(1), E, ptr(ls), ptr(ld),
                                          ls.element_size(), ls.numel(), ld.numel(), self.n_tiles, ptr(inv[src]), ptr(inv[dst]),
                                          ptr(new_ei), E, ptr(kept), ptr(rowptr), ptr(status), ptr(ws), ws.numel(),
                                          stream_ptr(dev)), "partition_edges")
            ops._count(10)
            statuses.append(status)
            edge_ptrs.append((et, new_ei, kept, rowptr))
        # one read-back for every pointer array and status word
        flat = torch.cat([p.to(torch.int64) for p in ptrs] + [r.to(torch.int64) for _, _, _, r in edge_ptrs] +
                         [s.to(torch.int64) for s in statuses]).tolist()
        o = 0
        for nt in data.node_types:
            self.node_indptr[nt] = flat[o:o + self.n_tiles + 1]
            o += self.n_tiles + 1
        for et, new_ei, kept, _ in edge_ptrs:
            rp = flat[o:o + self.n_tiles + 2]
            o += self.n_tiles + 2
            self.edge_indptr[et] = rp[:self.n_tiles + 1]
            n_kept = rp[self.n_tiles]
            out[et]["edge_index"] = new_ei[:, :n_kept]
            kept = kept[:n_kept]
            for name, attr in data[et].items():
                if name != "edge_index":
                    out[et][name] = (gather_rows(attr, kept) if isinstance(attr, Tensor) and attr.dim() >= 1
                                     and attr.size(0) == data[et]["edge_index"].size(1) else attr)
        if any(flat[o:]):
            raise IndexError("TilePartition: a node label is outside [0, n_tiles) or an edge names a missing node")
        self.data = out

    def __len__(self) -> int:
        return self.n_tiles

    @property
    def edge_sizes(self) -> Dict[EdgeType, List[int]]:
        return {et: [p[i + 1] - p[i] for i in range(self.n_tiles)] for et, p in self.edge_indptr.items()}

    @property
    def node_sizes(self) -> Dict[str, List[int]]:
        return {nt: [p[i + 1] - p[i] for i in range(self.n_tiles)] for nt, p in self.node_indptr.items()}

    def weights(self, mode: str = "edge") -> List[int]:
        """Per-tile packing weights of ``PartitionSampler`` (sum over edge / node types, sampler.py:346-354)."""
        sizes = self.edge_sizes if mode == "edge" else self.node_sizes
        return [sum(v[i] for v in sizes.values()) for i in range(self.n_tiles)]

    def batches(self, max_num: int, mode: str = "edge", subset: Optional[Sequence[int]] = None, shuffle: bool = False,
                skip_too_big: bool = False, rng: Optional[random.Random] = None) -> List[List[int]]:
        """The batches ``PartitionSampler`` would yield (sampler.py:364-382)."""
        idx = list(subset) if subset is not None else list(range(self.n_tiles))
        if shuffle:
            (rng or random).shuffle(idx)
        w = self.weights(mode)
        pack = first_fit_shuffled if shuffle else best_fit_decreasing
        kw = {"rng": rng} if shuffle else {}
        return [[idx[i] for i in b] for b in pack([w[i] for i in idx], max_num, skip_too_big=skip_too_big, **kw)]

    def __getitem__(self, index: int) -> HeteroBatch:
        if index < 0:
            index += self.n_tiles
        if not 0 <= index < self.n_tiles:
            raise IndexError(f"Index {index} is out of range for dataset with {self.n_tiles} partitions.")
        return self.collate([index])

    def collate(self, tiles: Sequence[int]) -> HeteroBatch:
        """``Batch.from_data_list([self[i] for i in tiles])``: node stores concatenated in list order, edges shifted
        to batch numbering, ``batch`` vectors per node type."""
        tiles = [int(t) + (self.n_tiles if t < 0 else 0) for t in tiles]
        K = len(tiles)
        lib = _lib.load()
        out = HeteroBatch()
        out._num_graphs = K
        dev = None
        n_start, n_off = {}, {}
        for nt, ip in self.node_indptr.items():
            starts = [ip[t] for t in tiles]
            off = [0]
            for t in tiles:
                off.append(off[-1] + ip[t + 1] - ip[t])
            store = self.data[nt]
            ref = next(v for v in store.values() if isinstance(v, Tensor))
            dev = ref.device
            d_start, d_off = _dev_i64(starts, dev), _dev_i64(off, dev)
            n_start[nt], n_off[nt] = d_start, d_off
            total = off[-1]
            n_all = ip[-1]
            for name, attr in store.items():
                if isinstance(attr, Tensor) and attr.dim() >= 1 and attr.size(0) == n_all:
                    a = attr.contiguous()
                    res = torch.empty((total,) + tuple(a.shape[1:]), dtype=a.dtype, device=dev)
                    row_bytes = a.element_size()
                    for d in a.shape[1:]:
                        row_bytes *= int(d)
                    if total > 0:
                        src_p = a.view(torch.uint8) if a.dtype == torch.bool else a
                        dst_p = res.view(torch.uint8) if res.dtype == torch.bool else res
                        check(lib.sgb_ranges_gather(ptr(src_p), row_bytes, ptr(d_start), ptr(d_off), K, total, ptr(dst_p),
                                                    stream_ptr(dev)), "ranges_gather")
                        ops._count(1)
                    out[nt][name] = res
                else:
                    out[nt][name] = attr
            bvec = torch.empty(total, dtype=torch.int64, device=dev)
            if total > 0:
                check(lib.sgb_batch_vector(ptr(d_off), K, total, ptr(bvec), stream_ptr(dev)), "batch_vector")
                ops._count(1)
            out[nt]["batch"] = set_num_graphs(bvec, K)
            out[nt]["ptr"] = d_off
        for et, ip in self.edge_indptr.items():
            src, _, dst = et
            ei = self.data[et]["edge_index"]
            e_start = [ip[t] for t in tiles]
            e_off = [0]
            for t in tiles:
                e_off.append(e_off[-1] + ip[t + 1] - ip[t])
            total = e_off[-1]
            res = torch.empty(2, total, dtype=ei.dtype, device=ei.device)
            if total > 0:
                d_es, d_eo = _dev_i64(e_start, dev), _dev_i64(e_off, dev)     # named: must outlive the launch
                check(lib.sgb_edges_collate(ptr(ei), ei.element_size(), ei.stride(0), ptr(d_es), ptr(d_eo), ptr(n_start[src]),
                                            ptr(n_off[src]), ptr(n_start[dst]), ptr(n_off[dst]), K, total, ptr(res), total,
                                            stream_ptr(ei.device)), "edges_collate")
                ops._count(1)
                out[et]["ptr"] = d_eo
            out[et]["edge_index"] = res
        return out


# ---------------------------------------------------------------------------------------------------------------------
# prediction tiles: tile + halo subgraph
# ---------------------------------------------------------------------------------------------------------------------
_MAX_CUT_RANGES = 1024            # candidate ranges of one cut (kMaxRanges of sgb_tilecut.cu)


def _merge_spans(spans: Sequence[Tuple[int, int]], budget: int) -> List[Tuple[int, int]]:
    """At most ``budget`` ranges covering ``spans`` (sorted, disjoint): the narrowest gaps are bridged.  The extra
    candidates are dropped by the exact box test of the cut kernels."""
    out = [list(r) for r in spans]
    while len(out) > max(1, budget):
        k = min(range(len(out) - 1), key=lambda i: out[i + 1][0] - out[i][1])
        out[k][1] = out[k + 1][1]
        del out[k + 1]
    return [tuple(r) for r in out]


class TilePredictSet:
    """``TilePredictDataset`` for a ``HeteroBatch`` on the GPU.  ``tiles``: [P, 4] (xmin, ymin, xmax, ymax) boxes;
    ``self[i]`` = the subgraph of the nodes inside box i grown by ``margin`` (half-open, tile_dataset.py:233-238) with
    ``predict_mask`` = inside the box itself (closed, :239-244), edges renumbered and in their original order.

    The reference scans every node and every edge of the dataset for every tile.  When the boxes form a regular
    ``grid = (nx, ny)`` (``square_tiles``) and the margin is smaller than a tile, an index built once (nodes sorted by
    grid cell, edges by the cell of their source -- two stable radix sorts per type) restricts a tile's scan to the
    3 x 3 neighbourhood of cells; the result is identical (same nodes, same order, same edges).

    ``tiles`` may also be a ``QuadTreeTiling``: the tiles are its leaves, and the index is built over the leaves (nodes
    stably sorted by leaf, edges by the leaf of their source).  A tile's candidates are the leaves whose box meets its
    margin-grown box (fp64, padded: a superset by construction), merged into ranges of adjacent leaf ids; the exact test
    stays in the cut kernels, so any margin works and the result is again identical to ``subset``."""

    def __init__(self, data: HeteroBatch, tiles, margin: float = 0.0, grid: Optional[Tuple[int, int]] = None):
        self.data = data
        tiling = tiles if isinstance(tiles, QuadTreeTiling) else None
        if tiling is not None:
            tiles = tiling.tiles
        self.tiles = [tuple(float(v) for v in t) for t in (tiles.tolist() if hasattr(tiles, "tolist") else tiles)]
        self.margin = float(margin)
        missing = [nt for nt in data.node_types if "pos" not in data[nt]]
        if missing:
            raise ValueError(f"Missing 'pos' attribute for node type: {', '.join(missing)}")
        self._index = None
        if tiling is not None:
            self._build_leaf_index(tiling)
        elif grid is not None and len(self.tiles) == grid[0] * grid[1] and len(self.tiles) > 1:
            self._build_index(grid)

    # -- coarse index ------------------------------------------------------------------------------------------------
    def _build_index(self, grid) -> None:
        nx, ny = grid
        x0, y0 = self.tiles[0][0], self.tiles[0][1]
        x1, y1 = self.tiles[-1][2], self.tiles[-1][3]
        w, h = (x1 - x0) / nx, (y1 - y0) / ny
        if not (self.margin < w and self.margin < h):
            return
        P = nx * ny
        labels, node_perm, node_ptr, maps = {}, {}, {}, {}
        ptrs = []
        for nt in self.data.node_types:
            pos = self.data[nt]["pos"]
            ix = torch.clamp(((pos[:, 0].double() - x0) / w).floor().long(), 0, nx - 1)
            iy = torch.clamp(((pos[:, 1].double() - y0) / h).floor().long(), 0, ny - 1)
            lab = (iy * nx + ix).to(torch.int32)
            perm, indptr, _ = stable_argsort(lab, P)
            labels[nt], node_perm[nt] = lab, perm
            ptrs.append(indptr)
            maps[nt] = torch.full((pos.size(0),), -1, dtype=torch.int32, device=pos.device)
        edge_perm = {}
        for et in self.data.edge_types:
            ei = self.data[et]["edge_index"]
            lab = labels[et[0]].index_select(0, ei[0].long())
            perm, indptr, _ = stable_argsort(lab, P)
            edge_perm[et] = perm
            ptrs.append(indptr)
        flat = torch.cat([p.to(torch.int64) for p in ptrs]).tolist()
        o = 0
        for nt in self.data.node_types:
            node_ptr[nt] = flat[o:o + P + 1]; o += P + 1
        edge_ptr = {}
        for et in self.data.edge_types:
            edge_ptr[et] = flat[o:o + P + 1]; o += P + 1
        self._index = dict(nx=nx, ny=ny, node_perm=node_perm, node_ptr=node_ptr, edge_perm=edge_perm, edge_ptr=edge_ptr, maps=maps)

    def _build_leaf_index(self, tiling: "QuadTreeTiling") -> None:
        P = len(self.tiles)
        bucket = P                        # nodes in no leaf (an empty quadrant): a candidate of every tile
        labels, node_perm, node_ptr, maps, ptrs = {}, {}, {}, {}, []
        for nt in self.data.node_types:
            pos = self.data[nt]["pos"]
            lab = tiling.label(pos)
            lab = torch.where(lab < 0, torch.full_like(lab, bucket), lab)
            perm, indptr, _ = stable_argsort(lab, P + 1)
            labels[nt], node_perm[nt] = lab, perm
            ptrs.append(indptr)
            maps[nt] = torch.full((pos.size(0),), -1, dtype=torch.int32, device=pos.device)
        edge_perm = {}
        for et in self.data.edge_types:
            ei = self.data[et]["edge_index"]
            perm, indptr, _ = stable_argsort(labels[et[0]].index_select(0, ei[0].long()), P + 1)
            edge_perm[et] = perm
            ptrs.append(indptr)
        flat = torch.cat([p.to(torch.int64) for p in ptrs]).tolist() if ptrs else []
        o = 0
        for nt in self.data.node_types:
            node_ptr[nt] = flat[o:o + P + 2]; o += P + 2
        edge_ptr = {}
        for et in self.data.edge_types:
            edge_ptr[et] = flat[o:o + P + 2]; o += P + 2
        # candidate leaves of every tile: leaf box (rim leaves open towards the outside: points beyond the root are
        # labelled with rim leaves) meets the tile's margin-grown box, padded by more than an fp32 rounding of the bounds
        b = tiling.tiles.detach().to("cpu", torch.float64)
        lo = b.min(0).values
        hi = b.max(0).values
        inf = float("inf")
        lb = b.clone()
        lb[:, 0][b[:, 0] <= lo[0]] = -inf
        lb[:, 1][b[:, 1] <= lo[1]] = -inf
        lb[:, 2][b[:, 2] >= hi[2]] = inf
        lb[:, 3][b[:, 3] >= hi[3]] = inf
        m = self.margin
        spans = []
        for t in range(P):
            x0, y0, x1, y1 = self.tiles[t]
            ob = torch.tensor([x0 - m, y0 - m, x1 + m, y1 + m], dtype=torch.float64)
            pad = 1e-6 * max(1.0, float(ob.abs().max()))
            hit = ((lb[:, 0] <= ob[2] + pad) & (lb[:, 2] >= ob[0] - pad) & (lb[:, 1] <= ob[3] + pad) & (lb[:, 3] >= ob[1] - pad))
            ids = hit.nonzero().flatten().tolist() + [bucket]
            rng = []
            for i in ids:
                if rng and rng[-1][1] == i:
                    rng[-1][1] = i + 1
                else:
                    rng.append([i, i + 1])
            spans.append([tuple(r) for r in rng])
        self._index = dict(spans=spans, node_perm=node_perm, node_ptr=node_ptr, edge_perm=edge_perm, edge_ptr=edge_ptr, maps=maps)

    def _neighbourhood(self, t: int) -> List[int]:
        if "spans" in self._index:
            return [c for a, b in self._index["spans"][t] for c in range(a, b)]
        nx, ny = self._index["nx"], self._index["ny"]
        i, j = t % nx, t // nx
        return [jj * nx + ii for jj in range(max(0, j - 1), min(ny, j + 2)) for ii in range(max(0, i - 1), min(nx, i + 2))]

    def _candidates(self, perm: Tensor, ptr_: List[int], cells: List[int]) -> Tensor:
        """ids of the given cells, ascending (the index stores them per cell; cells are disjoint)."""
        parts = [perm[ptr_[c]:ptr_[c + 1]] for c in cells if ptr_[c + 1] > ptr_[c]]
        if not parts:
            return perm[:0]
        return torch.sort(torch.cat(parts)).values       # index plumbing over the candidates only

    def __len__(self) -> int:
        return len(self.tiles)

    def __getitem__(self, idx: int) -> HeteroBatch:
        if idx < 0 or idx >= len(self):
            raise IndexError(f"Requested {idx}, but tiling only contains {len(self)} tiles.")
        if self._index is not None:
            return self._subset_indexed(idx)
        return self.subset(self.tiles[idx])

    def _boxes(self, bounds):
        x0, y0, x1, y1 = bounds
        m = self.margin
        return (C.c_double * 4)(x0 - m, y0 - m, x1 + m, y1 + m), (C.c_double * 4)(x0, y0, x1, y1)

    def _subset_indexed(self, t: int) -> HeteroBatch:
        outer, inner = self._boxes(self.tiles[t])
        lib = _lib.load()
        data, ix = self.data, self._index
        cells = self._neighbourhood(t)
        sel, pmask, counts, cand_n = {}, {}, [], {}
        for nt in data.node_types:
            pos = data[nt]["pos"]
            pos = (pos if pos.dtype in (torch.float32, torch.float64) else pos.float()).contiguous()
            cand = self._candidates(ix["node_perm"][nt], ix["node_ptr"][nt], cells)
            n, dev = cand.numel(), pos.device
            pos_c = gather_rows(pos, cand)
            s_loc = _i32(n, dev)
            pm = torch.empty(max(n, 1), dtype=torch.uint8, device=dev)
            cnt = torch.zeros(1, dtype=torch.int32, device=dev)
            ws = ops._ws(lib.sgb_select_workspace_bytes(n), dev)
            check(lib.sgb_box_select(ptr(pos_c), int(pos.dtype == torch.float64), n, outer, inner, ptr(s_loc), None, ptr(pm),
                                     ptr(cnt), ptr(ws), ws.numel(), stream_ptr(dev)), "box_select")
            s_glob = gather_rows(cand, s_loc, count=cnt)             # ascending node ids of the tile (+ halo)
            check(lib.sgb_scatter_rank(ptr(ix["maps"][nt]), ptr(s_glob), ptr(cnt), n, 0, 0, stream_ptr(dev)), "scatter_rank")
            ops._count(9)
            sel[nt], pmask[nt], cand_n[nt] = s_glob, pm, n
            counts.append(cnt)
        edges = {}
        for et in data.edge_types:
            src, _, dst = et
            ei = data[et]["edge_index"]
            ecand = self._candidates(ix["edge_perm"][et], ix["edge_ptr"][et], cells)
            E, dev = ecand.numel(), ei.device
            ei_c = torch.stack([gather_rows(ei[0], ecand), gather_rows(ei[1], ecand)])
            res = torch.empty(2, E, dtype=ei.dtype, device=dev)
            kept_loc = _i32(E, dev)
            cnt = torch.zeros(1, dtype=torch.int32, device=dev)
            ws = ops._ws(lib.sgb_select_workspace_bytes(E), dev)
            check(lib.sgb_edge_subset(ptr(ei_c), ei_c.element_size(), ei_c.stride(0), ei_c.stride(1), E, ptr(ix["maps"][src]),
                                      ix["maps"][src].numel(), ptr(ix["maps"][dst]), ix["maps"][dst].numel(), ptr(res), E,
                                      ptr(kept_loc), ptr(cnt), ptr(ws), ws.numel(), stream_ptr(dev)), "edge_subset")
            ops._count(7)
            edges[et] = (res, kept_loc, ecand)
            counts.append(cnt)
        for nt in data.node_types:                                   # leave the persistent maps clean for the next tile
            check(lib.sgb_scatter_rank(ptr(ix["maps"][nt]), ptr(sel[nt]), ptr(counts[data.node_types.index(nt)]), cand_n[nt], 1, -1,
                                       stream_ptr(sel[nt].device)), "scatter_rank")
        n_sel = torch.cat(counts).tolist()                           # the one read-back: sizes of the tile's stores
        out = HeteroBatch()
        out._num_graphs = 1
        for i, nt in enumerate(data.node_types):
            k = n_sel[i]
            n_all = data[nt]["pos"].size(0)
            for name, attr in data[nt].items():
                if isinstance(attr, Tensor) and attr.dim() >= 1 and attr.size(0) == n_all:
                    out[nt][name] = gather_rows(attr, sel[nt], m=k)
                else:
                    out[nt][name] = attr
            out[nt]["predict_mask"] = pmask[nt][:k].view(torch.bool)
            out[nt]["batch"] = set_num_graphs(torch.zeros(k, dtype=torch.int64, device=sel[nt].device), 1)
        for j, et in enumerate(data.edge_types):
            k = n_sel[len(data.node_types) + j]
            res, kept_loc, ecand = edges[et]
            out[et]["edge_index"] = res[:, :k]
            E_all = data[et]["edge_index"].size(1)
            extra = [n_ for n_, a_ in data[et].items() if n_ != "edge_index" and isinstance(a_, Tensor) and a_.dim() >= 1 and a_.size(0) == E_all]
            if extra:
                kept = gather_rows(ecand, kept_loc, m=k)
                for name in extra:
                    out[et][name] = gather_rows(data[et][name], kept, m=k)
            for name, attr in data[et].items():
                if name != "edge_index" and name not in extra:
                    out[et][name] = attr
        return out

    # -- several tiles at once --------------------------------------------------------------------------------------------
    def _slot_ranges(self, perm_ptr: List[int], tile_ids: Sequence[int], device):
        """Candidates of every slot as contiguous ranges of a cell-sorted id array: the 3 x 3 neighbourhood of a tile is
        one range per grid row; with the leaf index, one range per run of adjacent candidate leaves.
        -> (start [R], off [R + 1], slot [R]) device arrays, R, total candidates."""
        start, length, slot = [], [], []
        if "spans" in self._index:
            budget = _MAX_CUT_RANGES // len(tile_ids)
            for s_, t in enumerate(tile_ids):
                for c0, c1 in _merge_spans(self._index["spans"][t], budget):
                    a, b = perm_ptr[c0], perm_ptr[c1]
                    if b > a:
                        start.append(a); length.append(b - a); slot.append(s_)
        else:
            nx, ny = self._index["nx"], self._index["ny"]
            for s_, t in enumerate(tile_ids):
                i, j = t % nx, t // nx
                for jj in range(max(0, j - 1), min(ny, j + 2)):
                    c0, c1 = jj * nx + max(0, i - 1), jj * nx + min(nx, i + 2)
                    a, b = perm_ptr[c0], perm_ptr[c1]
                    if b > a:
                        start.append(a); length.append(b - a); slot.append(s_)
        off = [0]
        for n in length:
            off.append(off[-1] + n)
        packed = torch.tensor(start + off + slot, dtype=torch.int64).to(device, non_blocking=True)
        R = len(start)
        return packed[:R], packed[R:2 * R + 1], packed[2 * R + 1:].to(torch.int32), R, off[-1]

    def cut(self, tile_ids: Sequence[int]) -> Tuple[HeteroBatch, Dict]:
        """``collate_tiles([self[t] for t in tile_ids])`` -- the same nodes, order, edges and attributes -- assembled for
        all tiles together: two flag kernels per node / edge type (sgb_tilecut.cu), a compaction and a key sort each,
        and two device->host reads of the kept counts for the whole group (instead of ~100 launches and one read per
        tile).  Also returns ``info`` = per-slot node / edge counts (host lists) for batching by edge count."""
        if self._index is None:
            raise RuntimeError("TilePredictSet.cut needs an index: tiles from a QuadTreeTiling, or grid=(nx, ny) with margin "
                               "< tile size")
        tile_ids = [int(t) for t in tile_ids]
        T = len(tile_ids)
        if T == 0:
            raise ValueError("cut: no tiles")
        lib = _lib.load()
        data, ix = self.data, self._index
        dev = data[data.node_types[0]]["pos"].device
        m = self.margin
        boxes = torch.tensor([[x0 - m, y0 - m, x1 + m, y1 + m, x0, y0, x1, y1] for (x0, y0, x1, y1) in
                              (self.tiles[t] for t in tile_ids)], dtype=torch.float64).to(dev, non_blocking=True)
        st = stream_ptr(dev)

        def select(mask, C_):
            sel = _i32(C_, dev)
            cnt = torch.zeros(1, dtype=torch.int32, device=dev)
            ws = ops._ws(lib.sgb_select_workspace_bytes(C_), dev)
            check(lib.sgb_mask_select(ptr(mask), C_, ptr(sel), None, ptr(cnt), ptr(ws), ws.numel(), st), "mask_select")
            ops._count(5)
            return sel, cnt

        # ---- nodes: flag, compact, sort by (slot, id)
        node = {}
        for nt in data.node_types:
            pos = data[nt]["pos"]
            pos = (pos if pos.dtype in (torch.float32, torch.float64) else pos.float()).contiguous()
            r_start, r_off, r_slot, R, C_ = self._slot_ranges(ix["node_ptr"][nt], tile_ids, dev)
            keys = torch.empty(max(C_, 1), dtype=torch.int64, device=dev)
            mask = torch.empty(max(C_, 1), dtype=torch.uint8, device=dev)
            per_slot = torch.empty(T, dtype=torch.int32, device=dev)
            check(lib.sgb_tilecut_nodes(ptr(ix["node_perm"][nt]), ptr(pos), int(pos.dtype == torch.float64), ptr(r_start), ptr(r_off),
                                        ptr(r_slot), R, C_, ptr(boxes), T, ptr(keys), ptr(mask), ptr(per_slot), st), "tilecut_nodes")
            ops._count(1)
            sel, cnt = select(mask, C_) if C_ > 0 else (None, torch.zeros(1, dtype=torch.int32, device=dev))
            node[nt] = dict(pos=pos, keys=keys, sel=sel, cnt=cnt, per_slot=per_slot)
        counts = torch.cat([node[nt]["cnt"] for nt in data.node_types] + [node[nt]["per_slot"] for nt in data.node_types]).tolist()
        n_types = len(data.node_types)
        slot_arange = torch.arange(T + 1, dtype=torch.int64, device=dev) << 40
        info = {"nodes": {}, "edges": {}}
        for i, nt in enumerate(data.node_types):
            k = counts[i]
            d = node[nt]
            ks = gather_rows(d["keys"], d["sel"], m=k) if k > 0 else d["keys"][:0]
            ks = torch.sort(ks).values
            d["sorted"] = ks
            d["ptr"] = torch.searchsorted(ks, slot_arange).contiguous()
            d["ids"] = ((ks >> 1) & 0x7FFFFFFF).to(torch.int32)
            info["nodes"][nt] = counts[n_types + i * T:n_types + (i + 1) * T]
        # ---- edges: flag (both endpoints among the slot's nodes), compact, sort by (slot, edge id)
        edge = {}
        for et in data.edge_types:
            src, _, dst = et
            ei = data[et]["edge_index"]
            r_start, r_off, r_slot, R, C_ = self._slot_ranges(ix["edge_ptr"][et], tile_ids, dev)
            ekeys = torch.empty(max(C_, 1), dtype=torch.int64, device=dev)
            pu, pv = _i32(max(C_, 1), dev), _i32(max(C_, 1), dev)
            mask = torch.empty(max(C_, 1), dtype=torch.uint8, device=dev)
            per_slot = torch.empty(T, dtype=torch.int32, device=dev)
            sp = node[src]["pos"]
            check(lib.sgb_tilecut_edges(ptr(ix["edge_perm"][et]), ptr(ei), ei.element_size(), ei.stride(0), ei.stride(1), ptr(r_start),
                                        ptr(r_off), ptr(r_slot), R, C_, ptr(sp), int(sp.dtype == torch.float64), ptr(boxes), T,
                                        ptr(node[src]["sorted"]), ptr(node[src]["ptr"]), ptr(node[dst]["sorted"]),
                                        ptr(node[dst]["ptr"]), ptr(ekeys), ptr(pu), ptr(pv), ptr(mask), ptr(per_slot), st),
                  "tilecut_edges")
            ops._count(1)
            sel, cnt = select(mask, C_) if C_ > 0 else (None, torch.zeros(1, dtype=torch.int32, device=dev))
            edge[et] = dict(ekeys=ekeys, pu=pu, pv=pv, sel=sel, cnt=cnt, per_slot=per_slot)
        ecounts = torch.cat([edge[et]["cnt"] for et in data.edge_types] + [edge[et]["per_slot"] for et in data.edge_types]).tolist()
        # ---- assemble
        out = HeteroBatch()
        out._num_graphs = T
        for i, nt in enumerate(data.node_types):
            d = node[nt]
            k = counts[i]
            n_all = data[nt]["pos"].size(0)
            for name, attr in data[nt].items():
                if isinstance(attr, Tensor) and attr.dim() >= 1 and attr.size(0) == n_all:
                    out[nt][name] = gather_rows(attr, d["ids"], m=k)
                else:
                    out[nt][name] = attr
            out[nt]["predict_mask"] = (d["sorted"] & 1).to(torch.bool)
            out[nt]["batch"] = set_num_graphs(d["sorted"] >> 40, T)
        n_et = len(data.edge_types)
        for j, et in enumerate(data.edge_types):
            d = edge[et]
            k = ecounts[j]
            ei = data[et]["edge_index"]
            if k > 0:
                kk = gather_rows(d["ekeys"], d["sel"], m=k)
                kk, order = torch.sort(kk)
                sel_sorted = d["sel"][:k].index_select(0, order)
                res = torch.stack([gather_rows(d["pu"], sel_sorted, m=k), gather_rows(d["pv"], sel_sorted, m=k)]).to(ei.dtype)
            else:
                kk = d["ekeys"][:0]
                res = torch.empty(2, 0, dtype=ei.dtype, device=dev)
            out[et]["edge_index"] = res
            E_all = ei.size(1)
            eids = None
            for name, attr in data[et].items():
                if name == "edge_index":
                    continue
                if isinstance(attr, Tensor) and attr.dim() >= 1 and attr.size(0) == E_all:
                    if eids is None:
                        eids = (kk & 0x7FFFFFFF).to(torch.int32)
                    out[et][name] = gather_rows(attr, eids, m=k)
                else:
                    out[et][name] = attr
            info["edges"][et] = ecounts[n_et + j * T:n_et + (j + 1) * T]
        return out, info

    def subset(self, bounds: Sequence[float]) -> HeteroBatch:
        outer, inner = self._boxes(bounds)
        lib = _lib.load()
        data = self.data
        sel, amap, pmask, counts = {}, {}, {}, []
        for nt in data.node_types:
            pos = data[nt]["pos"]
            require_cuda(pos)
            pos = (pos if pos.dtype in (torch.float32, torch.float64) else pos.float()).contiguous()
            n, dev = pos.size(0), pos.device
            s, mp = _i32(n, dev), _i32(n, dev)
            pm = torch.empty(n, dtype=torch.uint8, device=dev)
            cnt = torch.zeros(1, dtype=torch.int32, device=dev)
            ws = ops._ws(lib.sgb_select_workspace_bytes(n), dev)
            check(lib.sgb_box_select(ptr(pos), int(pos.dtype == torch.float64), n, outer, inner, ptr(s), ptr(mp), ptr(pm), ptr(cnt),
                                     ptr(ws), ws.numel(), stream_ptr(dev)), "box_select")
            ops._count(6)
            sel[nt], amap[nt], pmask[nt] = s, mp, pm
            counts.append(cnt)
        edges = {}
        for et in data.edge_types:
            src, _, dst = et
            ei = data[et]["edge_index"]
            E, dev = ei.size(1), ei.device
            res = torch.empty(2, E, dtype=ei.dtype, device=dev)
            kept = _i32(E, dev)
            cnt = torch.zeros(1, dtype=torch.int32, device=dev)
            ws = ops._ws(lib.sgb_select_workspace_bytes(E), dev)
            check(lib.sgb_edge_subset(ptr(ei), ei.element_size(), ei.stride(0), ei.stride(1), E, ptr(amap[src]),
                                      amap[src].numel(), ptr(amap[dst]), amap[dst].numel(), ptr(res), E, ptr(kept), ptr(cnt),
                                      ptr(ws), ws.numel(), stream_ptr(dev)), "edge_subset")
            ops._count(5)
            edges[et] = (res, kept)
            counts.append(cnt)
        n_sel = torch.cat(counts).tolist()                   # the one read-back: sizes of the tile's stores
        out = HeteroBatch()
        out._num_graphs = 1
        for i, nt in enumerate(data.node_types):
            k = n_sel[i]
            n_all = data[nt]["pos"].size(0)
            for name, attr in data[nt].items():
                if isinstance(attr, Tensor) and attr.dim() >= 1 and attr.size(0) == n_all:
                    out[nt][name] = gather_rows(attr, sel[nt], m=k)
                else:
                    out[nt][name] = attr
            out[nt]["predict_mask"] = pmask[nt][:k].view(torch.bool)
            out[nt]["batch"] = set_num_graphs(torch.zeros(k, dtype=torch.int64, device=sel[nt].device), 1)
        for j, et in enumerate(data.edge_types):
            k = n_sel[len(data.node_types) + j]
            res, kept = edges[et]
            out[et]["edge_index"] = res[:, :k]
            E_all = data[et]["edge_index"].size(1)
            for name, attr in data[et].items():
                if name != "edge_index":
                    out[et][name] = (gather_rows(attr, kept, m=k) if isinstance(attr, Tensor) and attr.dim() >= 1
                                     and attr.size(0) == E_all else attr)
        return out


def square_tiles(xmin: float, ymin: float, xmax: float, ymax: float, nx: int, ny: int) -> List[Tuple[float, float, float, float]]:
    """nx x ny grid of boxes covering [xmin, xmax] x [ymin, ymax] (the synthetic counterpart of SquareTiling)."""
    w, h = (xmax - xmin) / nx, (ymax - ymin) / ny
    return [(xmin + i * w, ymin + j * h, xmin + (i + 1) * w if i + 1 < nx else xmax,
             ymin + (j + 1) * h if j + 1 < ny else ymax) for j in range(ny) for i in range(nx)]


def collate_tiles(tiles: Sequence[HeteroBatch]) -> HeteroBatch:
    """PyG collate of prediction tiles / groups of tiles (data_module.py:333-344): node stores concatenated, edge indices
    shifted by the node offsets, ``batch`` vectors shifted by the number of tiles that came before."""
    if len(tiles) == 1:
        return tiles[0]
    out = HeteroBatch()
    graphs = [int(getattr(t, "_num_graphs", 1) or 1) for t in tiles]
    out._num_graphs = sum(graphs)
    offs = {}
    for nt in tiles[0].node_types:
        sizes = [t[nt]["pos"].size(0) for t in tiles]
        off = [0]
        for n in sizes:
            off.append(off[-1] + n)
        offs[nt] = off
        for name in tiles[0][nt]:
            if name == "batch":
                continue
            a0 = tiles[0][nt][name]
            out[nt][name] = torch.cat([t[nt][name] for t in tiles]) if isinstance(a0, Tensor) and a0.dim() >= 1 else a0
        g0, parts = 0, []
        for t, g in zip(tiles, graphs):
            b = t[nt]["batch"]
            parts.append(b + g0 if g0 else b)
            g0 += g
        out[nt]["batch"] = set_num_graphs(torch.cat(parts), out._num_graphs)
    for et in tiles[0].edge_types:
        src, _, dst = et
        parts = []
        for i, t in enumerate(tiles):
            ei = t[et]["edge_index"]
            if offs[src][i] or offs[dst][i]:
                ei = ei + torch.tensor([[offs[src][i]], [offs[dst][i]]], dtype=ei.dtype).to(ei.device, non_blocking=True)
            parts.append(ei)
        out[et]["edge_index"] = torch.cat(parts, 1)
        for name in tiles[0][et]:
            if name == "edge_index":
                continue
            a0 = tiles[0][et][name]
            out[et][name] = torch.cat([t[et][name] for t in tiles]) if isinstance(a0, Tensor) and a0.dim() >= 1 else a0
    return out


def slice_slots(group: HeteroBatch, info: Dict, a: int, b: int) -> HeteroBatch:
    """Tiles (slots) [a, b) of a group made by ``TilePredictSet.cut``, renumbered to start at 0: views of the node / edge
    stores plus one subtraction per edge type."""
    T = int(group._num_graphs)
    if a == 0 and b == T:
        return group
    out = HeteroBatch()
    out._num_graphs = b - a
    n_lo, n_hi = {}, {}
    for nt in group.node_types:
        c = info["nodes"][nt]
        n_lo[nt], n_hi[nt] = sum(c[:a]), sum(c[:b])
        n_all = group[nt]["pos"].size(0)
        for name, attr in group[nt].items():
            if name == "batch":
                continue
            out[nt][name] = attr[n_lo[nt]:n_hi[nt]] if isinstance(attr, Tensor) and attr.dim() >= 1 and attr.size(0) == n_all else attr
        out[nt]["batch"] = set_num_graphs(group[nt]["batch"][n_lo[nt]:n_hi[nt]] - a, b - a)
    for et in group.edge_types:
        src, _, dst = et
        c = info["edges"][et]
        lo, hi = sum(c[:a]), sum(c[:b])
        ei = group[et]["edge_index"][:, lo:hi]
        if n_lo[src] or n_lo[dst]:
            ei = ei - torch.tensor([[n_lo[src]], [n_lo[dst]]], dtype=ei.dtype).to(ei.device, non_blocking=True)
        out[et]["edge_index"] = ei
        E_all = group[et]["edge_index"].size(1)
        for name, attr in group[et].items():
            if name != "edge_index":
                out[et][name] = attr[lo:hi] if isinstance(attr, Tensor) and attr.dim() >= 1 and attr.size(0) == E_all else attr
    return out
