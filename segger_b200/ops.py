"""Functional layer over the C ABI: torch tensors in, torch tensors out, autograd wired by hand.

Everything here enqueues hand-written sm_100a kernels from libsegger_b200.so on the current torch
stream.  torch provides device memory (caching allocator), streams and the autograd *graph*; no
torch operator computes anything on the hot path.
"""
from __future__ import annotations

import ctypes as C
import math
import os
from dataclasses import dataclass
from typing import Optional, Tuple

import torch
from torch import Tensor

from . import _lib
from ._lib import ACT_GELU, ACT_NONE, ACT_SILU, check, ptr, require_cuda, stream_ptr

LAUNCHES = 0  # kernels launched through this module (bench.py reports it as gpu_launches)


def _count(n: int) -> None:
    global LAUNCHES
    LAUNCHES += n


def _ws(nbytes: int, device) -> Tensor:
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)


def _rowmajor(t: Tensor) -> Tensor:
    """2-D fp32 tensor with unit inner stride (column slices of a wider buffer are fine)."""
    if t.dtype != torch.float32:
        raise TypeError(f"expected float32, got {t.dtype}")
    if t.dim() != 2:
        raise ValueError(f"expected a 2-D tensor, got shape {tuple(t.shape)}")
    if t.size(1) > 1 and t.stride(1) != 1:
        t = t.contiguous()
    if t.size(0) > 1 and t.stride(0) < t.size(1):
        t = t.contiguous()
    return t


def _ld(t: Tensor) -> int:
    return t.stride(0) if t.size(0) > 1 else max(t.size(1), t.stride(0))


def _vec(t: Optional[Tensor]) -> Optional[Tensor]:
    if t is None:
        return None
    if t.dtype != torch.float32:
        raise TypeError(f"expected float32, got {t.dtype}")
    return t.contiguous()


# ------------------------------------------------------------------------------------------------
# Graph layout
# ------------------------------------------------------------------------------------------------
@dataclass
class EdgeCSR:
    """dst-sorted CSR (+ src-sorted transposed CSR) of one edge type; all int32 on device."""
    rowptr: Tensor
    col: Tensor
    eid: Tensor
    t_rowptr: Optional[Tensor]
    t_dst: Optional[Tensor]
    t_pos: Optional[Tensor]
    n_src: int
    n_dst: int
    E: int
    status: Tensor
    src_index: Optional[Tensor] = None      # row 0 of the edge_index this CSR was built from (a view, kept alive)
    _src_unique: Optional[bool] = None      # lazily computed: source ids strictly increasing (each source once)
    _virtual: Optional["EdgeCSR"] = None
    one_source_per_edge: bool = False       # col is a permutation of [0, E): the backward needs no transposed pass

    def validate(self) -> "EdgeCSR":
        """One 8-byte D2H read per CSR build (cached): raises IndexError if the edge list held node ids outside
        [0, n_src) x [0, n_dst) -- what torch / PyG indexing does with such an edge_index -- and records whether
        the sources are unique and increasing."""
        if self._src_unique is None:
            validate_csrs(self, force=True)
        return self

    def sources_unique_increasing(self) -> bool:
        """True iff the edge list names every source at most once, in increasing order (what setup_heterodata emits
        for tx-belongs-bd)."""
        return bool(self.validate()._src_unique)

    def per_edge_sources(self) -> "EdgeCSR":
        """The same graph with one virtual source node per edge (valid when sources are unique and increasing, so
        that edge order == source order): column index = original edge id, trivial transposed row pointer."""
        if self._virtual is None:
            t_rowptr = None
            if self.t_rowptr is not None:
                t_rowptr = torch.arange(self.E + 1, dtype=torch.int32, device=self.rowptr.device)
            self._virtual = EdgeCSR(self.rowptr, self.eid, self.eid, t_rowptr, self.t_dst, self.t_pos, self.E, self.n_dst,
                                    self.E, self.status, self.src_index, one_source_per_edge=True)
        return self._virtual


def build_csr(edge_index: Tensor, n_src: int, n_dst: int, transpose: bool = True) -> EdgeCSR:
    """COO [2,E] (int32/int64, any strides) -> EdgeCSR.  Replaces PyG's per-call scatter indexing."""
    require_cuda(edge_index)
    if edge_index.dim() != 2 or edge_index.size(0) != 2:
        raise ValueError(f"edge_index must be [2, E], got {tuple(edge_index.shape)}")
    if edge_index.dtype not in (torch.int32, torch.int64):
        raise TypeError(f"edge_index must be int32 or int64, got {edge_index.dtype}")
    dev = edge_index.device
    E = edge_index.size(1)
    lib = _lib.load()
    i32 = dict(dtype=torch.int32, device=dev)
    rowptr = torch.empty(n_dst + 1, **i32)
    col = torch.empty(E, **i32)
    eid = torch.empty(E, **i32)
    t_rowptr = torch.empty(n_src + 1, **i32) if transpose else None
    t_dst = torch.empty(E, **i32) if transpose else None
    t_pos = torch.empty(E, **i32) if transpose else None
    status = torch.zeros(2, **i32)     # [0]: out-of-range ids seen (set by the build), [1]: sources strictly increasing
    ws = _ws(lib.sgb_csr_workspace_bytes(E), dev)
    with torch.cuda.device(dev):
        check(lib.sgb_csr_build(ptr(edge_index), edge_index.element_size(), edge_index.stride(0),
                                edge_index.stride(1), E, n_src, n_dst, ptr(rowptr), ptr(col), ptr(eid),
                                ptr(t_rowptr), ptr(t_dst), ptr(t_pos), ptr(status), ptr(ws), ws.numel(),
                                stream_ptr(dev)), "csr_build")
        _count(12 if transpose else 6)
        if E > 0:
            idx = edge_index[0]
            if idx.stride(0) != 1:
                idx = idx.contiguous()
            check(lib.sgb_index_strictly_increasing(ptr(idx), idx.element_size(), idx.numel(), ptr(status[1:]),
                                                    stream_ptr(dev)), "index_strictly_increasing")
            _count(2)
    return EdgeCSR(rowptr, col, eid, t_rowptr, t_dst, t_pos, n_src, n_dst, E, status, edge_index[0])


_DEFERRED: Optional[list] = None      # CSRs whose validation a caller folds into a later sync (predict_step)
VALIDATE = os.environ.get("SEGGER_B200_VALIDATE", "1") != "0"


class deferred_validation:
    """``with deferred_validation() as pending:`` -- CSRs built inside the block are not validated on the spot (no
    stream sync); the caller reads ``pending_status(pending)`` together with its own results and calls
    ``finish_validation``.  Used by predict_step, whose results need a device->host copy anyway."""

    def __enter__(self):
        global _DEFERRED
        self.prev, _DEFERRED = _DEFERRED, []
        return _DEFERRED

    def __exit__(self, *exc):
        global _DEFERRED
        _DEFERRED = self.prev
        return False


def pending_status(pending: list) -> Optional[Tensor]:
    todo = [c for c in pending if c._src_unique is None]
    return torch.stack([c.status for c in todo]) if todo else None


def finish_validation(pending: list, flags) -> None:
    todo = [c for c in pending if c._src_unique is None]
    _apply_status(todo, flags)


def _apply_status(todo, flags) -> None:
    for c, (bad, inc) in zip(todo, flags):
        if bad:
            raise IndexError(f"edge_index holds node ids outside [0, {c.n_src}) x [0, {c.n_dst}) "
                             f"(E={c.E}); PyG / torch indexing would fail on it")
        c._src_unique = bool(inc) and c.E > 0


def validate_csrs(*csrs: "EdgeCSR", force: bool = False) -> None:
    """Read the status words of several freshly built CSRs with ONE device->host copy (one stream sync per new
    graph, none once a CSR has been validated).  Out-of-range node ids raise IndexError: the kernels clamp such ids
    so they never fault, but a malformed edge_index must not train or predict silently.
    ``SEGGER_B200_VALIDATE=0`` turns the check (and its sync) off."""
    todo = [c for c in csrs if c is not None and c._src_unique is None]
    if not todo:
        return
    if not force:
        if _DEFERRED is not None:
            _DEFERRED.extend(todo)
            return
        if not VALIDATE:
            return
    _apply_status(todo, torch.stack([c.status for c in todo]).tolist())


class _CsrCache:
    """Tiny LRU so that the layers of one forward (and repeated forwards over a static graph) share
    one CSR build per edge type.  Keyed on storage identity + version; holds the tensor alive."""

    def __init__(self, size: int = 4):
        # one forward touches two edge types (+ the candidate edges of predict_step): 4 entries = the current batch
        # and nothing older; per-tile batches never hit across steps, so a larger cache would only pin dead graphs
        self.size = size
        self.items = []

    def get(self, edge_index: Tensor, n_src: int, n_dst: int, transpose: bool) -> EdgeCSR:
        # inference tensors (Lightning's predict / validation loops run under torch.inference_mode) carry no version
        # counter; they cannot be mutated in place outside inference mode, so identity + layout is the whole key
        ver = None if edge_index.is_inference() else edge_index._version
        key = (edge_index.data_ptr(), tuple(edge_index.shape), edge_index.stride(), edge_index.dtype, ver, n_src, n_dst,
               edge_index.device)
        for i, (k, t, csr) in enumerate(self.items):
            if k == key:
                if csr.t_rowptr is not None or not transpose:
                    self.items.append(self.items.pop(i))
                    return csr
                self.items.pop(i)          # built without the transpose: replaced below, not kept beside the new one
                break
        csr = build_csr(edge_index, n_src, n_dst, transpose)
        self.items.append((key, edge_index, csr))
        if len(self.items) > self.size:
            self.items.pop(0)
        return csr

    def has(self, edge_index: Tensor, n_src: int, n_dst: int, transpose: bool) -> bool:
        ver = None if edge_index.is_inference() else edge_index._version
        key = (edge_index.data_ptr(), tuple(edge_index.shape), edge_index.stride(), edge_index.dtype, ver, n_src, n_dst,
               edge_index.device)
        return any(k == key and (csr.t_rowptr is not None or not transpose) for k, _, csr in self.items)

    def clear(self):
        self.items.clear()


CSR_CACHE = _CsrCache()

_CSR_STREAMS: dict = {}
_CSR_OVERLAP_MIN_EDGES = 2_000_000


class CsrJoin:
    """Handle of CSR builds that were enqueued on the side stream (``csr_build_overlapped``)."""

    def __init__(self, csrs, event=None, status_host=None, todo=()):
        self.csrs, self.event, self.status_host, self.todo = csrs, event, status_host, list(todo)

    def join(self) -> None:
        """The current stream waits for the builds (device-side wait, no host synchronisation)."""
        if self.event is not None:
            torch.cuda.current_stream().wait_event(self.event)

    def resolve(self) -> None:
        """Host side of a NEW graph: wait for the builds only (not for whatever the main stream was given meanwhile)
        and apply the status words they left (IndexError on out-of-range node ids)."""
        if self.status_host is not None:
            self.event.synchronize()
            vals = self.status_host.tolist()
            pairs = [(c, vals[2 * i:2 * i + 2]) for i, c in enumerate(self.todo) if c._src_unique is None]
            self.status_host = None
            _apply_status([c for c, _ in pairs], [f for _, f in pairs])


def csr_overlap_mark(edge_index: Tensor):
    """Event on the current stream marking "the edge lists are ready" -- recorded BEFORE the caller enqueues the work the
    CSR builds are to overlap with.  None when the builds will not use the side stream."""
    # (small graphs are bound by the host's launch rate, where a second stream only adds host work: one tile of
    # BASELINE configs[0] steps in 4.1 ms on the caller's stream and 4.5 ms with the side stream)
    if (edge_index.size(-1) < _CSR_OVERLAP_MIN_EDGES or os.environ.get("SEGGER_B200_CSR_OVERLAP", "1") == "0"
            or torch.cuda.is_current_stream_capturing()):
        return None
    ev = torch.cuda.Event()
    ev.record(torch.cuda.current_stream(edge_index.device))
    return ev


def csr_build_overlapped(specs, transpose: bool, after=None) -> CsrJoin:
    """``specs`` = [(edge_index, n_src, n_dst), ...] -> CsrJoin with ``.csrs`` in the same order.

    A CSR build is ~55 small dependent launches per edge type (radix passes, scans, checks): ~1.2 ms of a 16 ms
    training step at 1M transcripts, almost all of it launch latency.  Nothing before the first graph convolution needs
    the CSRs, so new graphs are built on a side stream while the caller's stream runs the input stage (embedding,
    positional MLP); ``join()`` orders the caller's stream behind them.  The caller enqueues the input stage FIRST and
    passes the event it recorded before it (``after`` = ``csr_overlap_mark``): one host thread issues every launch, so
    the few long input-stage kernels must already be queued when the ~110 short build launches are issued.  Cache hits
    (static graphs, CUDA-graph capture) and ``SEGGER_B200_CSR_OVERLAP=0`` stay on the caller's stream."""
    dev = specs[0][0].device
    miss = [not CSR_CACHE.has(ei, ns, nd, transpose) for ei, ns, nd in specs]
    side_ok = any(miss) and after is not None
    if not side_ok:
        return CsrJoin([CSR_CACHE.get(ei, ns, nd, transpose) for ei, ns, nd in specs])
    main = torch.cuda.current_stream(dev)
    side = _CSR_STREAMS.get(dev)
    if side is None:
        side = _CSR_STREAMS[dev] = torch.cuda.Stream(dev)
    if after is not None:
        side.wait_event(after)      # the edge lists are ready (recorded before the work this build overlaps with)
    else:
        side.wait_stream(main)
    status_host, todo = None, []
    with torch.cuda.stream(side):
        csrs = [CSR_CACHE.get(ei, ns, nd, transpose) for ei, ns, nd in specs]
        for c, m in zip(csrs, miss):
            if m:   # allocated on the side stream, consumed on the caller's: tell the caching allocator
                for t in (c.rowptr, c.col, c.eid, c.t_rowptr, c.t_dst, c.t_pos, c.status):
                    if t is not None:
                        t.record_stream(main)
        if VALIDATE and _DEFERRED is None:
            todo = [c for c in csrs if c._src_unique is None]
            if todo:
                status_host = torch.empty(2 * len(todo), dtype=torch.int32, pin_memory=True)
                status_host.copy_(torch.stack([c.status for c in todo]).flatten(), non_blocking=True)
        event = torch.cuda.Event()
        event.record(side)
    return CsrJoin(csrs, event, status_host, todo)


_SEED_WORD: Optional[Tensor] = None      # device int64 [1] added to every dropout seed (see device_seed)
_SEED_SITE = 0


class device_seed:
    """``with device_seed(word):`` -- dropout seeds come from a DEVICE word instead of the CPU generator.

    Inside the block ``new_seed()`` returns ``(call-site number, word)``: the kernels add the word's current value to the
    call-site number when they run, so a CUDA graph captured inside the block draws a fresh mask on every replay once the
    word is advanced on the device (segger_b200/graphs.py does ``word += odd constant`` as the first node of the graph).
    Forward and backward of one step read the same value.  The call-site numbers restart at every ``with``."""

    def __init__(self, word: Tensor):
        if word.dtype != torch.int64 or word.numel() != 1 or not word.is_cuda:
            raise ValueError("device_seed: expected a CUDA int64 tensor with one element")
        self.word = word

    def __enter__(self):
        global _SEED_WORD, _SEED_SITE
        self._prev = (_SEED_WORD, _SEED_SITE)
        _SEED_WORD, _SEED_SITE = self.word, 0
        return self

    def __exit__(self, *exc):
        global _SEED_WORD, _SEED_SITE
        _SEED_WORD, _SEED_SITE = self._prev
        return False


def new_seed():
    """63-bit seed drawn from torch's default (CPU) generator: torch.manual_seed governs dropout.  Under
    ``device_seed`` -> (call-site number, device word) instead (no host RNG, graph-capturable)."""
    global _SEED_SITE
    if _SEED_WORD is not None:
        _SEED_SITE += 1
        return (_SEED_SITE * 0x9E3779B97F4A7C15) & (2 ** 62 - 1), _SEED_WORD
    return int(torch.randint(0, 2 ** 62, (1,), dtype=torch.int64).item())


def _split_seed(seed):
    """seed (int | (int, device word)) -> (by-value seed, device word or None)."""
    return seed if isinstance(seed, tuple) else (seed, None)


# ------------------------------------------------------------------------------------------------
# raw kernel wrappers (no autograd)
# ------------------------------------------------------------------------------------------------
def linear_fwd(x: Tensor, w: Tensor, b: Optional[Tensor], act: int = ACT_NONE,
               y: Optional[Tensor] = None, y_act: Optional[Tensor] = None,
               want_pre: bool = True, exact: Optional[bool] = None,
               gather: Optional[Tuple[Tensor, Tensor]] = None) -> Tuple[Optional[Tensor], Optional[Tensor]]:
    """(y, act(y)) with y = x w^T + b.  y / y_act may be preallocated (strided) views.

    ``exact``: 0/False = 3-product split-TF32, 1/True = 4 products (fp32-exact operand products);
    both accumulate 32-deep TMEM chunks in registers with round-to-nearest; 2 = force the fp32 SIMT
    kernel.  Default: exact while autograd is recording (the result will be
    differentiated through the attention layers, whose backward amplifies the tensor core's biased
    round-toward-zero accumulation -- DESIGN.md "GEMM precision"), fast under ``torch.no_grad()``."""
    if exact is None:
        exact = torch.is_grad_enabled()
    x, w = _rowmajor(x), _rowmajor(w)
    M, K = x.shape
    N = w.size(0)
    if w.size(1) != K:
        raise ValueError(f"linear: x is [*, {K}] but weight is {tuple(w.shape)}")
    dev = x.device
    if y is None:
        y = torch.empty(M, N, dtype=torch.float32, device=dev)
    if act != ACT_NONE and y_act is None:
        y_act = torch.empty(M, N, dtype=torch.float32, device=dev)
    b = _vec(b)
    lib = _lib.load()
    ws = _ws(lib.sgb_linear_workspace_bytes(N, K), dev)
    if gather is not None:          # y = x w^T + b + table[ids]   (ids [M] int32/int64, table [*, N])
        if act != ACT_NONE:
            raise ValueError("linear_fwd: gather cannot be combined with an activation epilogue")
        ids, table = gather
        ids = ids if ids.stride(0) == 1 else ids.contiguous()
        table = _rowmajor(table)
        if table.size(1) != N or ids.numel() != M:
            raise ValueError("linear_fwd: gather table / ids do not match the output shape")
        check(lib.sgb_linear_fwd_gather(ptr(x), _ld(x), ptr(w), _ld(w), ptr(b), M, N, K, ptr(y), _ld(y), ptr(ids),
                                        ids.element_size(), ptr(table), _ld(table), int(exact), ptr(ws), ws.numel(),
                                        stream_ptr(dev)), "linear_fwd_gather")
        _count(2)
        return y, None
    check(lib.sgb_linear_fwd(ptr(x), _ld(x), ptr(w), _ld(w), ptr(b), M, N, K, ptr(y), _ld(y), act,
                             ptr(y_act), _ld(y_act) if y_act is not None else 0, int(exact),
                             ptr(ws), ws.numel(), stream_ptr(dev)),
          "linear_fwd")
    _count(2)
    return y, y_act


def linear_dgrad(dy: Tensor, w: Tensor, dx: Optional[Tensor] = None, accumulate: bool = False,
                 act: int = ACT_NONE, act_pre: Optional[Tensor] = None) -> Tensor:
    dy, w = _rowmajor(dy), _rowmajor(w)
    M, N = dy.shape
    K = w.size(1)
    if dx is None:
        dx = torch.empty(M, K, dtype=torch.float32, device=dy.device)
    lib = _lib.load()
    ws = _ws(lib.sgb_linear_workspace_bytes(N, K), dy.device)
    check(lib.sgb_linear_dgrad(ptr(dy), _ld(dy), ptr(w), _ld(w), M, N, K, ptr(dx), _ld(dx),
                               int(accumulate), act, ptr(act_pre),
                               _ld(act_pre) if act_pre is not None else 0, ptr(ws), ws.numel(),
                               stream_ptr(dy.device)),
          "linear_dgrad")
    _count(2)
    return dx


def linear_wgrad(dy: Tensor, x: Tensor, dw: Optional[Tensor] = None, db: Optional[Tensor] = None,
                 want_db: bool = True, accumulate: bool = False) -> Tuple[Tensor, Optional[Tensor]]:
    dy, x = _rowmajor(dy), _rowmajor(x)
    M, N = dy.shape
    K = x.size(1)
    dev = dy.device
    if dw is None:
        dw = torch.empty(N, K, dtype=torch.float32, device=dev)
    if db is None and want_db:
        db = torch.empty(N, dtype=torch.float32, device=dev)
    lib = _lib.load()
    ws = _ws(lib.sgb_linear_wgrad_workspace_bytes(M, N, K), dev)
    check(lib.sgb_linear_wgrad(ptr(dy), _ld(dy), ptr(x), _ld(x), M, N, K, ptr(dw), _ld(dw), ptr(db),
                               int(accumulate), ptr(ws), ws.numel(), stream_ptr(dev)), "linear_wgrad")
    _count(4 if db is not None else 2)
    return dw, db


def gather_rows(x: Tensor, ids: Tensor) -> Tensor:
    """out[k, :] = x[ids[k], :] (x contiguous [N, D]); the embedding-gather kernel with x as the table."""
    x = x.contiguous()
    ids = ids if ids.stride(0) == 1 else ids.contiguous()
    n, D = ids.numel(), x.size(1)
    out = torch.empty(n, D, dtype=torch.float32, device=x.device)
    check(_lib.load().sgb_embedding_fwd(ptr(x), x.size(0), D, ptr(ids), ids.element_size(), n, ptr(out), D, None, 0,
                                        ACT_NONE, stream_ptr(x.device)), "gather_rows")
    _count(1)
    return out


def rows_add(dst: Tensor, ids: Tensor, src: Tensor) -> Tensor:
    """dst[ids[k], :] += src[k, :] for unique ids (in place)."""
    dst, src = _rowmajor(dst), _rowmajor(src)
    ids = ids if ids.stride(0) == 1 else ids.contiguous()
    check(_lib.load().sgb_rows_add(ptr(dst), _ld(dst), dst.size(0), ptr(ids), ids.element_size(), ids.numel(), src.size(1),
                                   ptr(src), _ld(src), stream_ptr(dst.device)), "rows_add")
    _count(1)
    return dst


def segment_sum_rows(g: Tensor, idx: Tensor, n_rows: int) -> Tensor:
    """out[r, :] = sum of g[k, :] over k with idx[k] == r, in a fixed order (sort by id + chunked segment sums + ordered
    merge: deterministic, no atomics).  The backward of a row gather."""
    g = _rowmajor(g)
    idx = idx if idx.stride(0) == 1 else idx.contiguous()
    lib = _lib.load()
    T, D = g.shape
    out = torch.empty(n_rows, D, dtype=torch.float32, device=g.device)
    ws = _ws(lib.sgb_embedding_bwd_workspace_bytes(T, D, n_rows), g.device)
    check(lib.sgb_embedding_bwd(ptr(g), _ld(g), ptr(idx), idx.element_size(), T, D, n_rows, None, 0, ptr(out), ptr(ws),
                                ws.numel(), stream_ptr(g.device)), "segment_sum_rows")
    _count(10)
    return out


class SelectRowsFn(torch.autograd.Function):
    """x[idx] for unique row indices (e.g. torch.nonzero(mask)): gather forward, rows_add into zeros backward."""

    @staticmethod
    def forward(ctx, x, idx):
        require_cuda(x, idx)
        ctx.n = x.size(0)
        ctx.save_for_backward(idx)
        return gather_rows(x, idx)

    @staticmethod
    def backward(ctx, g):
        (idx,) = ctx.saved_tensors
        dx = torch.zeros(ctx.n, g.size(1), dtype=torch.float32, device=g.device)
        if idx.numel() > 0:
            if g.size(1) % 4 == 0:
                rows_add(dx, idx, g.contiguous())
            else:
                dx.index_add_(0, idx, g)
        return dx, None


def select_rows(x: Tensor, mask: Tensor, idx: Optional[Tensor] = None) -> Tensor:
    """x[mask] (boolean row mask) with the gather / scatter done by library kernels.  ``idx`` = a precomputed
    ``torch.nonzero(mask).flatten()`` (callers that resolve their masks off the critical path)."""
    if idx is None:
        idx = torch.nonzero(mask, as_tuple=False).flatten()
    if idx.numel() == x.size(0):
        return x
    return SelectRowsFn.apply(x, idx)


class side_section:
    """``with side_section(after_event) as sec:`` -- host-synchronising bookkeeping (mask -> index lists, triplet
    sampling: ~100 short launches and half a dozen device->host reads that depend only on a batch's labels) runs on a
    side stream, so its stream synchronisations wait for that stream alone while the caller's stream keeps executing
    the forward pass it was already given.  ``after_event``: recorded on the caller's stream when the inputs of the
    section were ready.  On exit the caller's stream waits for the section; ``sec.keep(t, ...)`` marks tensors created
    inside that the caller's stream will use.  Under CUDA-graph capture (or ``SEGGER_B200_LOSS_OVERLAP=0``) the section
    runs inline."""

    def __init__(self, after_event, device):
        self.inline = (after_event is None or os.environ.get("SEGGER_B200_LOSS_OVERLAP", "1") == "0"
                       or torch.cuda.is_current_stream_capturing())
        self.after, self.device, self.kept = after_event, device, []

    def keep(self, *tensors):
        self.kept.extend(t for t in tensors if isinstance(t, Tensor) and t.is_cuda)
        return tensors[0] if len(tensors) == 1 else tensors

    def __enter__(self):
        if not self.inline:
            self.main = torch.cuda.current_stream(self.device)
            side = _CSR_STREAMS.get(("loss", self.device))
            if side is None:
                side = _CSR_STREAMS[("loss", self.device)] = torch.cuda.Stream(self.device)
            side.wait_event(self.after)
            self.ctx = torch.cuda.stream(side)
            self.ctx.__enter__()
            self.side = side
        return self

    def __exit__(self, *exc):
        if not self.inline:
            for t in self.kept:
                t.record_stream(self.main)
            ev = torch.cuda.Event()
            ev.record(self.side)
            self.ctx.__exit__(*exc)
            self.main.wait_event(ev)
        return False


def section_mark(t: Tensor):
    """Event on the current stream ("everything enqueued so far"), or None where a side section would run inline."""
    if not t.is_cuda or os.environ.get("SEGGER_B200_LOSS_OVERLAP", "1") == "0" or torch.cuda.is_current_stream_capturing():
        return None
    ev = torch.cuda.Event()
    ev.record(torch.cuda.current_stream(t.device))
    return ev


def act_bwd(dy: Tensor, pre: Tensor, act: int, dx: Optional[Tensor] = None) -> Tensor:
    dy, pre = _rowmajor(dy), _rowmajor(pre)
    M, N = dy.shape
    if dx is None:
        dx = torch.empty(M, N, dtype=torch.float32, device=dy.device)
    check(_lib.load().sgb_act_bwd(ptr(dy), _ld(dy), ptr(pre), _ld(pre), M, N, act, ptr(dx), _ld(dx),
                                  stream_ptr(dy.device)), "act_bwd")
    _count(1)
    return dx


def act_fwd(x: Tensor, act: int, y: Optional[Tensor] = None) -> Tensor:
    x = _rowmajor(x)
    M, N = x.shape
    if y is None:
        y = torch.empty(M, N, dtype=torch.float32, device=x.device)
    check(_lib.load().sgb_act_fwd(ptr(x), _ld(x), M, N, act, ptr(y), _ld(y), stream_ptr(x.device)), "act_fwd")
    _count(1)
    return y


_QUAD_SHAPES: dict = {}


def _quad_path(H: int, C: int, slope: float, *tensors) -> bool:
    """True iff sgb_gatv2_fwd / sgb_gatv2_bwd will run the sub-warp kernels on these operands (the library's own rule:
    shape covered, 0 <= slope <= 1, 16-byte aligned pointers, leading dimensions a multiple of 4 floats)."""
    ok = _QUAD_SHAPES.get((H, C))
    if ok is None:
        ok = _QUAD_SHAPES[(H, C)] = bool(_lib.load().sgb_gatv2_quad_supported(H, C))
    return (ok and 0.0 <= slope <= 1.0
            and os.environ.get("SEGGER_B200_GAT") != "legacy"
            and all(t is None or (t.data_ptr() % 16 == 0 and (t.dim() < 2 or _ld(t) % 4 == 0)) for t in tensors))


def gatv2_fwd(x_l: Tensor, x_r: Tensor, att: Tensor, bias: Optional[Tensor], csr: EdgeCSR, H: int, C: int,
              slope: float, p_drop: float, training: bool, seed: int, want_act: bool,
              out: Optional[Tensor] = None, out_act: Optional[Tensor] = None, want_pre: bool = True,
              want_logits: Optional[bool] = False):
    """-> (out_pre|None, out_act|None, stat_max, stat_den).  ``want_pre=False`` (with ``want_act``) writes only
    the activated output: the pre-activation is needed by the backward alone.  ``want_logits=True`` appends a fifth
    element: the raw attention logits [E, H] in dst-CSR order for ``gatv2_bwd(e_logit=...)`` (None where the sub-warp
    kernels do not apply; ``SEGGER_B200_GAT_LOGITS=0`` turns the saved-logit backward off)."""
    x_l, x_r = _rowmajor(x_l), _rowmajor(x_r)
    F = H * C
    dev = x_r.device
    n_dst = x_r.size(0)
    if x_l.size(0) != csr.n_src or n_dst != csr.n_dst:
        raise ValueError(f"gatv2: node counts ({x_l.size(0)}, {n_dst}) do not match the CSR "
                         f"({csr.n_src}, {csr.n_dst})")
    if x_l.size(1) != F or x_r.size(1) != F:
        raise ValueError("gatv2: projected features must be [*, heads*out_channels]")
    if out is None and (want_pre or not want_act):
        out = torch.empty(n_dst, F, dtype=torch.float32, device=dev)
    if want_act and out_act is None:
        out_act = torch.empty(n_dst, F, dtype=torch.float32, device=dev)
    smax = torch.empty(n_dst, H, dtype=torch.float32, device=dev)
    sden = torch.empty(n_dst, H, dtype=torch.float32, device=dev)
    att, bias = _vec(att.reshape(-1)), _vec(bias)
    seed_val, seed_dev = _split_seed(seed)
    e_logit = None
    if (want_logits and csr.E > 0 and n_dst > 0 and os.environ.get("SEGGER_B200_GAT_LOGITS", "1") != "0"
            and _quad_path(H, C, slope, x_l, x_r, att, bias, out, out_act)):
        e_logit = torch.empty(csr.E, H, dtype=torch.float32, device=dev)
    check(_lib.load().sgb_gatv2_fwd(ptr(x_l), _ld(x_l), ptr(x_r), _ld(x_r), ptr(att), ptr(bias), ptr(csr.rowptr),
                                    ptr(csr.col), ptr(csr.eid), n_dst, csr.E, H, C, slope, p_drop, seed_val,
                                    ptr(seed_dev), int(training), ptr(out), _ld(out) if out is not None else 0, ptr(out_act),
                                    _ld(out_act) if out_act is not None else 0, ptr(smax), ptr(sden), ptr(e_logit),
                                    stream_ptr(dev)), "gatv2_fwd")
    _count(1)
    if want_logits is not False:       # (None: "fifth element wanted, no logits" -- callers that always unpack five)
        return out, out_act, smax, sden, e_logit
    return out, out_act, smax, sden


def gatv2_bwd(x_l: Tensor, x_r: Tensor, att: Tensor, bias: Optional[Tensor], out_pre: Tensor, grad_out: Tensor,
              gelu_fused: bool, csr: EdgeCSR, H: int, C: int, slope: float, p_drop: float, training: bool,
              seed: int, smax: Tensor, sden: Tensor, grad_x_l: Optional[Tensor] = None,
              grad_x_r: Optional[Tensor] = None, e_logit: Optional[Tensor] = None):
    """-> (grad_x_l, grad_x_r, grad_att [H*C], grad_bias [H*C]).  ``e_logit``: what ``gatv2_fwd(want_logits=True)``
    returned for the same inputs (the dst pass then reads the logits back instead of recomputing them)."""
    if csr.t_rowptr is None:
        raise RuntimeError("gatv2_bwd needs the transposed CSR (build_csr(..., transpose=True))")
    x_l, x_r, out_pre, grad_out = _rowmajor(x_l), _rowmajor(x_r), _rowmajor(out_pre), _rowmajor(grad_out)
    F = H * C
    dev = x_r.device
    n_src, n_dst = csr.n_src, csr.n_dst
    if grad_x_l is None:
        grad_x_l = torch.empty(n_src, F, dtype=torch.float32, device=dev)
    if grad_x_r is None:
        grad_x_r = torch.empty(n_dst, F, dtype=torch.float32, device=dev)
    g_att = torch.empty(F, dtype=torch.float32, device=dev)
    g_bias = torch.empty(F, dtype=torch.float32, device=dev) if bias is not None else None
    g_buf = None
    if gelu_fused:
        g_buf = torch.empty(n_dst, _ld(grad_out), dtype=torch.float32, device=dev) if n_dst > 0 else grad_out
    lib = _lib.load()
    ws = _ws(lib.sgb_gatv2_bwd_workspace_bytes(n_dst, csr.E, H, C), dev)
    att, bias = _vec(att.reshape(-1)), _vec(bias)
    # one virtual source per edge: the dst pass writes grad_x_l itself (NULL transposed CSR) where the sub-warp kernels
    # apply -- the library's whole rule, slope included: elsewhere it needs the transposed pass
    direct = (csr.one_source_per_edge and n_dst > 0 and csr.E > 0 and os.environ.get("SEGGER_B200_GAT_DIRECT", "1") != "0"
              and _quad_path(H, C, slope, x_l, x_r, att, bias, out_pre, grad_out, g_buf, grad_x_l, grad_x_r))
    t_rowptr, t_dst, t_pos = (None, None, None) if direct else (csr.t_rowptr, csr.t_dst, csr.t_pos)
    seed_val, seed_dev = _split_seed(seed)
    if e_logit is not None and (n_dst == 0 or tuple(e_logit.shape) != (csr.E, H) or not e_logit.is_contiguous() or not
                                _quad_path(H, C, slope, x_l, x_r, att, bias, out_pre, grad_out, g_buf, grad_x_l, grad_x_r)):
        e_logit = None
    check(lib.sgb_gatv2_bwd(ptr(x_l), _ld(x_l), ptr(x_r), _ld(x_r), ptr(att), ptr(bias), ptr(out_pre), _ld(out_pre),
                            ptr(grad_out), _ld(grad_out), int(gelu_fused), ptr(g_buf), ptr(csr.rowptr), ptr(csr.col),
                            ptr(csr.eid), ptr(t_rowptr), ptr(t_dst), ptr(t_pos), n_src, n_dst, csr.E,
                            H, C, slope, p_drop, seed_val, ptr(seed_dev), int(training), ptr(smax), ptr(sden), ptr(e_logit),
                            ptr(grad_x_l),
                            _ld(grad_x_l), ptr(grad_x_r), _ld(grad_x_r), ptr(g_att), ptr(g_bias), ptr(ws),
                            ws.numel(), stream_ptr(dev)), "gatv2_bwd")
    _count(3)
    return grad_x_l, grad_x_r, g_att, g_bias


def gatv2_alpha(x_l, x_r, att, csr: EdgeCSR, H, C, slope, smax, sden) -> Tensor:
    x_l, x_r = _rowmajor(x_l), _rowmajor(x_r)
    alpha = torch.zeros(csr.E, H, dtype=torch.float32, device=x_r.device)
    att = _vec(att.reshape(-1))
    check(_lib.load().sgb_gatv2_alpha(ptr(x_l), _ld(x_l), ptr(x_r), _ld(x_r), ptr(att), ptr(csr.rowptr), ptr(csr.col),
                                      ptr(csr.eid), csr.n_dst, csr.E, H, C, slope, ptr(smax), ptr(sden), ptr(alpha),
                                      stream_ptr(x_r.device)), "gatv2_alpha")
    _count(1)
    return alpha


def dropout_keep_mask(seed: int, E: int, H: int, p: float, device) -> Tensor:
    """[E,H] bool keep mask identical to the one the fused kernels regenerate (test hook)."""
    mask = torch.empty(E, H, dtype=torch.uint8, device=device)
    seed, word = _split_seed(seed)
    if word is not None:          # test hook only: reading the word synchronises
        seed = (seed + int(word.item())) & (2 ** 64 - 1)
    check(_lib.load().sgb_dropout_mask(seed, E, H, p, ptr(mask), stream_ptr(device)), "dropout_mask")
    _count(1)
    return mask.bool()


# ------------------------------------------------------------------------------------------------
# autograd Functions
# ------------------------------------------------------------------------------------------------
class LinearFn(torch.autograd.Function):
    """y = act(x W^T + b) with a hand-written backward (dgrad + deterministic split-K wgrad)."""

    @staticmethod
    def forward(ctx, x, w, b, act, exact):
        require_cuda(x, w, b)
        lead = x.shape[:-1]
        x2 = x.reshape(-1, x.size(-1))
        y, y_act = linear_fwd(x2, w, b, act, exact=exact)
        ctx.act = act
        ctx.has_bias = b is not None
        ctx.lead = lead
        ctx.save_for_backward(x2, w, y if act != ACT_NONE else None)
        out = y_act if act != ACT_NONE else y
        return out.view(*lead, w.size(0))

    @staticmethod
    def backward(ctx, dout):
        x2, w, y = ctx.saved_tensors
        dy = dout.reshape(-1, w.size(0))
        if ctx.act != ACT_NONE:
            dy = act_bwd(dy, y, ctx.act)
        dx = linear_dgrad(dy, w).view(*ctx.lead, w.size(1)) if ctx.needs_input_grad[0] else None
        dw = db = None
        if ctx.needs_input_grad[1] or (ctx.has_bias and ctx.needs_input_grad[2]):
            dw, db = linear_wgrad(dy, x2, want_db=ctx.has_bias)
        return dx, dw, db, None, None


def linear(x: Tensor, w: Tensor, b: Optional[Tensor], act: int = ACT_NONE, exact: Optional[bool] = None) -> Tensor:
    # grad mode is decided HERE: inside autograd.Function.forward it always reads False
    if exact is None:
        exact = torch.is_grad_enabled()
    return LinearFn.apply(x, w, b, act, exact)


class GATv2AggregateFn(torch.autograd.Function):
    """Attention + softmax + aggregation (+bias, optional fused GELU) of one GATv2Conv."""

    @staticmethod
    def forward(ctx, x_l, x_r, att, bias, csr, H, C, slope, p_drop, training, seed, apply_gelu):
        require_cuda(x_l, x_r, att, bias)
        out, out_act, smax, sden, lg = gatv2_fwd(x_l, x_r, att, bias, csr, H, C, slope, p_drop, training, seed,
                                                 apply_gelu, want_logits=True if any(ctx.needs_input_grad[:4]) else None)
        ctx.csr, ctx.cfg = csr, (H, C, slope, p_drop, training, seed, apply_gelu)
        ctx.att_shape = att.shape
        ctx.save_for_backward(x_l, x_r, att, bias, out, smax, sden, lg)
        return out_act if apply_gelu else out

    @staticmethod
    def backward(ctx, dout):
        x_l, x_r, att, bias, out, smax, sden, lg = ctx.saved_tensors
        H, C, slope, p_drop, training, seed, apply_gelu = ctx.cfg
        gl, gr, ga, gb = gatv2_bwd(x_l, x_r, att, bias, out, dout.contiguous(), apply_gelu, ctx.csr, H, C, slope,
                                   p_drop, training, seed, smax, sden, e_logit=lg)
        return gl, gr, ga.view(ctx.att_shape), gb, None, None, None, None, None, None, None, None


class SkipGATLayerFn(torch.autograd.Function):
    """One hetero GATv2 layer of ISTEncoder fused end to end:

        Y_tx = x_tx [W_l^tt | W_r^tt | W_l^tb]^T + b      (one concatenated projection GEMM)
        Y_bd = x_bd W_r^tb^T + b
        h_tx = act(agg_tt(Y_tx[:, :F], Y_tx[:, F:2F]) + bias_tt)
        h_bd = act(agg_tb(Y_tx[:, 2F:], Y_bd) + bias_tb)

    which is HeteroConv({tt: GATv2Conv, tb: GATv2Conv}) (+ the following F.gelu when apply_gelu)
    of /root/reference/src/segger/models/ist_encoder.py:109-134,183-189,323-325.  The backward
    writes all three tx-side feature gradients into one [N, 3F] buffer so dgrad/wgrad are again
    single GEMMs.

    Source-subset variant: only transcripts that are sources of a belongs edge need W_l^tb.  When the
    belongs edge list names each source once in increasing order (setup_heterodata's nuclear-transcript
    list, data/utils/heterodata.py:147) the layer projects [W_l^tt | W_r^tt] over all N rows and W_l^tb
    over the E_tb gathered rows only, runs the tb conv on one virtual source per edge
    (EdgeCSR.per_edge_sources) and adds the input gradient of those rows back with rows_add.  Same
    arithmetic per element, a third fewer projection tiles (measured 22.05 -> 20.8 ms per step).
    """

    @staticmethod
    def forward(ctx, x_tx, x_bd, wl_tt, bl_tt, wr_tt, br_tt, att_tt, bias_tt, wl_tb, bl_tb, wr_tb, br_tb,
                att_tb, bias_tb, csr_tt, csr_tb, H, C, slope, p_drop, training, seed_tt, seed_tb, apply_gelu, exact,
                tx_ids=None, tx_table=None):
        """``tx_ids`` / ``tx_table`` (first layer only): the transcript input is cat(tx_table[tx_ids], x_tx) without that
        concatenation ever being built -- the table half of every tx-side projection is ``tx_table @ W[:, :D1]^T``
        ([n_genes, .], once per step) looked up per transcript in the GEMM epilogue, its weight gradient is a
        segment sum of the output gradient by gene id followed by an [n_genes]-row GEMM.  Half the reduction depth of
        the three largest GEMMs of the step."""
        require_cuda(x_tx, x_bd)
        F = H * C
        N, M = x_tx.size(0), x_bd.size(0)
        dev = x_tx.device
        D1 = tx_table.size(1) if tx_table is not None else 0
        # tx-belongs-bd sources only: when the belongs edge list names each source once (increasing), project just
        # those E_tb rows through tb.lin_l instead of all N transcripts (a third of the layer's projection GEMMs)
        # (the backward adds the row gradients back with a non-atomic rows_add and walks the transposed arrays in
        # edge order, hence "unique, increasing" -- without autograd any edge list qualifies and nothing is read back)
        subset = (F % 4 == 0 and x_tx.size(1) % 4 == 0 and 0 < csr_tb.E <= (3 * N) // 4
                  and (not exact or csr_tb.sources_unique_increasing()))
        ids_s = None

        def project(x, w, b, ids):
            """x w[:, D1:]^T + b (+ the table half, looked up by id)."""
            if D1 == 0:
                return linear_fwd(x, w, b, exact=exact)[0]
            tab, _ = linear_fwd(tx_table, w[:, :D1], None, exact=2)          # [n_genes, rows of w]: fp32 SIMT, tiny
            return linear_fwd(x, w[:, D1:], b, exact=exact, gather=(ids, tab))[0]

        if subset:
            w_cat = torch.cat([wl_tt, wr_tt], 0)
            b_cat = torch.cat([bl_tt, br_tt], 0)
            xs = gather_rows(x_tx, csr_tb.src_index)
            if D1:
                ids_s = tx_ids.index_select(0, csr_tb.src_index.long())     # index plumbing: ids of the belongs sources
            y_tb = project(xs, wl_tb, bl_tb, ids_s)
            csr_tb_run = csr_tb.per_edge_sources()
        else:
            w_cat = torch.cat([wl_tt, wr_tt, wl_tb], 0)
            b_cat = torch.cat([bl_tt, br_tt, bl_tb], 0)
            xs = None
            csr_tb_run = csr_tb
        y_tx = project(x_tx, w_cat, b_cat, tx_ids)
        if not subset:
            y_tb = y_tx[:, 2 * F:]
        y_bd, _ = linear_fwd(x_bd, wr_tb, br_tb, exact=exact)
        want_pre = bool(exact) or not apply_gelu      # `exact` = autograd is recording: the backward needs v
        # (`exact` = autograd is recording: the sub-warp forward then also leaves the raw logits for the backward)
        v_tx, h_tx, smax_tt, sden_tt, lg_tt = gatv2_fwd(y_tx[:, :F], y_tx[:, F:2 * F], att_tt, bias_tt, csr_tt, H, C,
                                                        slope, p_drop, training, seed_tt, apply_gelu, want_pre=want_pre,
                                                        want_logits=True if exact else None)
        v_bd, h_bd, smax_tb, sden_tb, lg_tb = gatv2_fwd(y_tb, y_bd, att_tb, bias_tb, csr_tb_run, H, C, slope,
                                                        p_drop, training, seed_tb, apply_gelu, want_pre=want_pre,
                                                        want_logits=True if exact else None)
        ctx.csr = (csr_tt, csr_tb, csr_tb_run)
        ctx.cfg = (H, C, slope, p_drop, training, seed_tt, seed_tb, apply_gelu, subset)
        ctx.att_shape = att_tt.shape
        ctx.D1 = D1
        ctx.save_for_backward(x_tx, x_bd, w_cat, wr_tb, y_tx, y_bd, v_tx, v_bd, att_tt, bias_tt, att_tb, bias_tb,
                              smax_tt, sden_tt, smax_tb, sden_tb, xs, y_tb if subset else None, wl_tb if subset else None,
                              tx_ids, tx_table, ids_s, lg_tt, lg_tb)
        if apply_gelu:
            return h_tx, h_bd
        return v_tx, v_bd

    @staticmethod
    def backward(ctx, d_tx, d_bd):
        (x_tx, x_bd, w_cat, wr_tb, y_tx, y_bd, v_tx, v_bd, att_tt, bias_tt, att_tb, bias_tb, smax_tt, sden_tt,
         smax_tb, sden_tb, xs, y_tb, wl_tb, tx_ids, tx_table, ids_s, lg_tt, lg_tb) = ctx.saved_tensors
        D1 = ctx.D1
        csr_tt, csr_tb, csr_tb_run = ctx.csr
        H, C, slope, p_drop, training, seed_tt, seed_tb, apply_gelu, subset = ctx.cfg
        F = H * C
        N, M = x_tx.size(0), x_bd.size(0)
        dev = x_tx.device
        if d_tx is None:
            d_tx = torch.zeros_like(v_tx)
        if d_bd is None:
            d_bd = torch.zeros_like(v_bd)
        g_tx = torch.empty(N, (2 if subset else 3) * F, dtype=torch.float32, device=dev)
        g_bd = torch.empty(M, F, dtype=torch.float32, device=dev)
        if subset:
            g_tb = torch.empty(csr_tb.E, F, dtype=torch.float32, device=dev)
        else:
            y_tb, g_tb = y_tx[:, 2 * F:], g_tx[:, 2 * F:]
        _, _, ga_tt, gb_tt = gatv2_bwd(y_tx[:, :F], y_tx[:, F:2 * F], att_tt, bias_tt, v_tx, d_tx.contiguous(),
                                       apply_gelu, csr_tt, H, C, slope, p_drop, training, seed_tt, smax_tt, sden_tt,
                                       grad_x_l=g_tx[:, :F], grad_x_r=g_tx[:, F:2 * F], e_logit=lg_tt)
        _, _, ga_tb, gb_tb = gatv2_bwd(y_tb, y_bd, att_tb, bias_tb, v_bd, d_bd.contiguous(), apply_gelu,
                                       csr_tb_run, H, C, slope, p_drop, training, seed_tb, smax_tb, sden_tb,
                                       grad_x_l=g_tb, grad_x_r=g_bd, e_logit=lg_tb)
        d_table = None
        n_genes = tx_table.size(0) if D1 else 0
        want_table = D1 > 0 and ctx.needs_input_grad[26]

        def back(g, x, w, ids):
            """-> (dx of the dense columns, dw [rows, D1 + D2], db) of y = x w[:, D1:]^T + table[ids] + b."""
            nonlocal d_table
            dx = linear_dgrad(g, w[:, D1:] if D1 else w) if ctx.needs_input_grad[0] else None
            dw_dense, db = linear_wgrad(g, x)
            if D1 == 0:
                return dx, dw_dense, db
            seg = segment_sum_rows(g, ids, n_genes)                        # [n_genes, rows]: sum of dL/dy by gene
            dw_tab, _ = linear_wgrad(seg, tx_table, want_db=False)         # [rows, D1]
            if want_table:
                dt = linear_dgrad(seg, w[:, :D1])                          # [n_genes, D1]
                d_table = dt if d_table is None else d_table.add_(dt)
            return dx, torch.cat([dw_tab, dw_dense], 1), db

        dx_tx, dw_cat, db_cat = back(g_tx, x_tx, w_cat, tx_ids)
        dx_bd = linear_dgrad(g_bd, wr_tb) if ctx.needs_input_grad[1] else None
        dwr_tb, dbr_tb = linear_wgrad(g_bd, x_bd)
        if subset:
            dxs, dwl_tb, dbl_tb = back(g_tb, xs, wl_tb, ids_s)
            if dx_tx is not None:
                rows_add(dx_tx, csr_tb.src_index, dxs)
        else:
            dwl_tb, dbl_tb = dw_cat[2 * F:], db_cat[2 * F:]
        return (dx_tx, dx_bd,
                dw_cat[:F], db_cat[:F], dw_cat[F:2 * F], db_cat[F:2 * F], ga_tt.view(ctx.att_shape), gb_tt,
                dwl_tb, dbl_tb, dwr_tb, dbr_tb, ga_tb.view(ctx.att_shape), gb_tb,
                None, None, None, None, None, None, None, None, None, None, None, None, d_table)


def sinusoid_freqs(dim: int, max_period: float, device) -> Tensor:
    """Frequency table of sinusoidal_embedding, computed with the reference's own formula
    (/root/reference/src/segger/models/ist_encoder.py:24-26) so the table is bit-identical."""
    half = dim // 2
    freqs = torch.exp(-math.log(max_period) * torch.arange(start=0, end=half, dtype=torch.float32) / half)
    return freqs.to(device)


def posfreq(pos: Tensor, batch: Optional[Tensor], n_batches: int, dim: int, freqs: Tensor) -> Tensor:
    """[2, N, dim] sinusoid features of the per-tile-normalised coordinates (x block, then y block)."""
    require_cuda(pos, batch)
    pos = pos.to(torch.float32).contiguous()
    N = pos.size(0)
    dev = pos.device
    feat = torch.empty(2, N, dim, dtype=torch.float32, device=dev)
    if batch is not None:
        if batch.dtype not in (torch.int32, torch.int64):
            batch = batch.long()
        batch = batch.contiguous()
    lib = _lib.load()
    ws = _ws(lib.sgb_posfreq_workspace_bytes(n_batches), dev)
    check(lib.sgb_posfreq_fwd(ptr(pos), N, ptr(batch), batch.element_size() if batch is not None else 0, n_batches,
                              dim, ptr(freqs), ptr(feat), dim, ptr(ws), ws.numel(), stream_ptr(dev)), "posfreq_fwd")
    _count(3)
    return feat


CHEB_DEG = 12   # basis columns of the low-rank positional front end (multiple of 4)


def cheb_feature_matrix(freqs: Tensor, deg: int = CHEB_DEG) -> Tensor:
    """Constant M [deg, 2*half] (fp32, on freqs' device) with  sinusoid(p) = T(2p-1) @ M  for p in [0,1]:
    column k < half holds the Chebyshev coefficients of cos(f_k (t+1)/2), column half+k those of
    sin(f_k (t+1)/2).  Computed in float64 by Chebyshev-Gauss quadrature; raises if the series is not
    converged to 1e-9 at ``deg`` (cannot happen for the reference's table, f_k <= 1)."""
    import numpy as np
    f = freqs.detach().double().cpu().numpy()
    m = 64
    j = np.arange(m)
    theta = np.pi * (j + 0.5) / m
    t = np.cos(theta)                                        # nodes
    arg = f[None, :] * (t[:, None] + 1.0) * 0.5              # [m, half]
    g = np.concatenate([np.cos(arg), np.sin(arg)], axis=1)   # [m, 2*half]
    n = np.arange(deg + 4)
    basis = np.cos(n[:, None] * theta[None, :])              # [deg+4, m]
    c = (2.0 / m) * basis @ g
    c[0] *= 0.5
    tail = float(np.abs(c[deg:]).max())
    if not tail < 1e-9:
        raise ValueError(f"Chebyshev series of the sinusoid features not converged at degree {deg} (tail {tail:.1e})")
    return torch.from_numpy(c[:deg].astype(np.float32)).to(freqs.device)


def poscheb(pos: Tensor, batch: Optional[Tensor], n_batches: int, deg: int = CHEB_DEG) -> Tensor:
    """[2N, deg] Chebyshev basis T_n(2p-1) of the per-tile-normalised coordinates (x rows, then y rows)."""
    require_cuda(pos, batch)
    pos = pos.to(torch.float32).contiguous()
    N = pos.size(0)
    dev = pos.device
    out = torch.empty(2 * N, deg, dtype=torch.float32, device=dev)
    if batch is not None:
        if batch.dtype not in (torch.int32, torch.int64):
            batch = batch.long()
        batch = batch.contiguous()
    lib = _lib.load()
    ws = _ws(lib.sgb_posfreq_workspace_bytes(n_batches), dev)
    check(lib.sgb_poscheb_fwd(ptr(pos), N, ptr(batch), batch.element_size() if batch is not None else 0, n_batches,
                              deg, ptr(out), deg, ptr(ws), ws.numel(), stream_ptr(dev)), "poscheb_fwd")
    _count(3)
    return out


class InputStageFn(torch.autograd.Function):
    """Input stage of ISTEncoder.forward for one node type
    (/root/reference/src/segger/models/ist_encoder.py:312-320):

        h = gelu( cat( first(x), pos_mlp(sinusoid(normalise(pos))) ) )

    ``first`` is an Embedding gather (tx: integer gene ids) or a Linear (bd: float features).
    GELU is applied per column block straight into the concatenated buffer.

    ``feat`` is either the [2, N, 256] sinusoid features (``coef`` None) or their low-rank form: the
    [2N, deg] Chebyshev basis from ``poscheb`` with ``coef`` = ``cheb_feature_matrix`` ([deg, 256]),
    sinusoid = feat @ coef.  In the low-rank form the first positional Linear runs as
    feat @ (w0 coef^T)^T and its weight gradient as (dy^T feat) coef: both contract over deg columns.
    """

    @staticmethod
    def forward(ctx, x, first_w, first_b, feat, w0, b0, w2, b2, is_embedding, exact, coef=None, skip_first=False):
        """``skip_first``: emit only the positional columns (the embedding half is consumed in factored form by the
        first SkipGAT layer, see SkipGATLayerFn)."""
        dev = first_w.device
        N = x.size(0)
        D = 0 if skip_first else (first_w.size(1) if is_embedding else first_w.size(0))
        use_pos = feat is not None
        dim = w2.size(0) if use_pos else 0
        h = torch.empty(N, D + 2 * dim, dtype=torch.float32, device=dev)
        lib = _lib.load()
        pre_first = None
        if skip_first:
            saved_x = None
        elif is_embedding:
            ids = x if x.dtype in (torch.int32, torch.int64) else x.long()
            ids = ids.contiguous()
            tab = first_w.contiguous()
            check(lib.sgb_embedding_fwd(ptr(tab), tab.size(0), D, ptr(ids), ids.element_size(), N, None, 0,
                                        ptr(h), _ld(h), ACT_GELU, stream_ptr(dev)), "embedding_fwd")
            _count(1)
            saved_x = ids
        else:
            x2 = _rowmajor(x.to(torch.float32))
            pre_first, _ = linear_fwd(x2, first_w, first_b, ACT_GELU, y_act=h[:, :D], exact=exact)
            saved_x = x2
        y0 = a0 = y2 = None
        if use_pos:
            f2 = feat.view(2 * N, feat.size(-1))
            w_in = w0
            if coef is not None:
                w_in, _ = linear_fwd(w0, coef, None, exact=exact)         # [dim, deg] = w0 coef^T
            y0, a0 = linear_fwd(f2, w_in, b0, ACT_SILU, exact=exact)       # [2N, dim] pre / SiLU
            y2 = torch.empty(2 * N, dim, dtype=torch.float32, device=dev)
            for d in range(2):                                            # x block, y block
                linear_fwd(a0[d * N:(d + 1) * N], w2, b2, ACT_GELU, y=y2[d * N:(d + 1) * N],
                           y_act=h[:, D + d * dim: D + (d + 1) * dim], exact=exact)
        ctx.is_embedding, ctx.use_pos, ctx.D, ctx.dim, ctx.N = is_embedding, use_pos, D, dim, N
        ctx.skip_first = skip_first
        ctx.has_first_b = first_b is not None
        ctx.save_for_backward(saved_x, first_w, pre_first, feat, w0, y0, a0, w2, y2, coef)
        return h

    @staticmethod
    def backward(ctx, dh):
        saved_x, first_w, pre_first, feat, w0, y0, a0, w2, y2, coef = ctx.saved_tensors
        N, D, dim = ctx.N, ctx.D, ctx.dim
        dev = dh.device
        dh = _rowmajor(dh)
        lib = _lib.load()
        d_first_w = d_first_b = dw0 = db0 = dw2 = db2 = None
        if ctx.skip_first:
            pass
        elif ctx.is_embedding:
            if ctx.needs_input_grad[1]:
                tab = first_w.contiguous()
                d_first_w = torch.empty_like(tab)
                ws = _ws(lib.sgb_embedding_bwd_workspace_bytes(N, D, tab.size(0)), dev)
                check(lib.sgb_embedding_bwd(ptr(dh), _ld(dh), ptr(saved_x), saved_x.element_size(), N, D,
                                            tab.size(0), ptr(tab), ACT_GELU, ptr(d_first_w), ptr(ws), ws.numel(),
                                            stream_ptr(dev)), "embedding_bwd")
                _count(10)
        else:
            dpre = act_bwd(dh[:, :D], pre_first, ACT_GELU)
            d_first_w, d_first_b = linear_wgrad(dpre, saved_x, want_db=ctx.has_first_b)
        if ctx.use_pos:
            dy2 = torch.empty(2 * N, dim, dtype=torch.float32, device=dev)
            for d in range(2):
                act_bwd(dh[:, D + d * dim: D + (d + 1) * dim], y2[d * N:(d + 1) * N], ACT_GELU,
                        dx=dy2[d * N:(d + 1) * N])
            dw2, db2 = linear_wgrad(dy2, a0)
            # SiLU' as a separate 128-bit streaming pass: fused into the dgrad epilogue its y0 loads are serialised
            # behind the tile write-out (0.91 ms fused vs 0.36 + 0.18 ms split on the 2M x 64 x 64 case)
            dy0 = linear_dgrad(dy2, w2)
            act_bwd(dy0, y0, ACT_SILU, dx=dy0)
            dw0, db0 = linear_wgrad(dy0, feat.view(2 * N, feat.size(-1)))
            if coef is not None:
                dw0 = linear_dgrad(dw0, coef)                             # [dim, deg] @ [deg, 256]
        return None, d_first_w, d_first_b, None, dw0, db0, dw2, db2, None, None, None, None


class OutputStageFn(torch.autograd.Function):
    """lin_last + F.normalize for one node type (ist_encoder.py:328-332)."""

    @staticmethod
    def forward(ctx, h, w, b, normalize):
        require_cuda(h, w, b)
        y, _ = linear_fwd(h, w, b, exact=False)   # nothing downstream amplifies its error
        ctx.normalize = normalize
        if not normalize:
            ctx.save_for_backward(h, w, None, None)
            return y
        M, D = y.shape
        e = torch.empty_like(y)
        nrm = torch.empty(M, dtype=torch.float32, device=y.device)
        check(_lib.load().sgb_l2norm_fwd(ptr(y), _ld(y), M, D, 1e-12, ptr(e), _ld(e), ptr(nrm), stream_ptr(y.device)),
              "l2norm_fwd")
        _count(1)
        ctx.save_for_backward(h, w, e, nrm)
        return e

    @staticmethod
    def backward(ctx, de):
        h, w, e, nrm = ctx.saved_tensors
        de = _rowmajor(de)
        if ctx.normalize:
            M, D = e.shape
            dy = torch.empty_like(e)
            check(_lib.load().sgb_l2norm_bwd(ptr(de), _ld(de), ptr(e), _ld(e), ptr(nrm), M, D, 1e-12, ptr(dy), _ld(dy),
                                             stream_ptr(e.device)), "l2norm_bwd")
            _count(1)
        else:
            dy = de
        dh = linear_dgrad(dy, w) if ctx.needs_input_grad[0] else None
        dw, db = linear_wgrad(dy, h)
        return dh, dw, db, None


# ------------------------------------------------------------------------------------------------
# scoring
# ------------------------------------------------------------------------------------------------
def candidate_csr(edge_index: Tensor, n_tx: int, n_bd: int) -> EdgeCSR:
    """Candidate CSR over transcripts for ``score_argmax``: the "destination" of the sort is the transcript row."""
    return build_csr(edge_index.flip(0), n_bd, n_tx, transpose=False)


def score_argmax(emb_tx: Tensor, emb_bd: Tensor, edge_index: Tensor, bd_index: Optional[Tensor],
                 min_similarity: Optional[float] = None, eps: float = 1e-8, csr: Optional[EdgeCSR] = None):
    """Fused cosine-similarity / scatter-max / cell lookup over candidate edges [2,E] (tx -> bd).

    Returns (max_sim fp32 [N_tx], max_idx int64 [N_tx] (E where a transcript has no candidate),
    seg_idx int64 [N_tx] (-1 where unassigned)) -- models/lightning_model.py:275-293.
    """
    require_cuda(emb_tx, emb_bd, edge_index, bd_index)
    emb_tx, emb_bd = _rowmajor(emb_tx), _rowmajor(emb_bd)
    n_tx, D = emb_tx.shape
    dev = emb_tx.device
    E = edge_index.size(1)
    if csr is None:
        csr = candidate_csr(edge_index, n_tx, emb_bd.size(0))
        validate_csrs(csr)
    max_sim = torch.empty(n_tx, dtype=torch.float32, device=dev)
    arg = torch.empty(n_tx, dtype=torch.int64, device=dev)
    seg = torch.empty(n_tx, dtype=torch.int64, device=dev)
    if bd_index is not None:
        if bd_index.dtype not in (torch.int32, torch.int64):
            bd_index = bd_index.long()
        bd_index = bd_index.contiguous()
    ms = float("nan") if min_similarity is None else float(min_similarity)
    check(_lib.load().sgb_score_argmax(ptr(emb_tx), _ld(emb_tx), ptr(emb_bd), _ld(emb_bd), D, ptr(csr.rowptr),
                                       ptr(csr.col), ptr(csr.eid), n_tx, E, eps, ptr(bd_index),
                                       bd_index.element_size() if bd_index is not None else 0, ms, ptr(max_sim),
                                       ptr(arg), ptr(seg), stream_ptr(dev)), "score_argmax")
    _count(1)
    return max_sim, arg, seg


def compact_predictions(mask: Tensor, src_idx: Tensor, seg_idx: Tensor, max_sim: Tensor, gene: Tensor):
    """(src_idx[mask], seg_idx[mask], max_sim[mask], gene[mask]) in one pass: -> (out_src, out_seg, out_sim, out_gene,
    count) with the outputs sized like the inputs (``count`` rows valid, device int32 scalar).  The index plumbing
    at the end of predict_step (models/lightning_model.py:294-298)."""
    require_cuda(mask, src_idx, seg_idx, max_sim, gene)
    n = mask.numel()
    dev = mask.device
    m8 = mask.contiguous().view(torch.uint8) if mask.dtype == torch.bool else (mask != 0).contiguous().view(torch.uint8)
    src_idx = src_idx.to(torch.int64).contiguous()
    seg_idx = seg_idx.to(torch.int64).contiguous()
    max_sim = max_sim.to(torch.float32).contiguous()
    if gene.dtype not in (torch.int32, torch.int64):
        gene = gene.to(torch.int64)
    gene = gene.contiguous()
    o_src, o_seg = torch.empty_like(src_idx), torch.empty_like(seg_idx)
    o_sim, o_gene = torch.empty_like(max_sim), torch.empty_like(gene)
    count = torch.empty(1, dtype=torch.int32, device=dev)
    lib = _lib.load()
    ws = _ws(lib.sgb_select_workspace_bytes(n), dev)
    check(lib.sgb_compact_predictions(ptr(m8), n, ptr(src_idx), ptr(seg_idx), ptr(max_sim), ptr(gene), gene.element_size(),
                                      ptr(o_src), ptr(o_seg), ptr(o_sim), ptr(o_gene), ptr(count), ptr(ws), ws.numel(),
                                      stream_ptr(dev)), "compact_predictions")
    _count(5)
    return o_src, o_seg, o_sim, o_gene, count
