"""GPU tests of the ring-search kNN (sgb_knn2d_ring: any k <= 1024, any radius up to inf), bit-exact against scipy's
cKDTree in the canonical (d^2, index) order, and of edge offsets past 2^31 edges."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from oracle import neighbors_ref
from segger_b200 import _lib
from segger_b200._lib import check, ptr, stream_ptr
from segger_b200.neighbors import _knn_table, kdtree_neighbors, knn_table, setup_prediction_graph

pytestmark = pytest.mark.gpu
INF = math.inf


def _points(kind, n, dtype, seed):
    rng = np.random.default_rng(seed)
    side = (n / 0.5) ** 0.5                                              # 0.5 points / um^2
    if kind == "uniform":
        return rng.uniform(0, side, (n, 2)).astype(dtype)
    c = rng.uniform(0, side, (max(1, n // 100), 2))                      # ~100 points per cluster, sigma 3 um
    return (c[rng.integers(0, c.shape[0], n)] + rng.normal(0, 3.0, (n, 2))).astype(dtype)


def _check_ring(points, k, r, query=None):
    """The ring search against scipy, table and count compared as test_gpu_encoder._check_knn does."""
    table, count = _knn_table(points, k, r, query, None, True)
    canon, n_tie, _, _ = neighbors_ref.canonical_knn_table(points, k, r, query=query)
    got = table.cpu().numpy()
    assert got.shape == canon.shape
    assert np.array_equal(got, canon), f"{(got != canon).any(1).sum()} rows differ"
    assert np.array_equal(count.cpu().numpy(), (canon != points.shape[0]).sum(1))
    return n_tie, got


@pytest.mark.parametrize("kind", ["uniform", "clustered"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("r", [5.0, INF])
@pytest.mark.parametrize("k", [1, 33, 64, 200, 1024])
def test_ring_bit_exact_vs_scipy(k, r, dtype, kind):
    n = 20000 if k <= 64 else 6000
    pts = _points(kind, n, dtype, seed=k + (7 if r == INF else 0))
    _check_ring(pts, k, r)


@pytest.mark.parametrize("k,r", [(1, INF), (64, INF), (300, INF), (40, 5.0), (40, 60.0)])
def test_ring_queries_outside_the_box_and_far_from_any_point(k, r):
    pts = _points("clustered", 8000, np.float32, seed=3)
    hi = pts.max(0)
    rng = np.random.default_rng(4)
    qry = np.concatenate([rng.uniform(-50, hi + 50, (1500, 2)),                     # around and beyond the box
                          rng.uniform(-3000, -2000, (20, 2)),                        # far outside, many rings
                          np.array([[hi[0] / 2, 1e4], [-1e4, hi[1] / 2], [1e4, 1e4]])]).astype(np.float32)
    _check_ring(pts, k, r, query=qry)
    # fp64 queries over fp32 points: both promoted to fp64, as knn_table does
    _check_ring(pts, k, r, query=qry.astype(np.float64) + 0.1)


@pytest.mark.parametrize("r", [5.0, INF])
def test_ring_fewer_points_than_k_pads_rows(r):
    pts = _points("uniform", 50, np.float32, seed=5)
    _, got = _check_ring(pts, 200, r)
    assert (got[:, 50:] == 50).all()
    if r == INF:
        assert (np.sort(got[:, :50], 1) == np.arange(50)).all()
    t0, c0 = _knn_table(np.zeros((0, 2), np.float32), 64, r, pts, None, True)
    assert (t0 == 0).all() and (c0 == 0).all() and t0.shape == (50, 64)     # no points: all padding


def test_ring_exact_ties_and_coincident_points():
    g = np.arange(40, dtype=np.float32)
    lattice = np.stack(np.meshgrid(g, g), -1).reshape(-1, 2)            # massive exact ties at every k-th distance
    for k, r in ((64, INF), (64, 3.5), (200, INF), (33, 4.0)):
        n_tie, _ = _check_ring(lattice, k, r)
        assert n_tie > 0
    pts = _points("uniform", 3000, np.float32, seed=6)
    pts[100:180] = pts[100]                                             # 80 coincident points
    pts[500:540] = pts[501]
    for k, r in ((64, INF), (100, 5.0), (1024, INF)):
        _check_ring(pts, k, r)


def test_ring_point_at_exactly_max_dist_is_excluded():
    ex = np.array([[0, 0], [5, 0], [0, 3], [100, 100]], dtype=np.float32)
    t, c = _knn_table(ex, 40, 5.0, None, None, True)
    assert t[:, :3].cpu().tolist() == [[0, 2, 4], [1, 4, 4], [2, 0, 4], [3, 4, 4]]
    assert (t[:, 3:] == 4).all() and c.cpu().tolist() == [2, 1, 2, 1]
    t, c = knn_table(ex, 3, INF)                                        # no cap: the point at 5 is in
    assert t.cpu().tolist() == [[0, 2, 1], [1, 0, 2], [2, 0, 1], [3, 1, 2]] and (c == 3).all()


@pytest.mark.parametrize("k", [1, 5, 20, 32])
@pytest.mark.parametrize("kind", ["uniform", "clustered"])
def test_ring_equals_register_kernel_for_small_k(k, kind):
    pts = _points(kind, 50000, np.float32, seed=k)
    qry = np.random.default_rng(k).uniform(-20, pts.max() + 20, (5000, 2)).astype(np.float32)
    for q in (None, qry):
        a, ca = _knn_table(pts, k, 5.0, q, None, False)
        b, cb = _knn_table(pts, k, 5.0, q, None, True)
        assert torch.equal(a, b) and torch.equal(ca, cb)


def test_public_entry_points_route_large_k_and_infinite_radius():
    pts = _points("uniform", 20000, np.float32, seed=9)
    for k, r in ((50, 5.0), (5, INF)):                                  # both raised before
        ei, none = kdtree_neighbors(pts, k, r)
        canon, _, _, _ = neighbors_ref.canonical_knn_table(pts, k, r)
        ce, _ = neighbors_ref.knn_to_edge_index(torch.from_numpy(canon), padding_value=pts.shape[0])
        assert none is None and torch.equal(ei, ce)
    with pytest.raises(RuntimeError, match="1..1024"):
        knn_table(pts, 1025, 5.0)
    with pytest.raises(RuntimeError, match="max_dist"):
        knn_table(pts, 40, math.nan)


def test_uniform_prediction_graph_k64_equals_scipy():
    tx = _points("clustered", 30000, np.float32, seed=11)
    rng = np.random.default_rng(12)
    cen = np.concatenate([rng.uniform(0, tx.max(), (300, 2)), [[-500.0, -500.0]]])   # one far from every point
    ei = setup_prediction_graph(tx, cen, 64, 0, mode="uniform")
    canon, _, _, _ = neighbors_ref.canonical_knn_table(tx, 64, INF, query=cen)
    ce, _ = neighbors_ref.knn_to_edge_index(torch.from_numpy(canon), padding_value=tx.shape[0])
    assert ei.shape == (2, 301 * 64) and torch.equal(ei, ce)


def _count_edges(count):
    lib = _lib.load()
    n = count.numel()
    index_ptr = torch.empty(n + 1, dtype=torch.int64, device="cuda")
    ws = torch.empty(max(int(lib.sgb_knn_coo_workspace_bytes(n)), 16), dtype=torch.uint8, device="cuda")
    n_edges = C.c_int64(0)
    check(lib.sgb_knn_count_edges(ptr(count), n, ptr(index_ptr), C.byref(n_edges), ptr(ws), ws.numel(),
                                  stream_ptr()), "knn_count_edges")
    return index_ptr, int(n_edges.value)


def test_count_edges_offsets_exact_past_2_31():
    n = 70_000_000
    index_ptr, E = _count_edges(torch.full((n,), 31, dtype=torch.int32, device="cuda"))
    assert E == 31 * n > 2 ** 31 and int(index_ptr[-1]) == E and int(index_ptr[0]) == 0
    rows = torch.cat([torch.tensor([1, 2047, 2048, 69_273_666, 69_273_667, n - 1, n]),
                      torch.randint(0, n + 1, (10000,), generator=torch.Generator().manual_seed(0))]).cuda()
    assert torch.equal(index_ptr[rows], rows * 31)
    del index_ptr
    # mixed counts below 2^31: the same offsets as an int64 cumulative sum
    gen = torch.Generator("cuda").manual_seed(1)
    c = torch.randint(0, 1025, (3_000_001,), dtype=torch.int32, device="cuda", generator=gen)
    index_ptr, E = _count_edges(c)
    ref = torch.cat([torch.zeros(1, dtype=torch.int64, device="cuda"), c.long().cumsum(0)])
    assert torch.equal(index_ptr, ref) and E == int(ref[-1])
