"""CPU tests of the kNN search without a radius cap and with k > 32: the oracle's canonical table against brute
force, and the host-side argument checks of the ring-search entry points (no CUDA call is reached)."""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest

from oracle import neighbors_ref
from segger_b200 import _lib
from segger_b200._lib import KnnPlan

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RING = ("sgb_knn2d_ring_plan", "sgb_knn2d_ring_workspace_bytes", "sgb_knn2d_ring")


@pytest.mark.parametrize("n,k,r", [(3000, 64, np.inf), (3000, 200, np.inf), (3000, 200, 5.0), (40, 100, np.inf),
                                   (40, 100, 5.0), (1, 33, np.inf)])
def test_canonical_table_matches_brute_force_without_radius_cap(n, k, r):
    rng = np.random.default_rng(n + k)
    side = (n / 0.5) ** 0.5
    pts = rng.uniform(0, side, (n, 2)).astype(np.float32)
    qry = rng.uniform(-20, side + 20, (300, 2))
    for q in (None, qry):
        canon, _, _, _ = neighbors_ref.canonical_knn_table(pts, k, r, query=q)
        assert np.array_equal(canon, neighbors_ref.brute_force_knn_table(pts, k, r, query=q))
    if n < k and r == np.inf:                         # every row holds every point, then padding
        assert (canon[:, n:] == n).all() and (np.sort(canon[:, :n], 1) == np.arange(n)).all()


def test_canonical_table_ties_without_radius_cap():
    g = np.arange(12, dtype=np.float64)
    lattice = np.stack(np.meshgrid(g, g), -1).reshape(-1, 2)
    canon, n_tie, _, _ = neighbors_ref.canonical_knn_table(lattice, 50, np.inf)
    assert n_tie > 0
    assert np.array_equal(canon, neighbors_ref.brute_force_knn_table(lattice, 50, np.inf))


@pytest.mark.parametrize("k,r,what", [(0, 5.0, b"k=0"), (1025, 5.0, b"k=1025"), (33, math.nan, b"max_dist"),
                                      (33, 0.0, b"max_dist"), (33, -1.0, b"max_dist"), (33, -math.inf, b"max_dist")])
def test_ring_plan_rejects_out_of_range_arguments_without_gpu(lib, k, r, what):
    plan = KnnPlan()
    assert lib.sgb_knn2d_ring_plan(None, 0, 10, None, 0, k, r, C.byref(plan), None, None) == -1   # SGB_ERR_ARG
    msg = lib.sgb_last_error()
    assert what in msg and (b"1..1024" in msg if k != 33 else b"> 0" in msg)


def test_ring_plan_and_run_accept_the_full_range_without_gpu(lib):
    # k = 1024 and an infinite radius pass the checks; with no points the plan needs no device work
    plan = KnnPlan()
    assert lib.sgb_knn2d_ring_plan(None, 0, 0, None, 0, 1024, math.inf, C.byref(plan), None, None) == 0
    assert plan.k == 1024 and plan.max_dist == math.inf and plan.n_query == 0
    assert lib.sgb_knn2d_ring(C.byref(plan), None, 0, None, None, None, None, 0, None) == 0   # nothing to do
    assert lib.sgb_knn2d_ring_workspace_bytes(C.byref(plan)) > 0
    plan.k = 2000                                                                             # a corrupted plan
    assert lib.sgb_knn2d_ring(C.byref(plan), None, 0, None, None, None, None, 0, None) == -1
    # the register kernel keeps its own range
    assert lib.sgb_knn2d_plan(None, 0, 10, None, 0, 33, 5.0, C.byref(plan), None, None) == -1
    assert lib.sgb_knn2d_plan(None, 0, 10, None, 0, 5, math.inf, C.byref(plan), None, None) == -1


def test_ring_entry_points_declared_and_bound():
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "segger_b200.h")).read(), flags=re.S)
    for name in RING:
        m = re.search(r"\b%s\s*\((.*?)\)\s*;" % name, src, flags=re.S)
        assert m and name in _lib.EXPORTED_SYMBOLS, name
        assert len(m.group(1).split(",")) == len(_lib._PROTOS[name][1]), name
    assert _lib._PROTOS["sgb_knn2d_ring_plan"][1] == _lib._PROTOS["sgb_knn2d_plan"][1]
    assert _lib._PROTOS["sgb_knn2d_ring"][1] == _lib._PROTOS["sgb_knn2d"][1]
