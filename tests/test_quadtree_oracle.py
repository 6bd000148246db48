"""CPU checks of oracle/quadtree_ref.py on its own (the tree's invariants, known answers on hand-built sets) and of the
host helpers of segger_b200.tiles.QuadTreeTiling."""
import numpy as np
import pytest

from oracle import quadtree_ref as Q


def _points(kind, n, seed):
    rng = np.random.default_rng(seed)
    if kind == "uniform":
        return rng.uniform(0, 3000, (n, 2)).astype(np.float32)
    c = rng.uniform(0, 3000, (max(1, n // 100), 2))
    return (c[rng.integers(0, c.shape[0], n)] + rng.normal(0, 3.0, (n, 2))).astype(np.float32)


def _key_range(t, i):
    """Morton key range [start, end) of leaf i at full depth."""
    D, L = t["max_depth"], int(t["levels"][i])
    qx, qy = int(t["qx"][i]), int(t["qy"][i])
    k = 0
    for b in range(L):
        k |= ((qx >> b) & 1) << (2 * b) | ((qy >> b) & 1) << (2 * b + 1)
    return k << 2 * (D - L), (k + 1) << 2 * (D - L)


@pytest.mark.parametrize("kind,n,S,D", [("uniform", 20000, 700, 15), ("clustered", 30000, 500, 15), ("clustered", 20000, 300, 4)])
def test_tree_invariants(kind, n, S, D):
    p = _points(kind, n, seed=n + S)
    t = Q.build(p, S, D)
    P = len(t["counts"])
    lab = t["labels"]
    # every point in exactly one leaf, counts agree
    assert lab.min() >= 0 and lab.max() < P
    assert np.array_equal(np.bincount(lab, minlength=P), t["counts"])
    # leaves disjoint (key ranges ascending = Morton order, non-overlapping), inside the root, and cover every point
    rngs = [_key_range(t, i) for i in range(P)]
    assert all(rngs[i][1] <= rngs[i + 1][0] for i in range(P - 1))
    xmin, ymin, scale = t["root"]
    side = scale * 2 ** D
    assert (t["boxes"][:, 0] >= xmin).all() and (t["boxes"][:, 2] <= xmin + side).all()
    assert (t["boxes"][:, 1] >= ymin).all() and (t["boxes"][:, 3] <= ymin + side).all()
    ix, iy = Q.cells(p[:, 0], xmin, scale, D), Q.cells(p[:, 1], ymin, scale, D)
    for i in range(P):                                  # each point's cell lies in its leaf's quadrant
        sh = D - int(t["levels"][i])
        m = lab == i
        assert ((ix[m] >> sh) == t["qx"][i]).all() and ((iy[m] >> sh) == t["qy"][i]).all()
    # every point in the closed box of its leaf
    b = t["boxes"][lab]
    pd = p.astype(np.float64)
    assert ((pd[:, 0] >= b[:, 0]) & (pd[:, 0] <= b[:, 2]) & (pd[:, 1] >= b[:, 1]) & (pd[:, 1] <= b[:, 3])).all()
    # size rule: a leaf holds <= S points unless at depth D; every split parent holds > S
    assert ((t["counts"] <= S) | (t["levels"] == D)).all()
    for i in range(P):
        L = int(t["levels"][i])
        if L == 0:
            continue
        sh = D - L + 1
        parent = ((ix >> sh) == (t["qx"][i] >> 1)) & ((iy >> sh) == (t["qy"][i] >> 1))
        assert parent.sum() > S
    assert Q.label(t, p).tolist() == lab.tolist()


def test_four_clusters_known_answer():
    rng = np.random.default_rng(0)
    pts = []
    for cx, cy in ((0.25, 0.25), (0.75, 0.25), (0.25, 0.75), (0.75, 0.75)):
        pts.append(np.column_stack([cx + rng.uniform(-0.1, 0.1, 10), cy + rng.uniform(-0.1, 0.1, 10)]))
    pts[0][0] = (0.0, 0.0)
    pts[3][0] = (1.0, 1.0)
    t = Q.build(np.concatenate(pts), max_tile_size=10, max_depth=15)
    assert t["labels"].tolist() == [0] * 10 + [1] * 10 + [2] * 10 + [3] * 10
    assert t["boxes"].tolist() == [[0, 0, .5, .5], [.5, 0, 1, .5], [0, .5, .5, 1], [.5, .5, 1, 1]]
    assert t["levels"].tolist() == [1] * 4 and t["counts"].tolist() == [10] * 4


def test_duplicates_single_point_and_empty_input():
    t = Q.build(np.tile([[3.0, 4.0]], (100, 1)), max_tile_size=10, max_depth=5)
    assert t["counts"].tolist() == [100] and t["levels"].tolist() == [5]          # depth-D leaf over the limit
    assert t["boxes"].tolist() == [[3.0, 4.0, 3.0 + 1 / 32, 4.0 + 1 / 32]]
    t = Q.build(np.array([[2.5, -1.0]]), max_tile_size=10, max_depth=15)
    assert t["counts"].tolist() == [1] and t["levels"].tolist() == [0] and t["boxes"].tolist() == [[2.5, -1.0, 3.5, 0.0]]
    t = Q.build(np.zeros((0, 2)), max_tile_size=10, max_depth=15)
    assert len(t["counts"]) == 0 and t["labels"].shape == (0,)
    with pytest.raises(ValueError):
        Q.build(np.zeros((1, 2)), max_depth=16)


def test_points_exactly_on_cell_edges():
    D = 3
    base = np.array([[0.0, 0.0], [0.7, 0.7]])
    xmin, ymin, scale = Q.root_of(base, D)
    edges = xmin + np.arange(2 ** D + 1, dtype=np.float64) * scale
    below = np.nextafter(edges, -np.inf)
    xs = np.concatenate([edges, below, edges + scale / 2])
    c = Q.cells(xs, xmin, scale, D)
    lo = xmin + c * scale
    hi = xmin + (c + 1) * scale
    inside = (xs >= 0) & (xs < edges[-1])
    assert ((lo <= xs) & (xs < hi))[inside].all()
    assert c[:2 ** D].tolist() == list(range(2 ** D))                              # x = edge(c) lands in cell c
    assert c[2 ** D] == 2 ** D - 1 and c[2 ** D + 1] == 0                          # rim clamps
    # a leaf boundary on an edge: points on it belong to the right / upper leaf
    pts = np.array([[0.0, 0.0], [0.35, 0.1], [0.7, 0.7], [0.1, 0.35], [0.5, 0.5]])
    t = Q.build(pts, max_tile_size=1, max_depth=1)
    assert t["labels"].tolist() == [0, 1, 3, 2, 3]


def test_margin_halving_and_fit_mask():
    boxes = np.array([[0.0, 0.0, 1.0, 10.0], [0.0, 0.0, 10.0, 10.0], [0.0, 0.0, 0.1, 0.1]])
    m = Q.margins(boxes, 0.75)
    assert m.tolist() == [0.375, 0.75, 0.75 / 16]
    assert Q.margins(boxes, 0.0).tolist() == [0.0, 0.0, 0.0]
    t = dict(boxes=boxes[:1])
    pts = np.array([[0.375, 5.0], [0.37, 5.0], [0.625, 0.375], [0.626, 5.0], [0.5, 9.625], [0.5, 9.7]])
    got = Q.fit_mask(t, pts, np.zeros(6, dtype=np.int32), 0.75)
    assert got.tolist() == [True, False, True, False, True, False]
    assert Q.fit_mask(t, pts[:1], np.array([-1], dtype=np.int32), 0.75).tolist() == [False]


def test_label_of_other_points():
    pts = np.array([[0.0, 0.0], [0.1, 0.1], [0.2, 0.1], [1.0, 1.0]])
    t = Q.build(pts, max_tile_size=2, max_depth=2)
    # (0,0)-quadrant split again; (1,1)-quadrant a leaf; (1,0) and (0,1) empty
    q = np.array([[0.05, 0.05], [0.9, 0.1], [0.9, 0.9], [-5.0, -5.0], [5.0, 5.0], [0.1, 0.9]])
    lab = Q.label(t, q)
    assert lab[1] == -1 and lab[5] == -1
    assert lab[2] == lab[4] == t["labels"][3]
    assert lab[0] == lab[3] == t["labels"][0]


def test_host_margins_match_oracle_and_span_merge():
    import torch
    from segger_b200 import tiles
    boxes = np.array([[0.0, 0.0, 1.0, 10.0], [0.0, 0.0, 10.0, 10.0], [0.0, 0.0, 0.1, 0.1], [-3.0, 2.0, -2.9, 7.0]])
    for margin in (0.0, 0.75, 20.0):
        assert tiles.fit_margins(torch.from_numpy(boxes), margin).tolist() == Q.margins(boxes, margin).tolist()
    spans = [(0, 2), (5, 6), (7, 9), (20, 21)]
    assert tiles._merge_spans(spans, 8) == spans
    assert tiles._merge_spans(spans, 3) == [(0, 2), (5, 9), (20, 21)]
    assert tiles._merge_spans(spans, 0) == [(0, 21)]
