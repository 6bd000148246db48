"""GPU parity of quadtree tiling (sgb_quadtree.cu, segger_b200.tiles.QuadTreeTiling) against oracle/quadtree_ref.py --
bit-exact -- and the tiling driving TilePartition, TilePredictSet (per tile and grouped cut) and a training step."""
import numpy as np
import pytest
import torch

from oracle import quadtree_ref as Q
from oracle import tiles_ref
from segger_b200 import tiles
from segger_b200.lightning_model import LitISTEncoder
from tests.test_gpu_tiles import _graph
from tests.util import PRED, TB, TT

pytestmark = pytest.mark.gpu


def _points(kind, n, seed):
    rng = np.random.default_rng(seed)
    side = (n / 0.5) ** 0.5                                  # Xenium-like density, 0.5 points / um^2
    if kind == "uniform":
        return rng.uniform(0, side, (n, 2)).astype(np.float32)
    c = rng.uniform(0, side, (max(1, n // 100), 2))
    return (c[rng.integers(0, c.shape[0], n)] + rng.normal(0, 3.0, (n, 2))).astype(np.float32)


def _check_tree(qt, ref, pts_dev):
    assert len(qt) == len(ref["counts"])
    assert torch.equal(qt.labels.cpu(), torch.from_numpy(ref["labels"]))
    assert torch.equal(qt.tiles.cpu(), torch.from_numpy(ref["boxes"]))
    assert qt.counts.cpu().tolist() == ref["counts"].tolist()
    assert qt.levels.cpu().tolist() == ref["levels"].tolist()
    assert qt.root.cpu().tolist() == list(ref["root"])
    # every point in the closed box of its own tile
    b = qt.tiles[qt.labels.long()]
    p = pts_dev.double()
    assert bool(((p[:, 0] >= b[:, 0]) & (p[:, 0] <= b[:, 2]) & (p[:, 1] >= b[:, 1]) & (p[:, 1] <= b[:, 3])).all())


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("kind", ["uniform", "clustered"])
def test_build_bit_exact_vs_oracle(kind, dtype):
    pts = _points(kind, 300_000, seed=1 if kind == "uniform" else 2)
    if dtype == torch.float64:
        pts = pts.astype(np.float64) + np.random.default_rng(3).uniform(0, 1e-3, pts.shape)
    dev = torch.from_numpy(pts).cuda()
    for S, D in ((5_000, 15), (700, 15), (2_000, 3)):
        qt = tiles.QuadTreeTiling(dev, max_tile_size=S, max_depth=D)
        ref = Q.build(pts, S, D)
        _check_tree(qt, ref, dev)
        # other points: inside, outside the root (rim clamp), in empty quadrants (-1)
        q = np.concatenate([pts[::97], pts[:50] * 3 - 100.0]).astype(pts.dtype)
        assert qt.label(torch.from_numpy(q).cuda()).cpu().tolist() == Q.label(ref, q).tolist()


def test_build_20m_clustered_bit_exact():
    pts = _points("clustered", 20_000_000, seed=4)
    dev = torch.from_numpy(pts).cuda()
    qt = tiles.QuadTreeTiling(dev)
    _check_tree(qt, Q.build(pts, 50_000, 15), dev)


def test_small_and_degenerate_inputs():
    for pts, S, D in ((np.tile([[3.0, 4.0]], (100, 1)), 10, 5), (np.array([[2.5, -1.0]]), 10, 15), (np.zeros((0, 2)), 10, 15),
                      (np.array([[0.0, 0.0], [0.35, 0.1], [0.7, 0.7], [0.1, 0.35], [0.5, 0.5]]), 1, 1)):
        dev = torch.from_numpy(pts.astype(np.float32)).cuda()
        qt = tiles.QuadTreeTiling(dev, max_tile_size=S, max_depth=D)
        _check_tree(qt, Q.build(pts.astype(np.float32), S, D), dev)
    with pytest.raises(ValueError):
        tiles.QuadTreeTiling(dev, max_depth=16)


def _tiling_and_graph(n_tx, n_cells, seed, S):
    ts, nodes, edges, b = _graph(n_tx=n_tx, n_cells=n_cells, seed=seed)
    bc = b.cuda()
    qt = tiles.QuadTreeTiling({"tx": bc["tx"]["pos"], "bd": bc["bd"]["pos"]}, max_tile_size=S)
    return ts, nodes, edges, b, bc, qt


def test_fit_labels_and_masks_vs_oracle_and_tile_partition():
    ts, nodes, edges, b, bc, qt = _tiling_and_graph(12000, 120, 0, 1500)
    allpos = np.concatenate([nodes["tx"]["pos"].numpy(), nodes["bd"]["pos"].numpy()])
    ref = Q.build(allpos, 1500, 15)
    n_tx = nodes["tx"]["pos"].size(0)
    assert torch.equal(qt.labels["tx"].cpu(), torch.from_numpy(ref["labels"][:n_tx]))
    assert torch.equal(qt.labels["bd"].cpu(), torch.from_numpy(ref["labels"][n_tx:]))
    for margin in (10.0, 1e4):                                   # 1e4: halved on every tile
        labels, masks = qt.fit_labels_and_masks(bc, margin)
        for nt in ("tx", "bd"):
            assert torch.equal(labels[nt], qt.labels[nt])
            p = nodes[nt]["pos"].numpy()
            want = Q.fit_mask(ref, p, Q.label(ref, p), margin)
            assert masks[nt].dtype == torch.bool and masks[nt].cpu().tolist() == want.tolist(), (nt, margin)
        if margin == 10.0:
            assert 0 < int(masks["tx"].sum()) < n_tx
    # bd labelled against a tree over transcripts only: same cell rule, -1 in empty quadrants
    qt_tx = tiles.QuadTreeTiling(bc["tx"]["pos"], max_tile_size=1500)
    ref_tx = Q.build(nodes["tx"]["pos"].numpy(), 1500, 15)
    assert qt_tx.label(bc["bd"]["pos"]).cpu().tolist() == Q.label(ref_tx, nodes["bd"]["pos"].numpy()).tolist()
    # TilePartition on quadtree labels == the oracle partition
    lab = {nt: qt.labels[nt] for nt in ("tx", "bd")}
    P = len(qt)
    part = tiles.TilePartition(bc, lab, P)
    rn, re, indptr, e_indptr, perm = tiles_ref.partition_ref(nodes, edges, {k: v.cpu() for k, v in lab.items()}, P)
    for nt in ("tx", "bd"):
        assert part.node_indptr[nt] == indptr[nt].tolist()
        assert torch.equal(part.node_perm[nt].cpu().long(), perm[nt])
        for k, v in rn[nt].items():
            assert torch.equal(part.data[nt][k].cpu(), v), (nt, k)
    for et in (TT, TB, PRED):
        assert part.edge_indptr[et] == e_indptr[et].tolist(), et
        assert torch.equal(part.data[et]["edge_index"].cpu().long(), re[et]), et


def test_predict_subsets_and_grouped_cut_on_quadtree_tiles():
    for pos_dtype, e_dtype, margin in ((torch.float32, torch.int64, 15.0), (torch.float64, torch.int32, 45.0)):
        ts, nodes, edges, b = _graph(n_tx=40000, n_cells=400, seed=9)
        for nt in ("tx", "bd"):
            b[nt]["pos"] = nodes[nt]["pos"].to(pos_dtype)
        for et in (TT, TB, PRED):
            b[et]["edge_index"] = edges[et].to(e_dtype)
        b[TT]["weight"] = torch.arange(edges[TT].size(1), dtype=torch.float32)
        bc = b.cuda()
        # a tree over transcripts only: bd nodes outside the root / in empty quadrants take the other index paths
        qt = tiles.QuadTreeTiling(bc["tx"]["pos"], max_tile_size=2500)
        ds = tiles.TilePredictSet(bc, qt, margin=margin)
        assert ds._index is not None and len(ds) == len(qt) > 8
        n64 = {nt: {k: (v.to(pos_dtype) if k == "pos" else v) for k, v in st.items()} for nt, st in nodes.items()}
        for i in (0, len(ds) // 2, len(ds) - 1):
            n_ref, e_ref, _ = tiles_ref.subset_ref(n64, edges, ds.tiles[i], margin)
            t = ds[i]
            for nt in ("tx", "bd"):
                for k, v in n_ref[nt].items():
                    assert torch.equal(t[nt][k].cpu(), v), (i, nt, k)
            for et in (TT, TB, PRED):
                assert torch.equal(t[et]["edge_index"].cpu().long(), e_ref[et]), (i, et)
        assert all(int((m != -1).sum()) == 0 for m in ds._index["maps"].values())
        ids = [3, 0, len(ds) - 1, 5, 1, 7]
        want = tiles.collate_tiles([ds[t] for t in ids])
        got, info = ds.cut(ids)
        assert got.num_graphs == 6
        for nt in ("tx", "bd"):
            assert set(got[nt]) == set(want[nt])
            for k in want[nt]:
                assert got[nt][k].dtype == want[nt][k].dtype and torch.equal(got[nt][k], want[nt][k]), (nt, k)
            assert info["nodes"][nt] == [int(ds[t][nt]["pos"].size(0)) for t in ids]
        for et in (TT, TB, PRED):
            assert got[et]["edge_index"].dtype == e_dtype
            assert torch.equal(got[et]["edge_index"], want[et]["edge_index"]), et
            assert info["edges"][et] == [int(ds[t][et]["edge_index"].size(1)) for t in ids]
        assert torch.equal(got[TT]["weight"], want[TT]["weight"])
    # small leaves, every tile in one group: the candidate ranges are merged to fit one launch, the result stays the collate
    ds = tiles.TilePredictSet(bc, tiles.QuadTreeTiling(bc["tx"]["pos"], max_tile_size=200), margin=margin)
    all_ids = list(range(len(ds)))
    assert sum(len(sp) for sp in ds._index["spans"]) > 1024
    got, _ = ds.cut(all_ids)
    want = tiles.collate_tiles([ds[t] for t in all_ids])
    for nt in ("tx", "bd"):
        for k in want[nt]:
            assert torch.equal(got[nt][k], want[nt][k]), (nt, k)
    for et in (TT, TB, PRED):
        assert torch.equal(got[et]["edge_index"], want[et]["edge_index"]), et


def test_quadtree_tiled_prediction_with_halo_equals_whole_graph_prediction():
    """Quadtree tiles + 20 um halo, de-duplicated: every transcript gets exactly one row and the assignments of one pass
    over the whole graph."""
    ts, nodes, edges, b = _graph(n_tx=30000, n_cells=300, seed=5)
    torch.manual_seed(0)
    lit = LitISTEncoder(ts.n_genes, in_channels=32, n_mid_layers=0).cuda().eval()
    lit.model.use_positional_embeddings = False
    b["tx"]["predict_mask"] = torch.ones(30000, dtype=torch.bool)
    for nt in ("tx", "bd"):
        b[nt]["batch"] = torch.zeros(nodes[nt]["pos"].size(0), dtype=torch.long)
    full = b.cuda()
    with torch.no_grad():
        src, seg, sim, gene = lit.predict_step(full, 0)
    whole = {int(i): (int(s), float(v)) for i, s, v in zip(src, seg, sim)}
    qt = tiles.QuadTreeTiling({"tx": full["tx"]["pos"], "bd": full["bd"]["pos"]}, max_tile_size=4000)
    ds = tiles.TilePredictSet(full, qt, margin=20.0)
    group, info = ds.cut(list(range(len(ds))))
    with torch.no_grad():
        s_i, g_i, v_i, _ = lit.predict_step(group, 0)
    seen = {}
    for a, c, v in zip(s_i.tolist(), g_i.tolist(), v_i.tolist()):
        if a not in seen or v > seen[a][1]:
            seen[a] = (c, v)
    assert set(seen) == set(whole)
    agree = np.mean([seen[k][0] == whole[k][0] for k in whole])
    assert agree >= 0.9999, agree
    assert max(abs(seen[k][1] - whole[k][1]) for k in whole) < 1e-5


def test_training_batch_from_quadtree_tiles_runs_get_losses():
    ts, nodes, edges, b, bc, qt = _tiling_and_graph(9000, 90, 7, 1200)
    labels, masks = qt.fit_labels_and_masks(bc, 5.0)
    g = torch.Generator().manual_seed(4)
    bc["tx"]["mask"], bc["bd"]["mask"] = masks["tx"], masks["bd"]
    bc["tx"]["cluster"] = torch.randint(0, 8, (9000,), generator=g).cuda()
    bc["bd"]["cluster"] = torch.randint(-1, 4, (90,), generator=g).cuda()
    part = tiles.TilePartition(bc, labels, len(qt))
    torch.manual_seed(0)
    lit = LitISTEncoder(ts.n_genes, in_channels=32, hidden_channels=32, out_channels=32, n_mid_layers=0).cuda().train()
    sim = torch.rand(8, 8, generator=g)
    sim_bd = torch.rand(4, 4, generator=g)
    lit.setup_losses((sim + sim.t()) / 2, (sim_bd + sim_bd.t()) / 2)
    batch = part.collate(part.batches(max_num=max(part.weights("edge")) * 3)[0])
    assert batch["tx"]["mask"].dtype == torch.bool and bool(batch["tx"]["mask"].any())
    loss = lit.training_step(batch, 0)
    loss.backward()
    assert bool(torch.isfinite(loss))
    assert all(p.grad is not None and bool(torch.isfinite(p.grad).all()) for n, p in lit.model.named_parameters() if "contains" not in n)
