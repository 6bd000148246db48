"""Quadtree tiling (sgb_quadtree.cu) and the grouped prediction-tile cut on quadtree tiles.

    python scripts/bench_tiling.py [--out profiles/bench_tiling_b200.json] [--max-n 100000000] [--cut-tx 20000000]

* build: ``QuadTreeTiling(points, 50_000)`` at 1, 20 and 100 M points, uniform and clustered (0.5 points / um^2, clusters
  of 100 with sigma 3 um, as scripts/bench_knn.py), fp32; ms per build incl. its one device->host read.
* cut: BASELINE configs[2] (20 M synthetic transcripts, kNN k=5 r=5 um, point-in-polygon tx-neighbors-bd, 20 um halo), one
  pass of ``TilePredictSet.cut`` over every tile in groups of 32, on (a) the leaves of a ``QuadTreeTiling`` over all node
  positions, (b) ``square_tiles`` + ``grid`` (bench.py's inference leg), (c) the same squares through the per-tile
  ``subset()`` fallback (what quadtree tiles cost before the leaf index).  Candidates = nodes scanned by the cut kernels.

CUDA events, best of --reps after one warm-up pass; the GPU name and power limit are read in the same run."""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from segger_b200 import tiles  # noqa: E402
from tests.util import PRED, TB, TT  # noqa: E402


def points(kind, n, rng):
    side = (n / 0.5) ** 0.5
    if kind == "uniform":
        return rng.uniform(0, side, (n, 2)).astype(np.float32)
    n_c = max(1, n // 100)
    c = rng.uniform(0, side, (n_c, 2))
    return (c[rng.integers(0, n_c, n)] + rng.normal(0, 3.0, (n, 2))).astype(np.float32)


def best_ms(fn, reps):
    fn()
    best = 1e30
    for _ in range(reps):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return best


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip()}


def cfg2_graph(n_tx, device):
    """bench.py inference_cfg3_leg's graph: synthetic transcripts, kNN, point-in-polygon candidates."""
    from segger_b200.geometry import PackedPolygons, points_in_polygons
    from segger_b200.hetero import HeteroBatch
    from segger_b200.neighbors import kdtree_neighbors
    from segger_b200.synth import synth
    n_cells = n_tx // 100
    ts = synth(n_tx, n_cells, seed=0, pred_edges=False)
    pos = torch.from_numpy(ts.tx_pos).to(device)
    ei, _ = kdtree_neighbors(pos, 5, 5.0, device_output=True, device=device)
    ang = np.linspace(0, 2 * np.pi, 16, endpoint=False)
    c = ts.bd_pos.astype(np.float64)
    verts = np.stack([c[:, None, 0] + 6.5 * 1.05 * np.cos(ang)[None], c[:, None, 1] + 6.5 * 1.05 * np.sin(ang)[None]], -1).reshape(-1, 2)
    off = np.arange(n_cells + 1, dtype=np.int64) * 16
    ep = points_in_polygons(pos, PackedPolygons(verts, off), device=device, device_output=True)
    b = HeteroBatch()
    b["tx"]["x"], b["tx"]["pos"] = torch.from_numpy(ts.tx_gene).to(device), pos
    b["tx"]["index"] = torch.from_numpy(ts.tx_index).to(device)
    b["bd"]["x"], b["bd"]["pos"] = torch.from_numpy(ts.bd_x).to(device), torch.from_numpy(ts.bd_pos).to(device)
    b["bd"]["index"] = torch.from_numpy(ts.bd_index).to(device)
    b[TT]["edge_index"], b[TB]["edge_index"], b[PRED]["edge_index"] = ei, torch.from_numpy(ts.edge_tb).to(device), ep
    return ts, b


def cut_pass(ds, G):
    kept = [0]

    def run():
        n = 0
        for g0 in range(0, len(ds), G):
            group, _ = ds.cut(list(range(g0, min(len(ds), g0 + G))))
            n += group["tx"]["pos"].size(0)
        kept[0] = n
    return run, kept


def candidates(ds, G):
    ix = ds._index
    dev = ds.data["tx"]["pos"].device
    return sum(ds._slot_ranges(ix["node_ptr"]["tx"], list(range(g0, min(len(ds), g0 + G))), dev)[4] for g0 in range(0, len(ds), G))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_tiling_b200.json"))
    ap.add_argument("--max-n", type=int, default=100_000_000)
    ap.add_argument("--cut-tx", type=int, default=20_000_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--group", type=int, default=32)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_tiling.py measures on a GPU; none found")
    dev = torch.device("cuda")
    result = {"gpu": gpu_info(), "build": [], "cut": None}
    rng = np.random.default_rng(0)
    for kind in ("uniform", "clustered"):
        for n in (1_000_000, 20_000_000, 100_000_000):
            if n > a.max_n:
                continue
            pts = torch.from_numpy(points(kind, n, rng)).to(dev)
            box = {}

            def build():
                box["qt"] = tiles.QuadTreeTiling(pts, max_tile_size=50_000)
            ms = best_ms(build, a.reps)
            qt = box.pop("qt")
            row = dict(kind=kind, n=n, max_tile_size=50_000, ms=ms, points_per_s=n / ms * 1e3, tiles=len(qt),
                       max_level=int(qt.levels.max()), max_count=int(qt.counts.max()))
            print(json.dumps(row), flush=True)
            result["build"].append(row)
            del qt, pts
            torch.cuda.empty_cache()

    if a.cut_tx > 0:
        t0 = time.perf_counter()
        ts, b = cfg2_graph(a.cut_tx, dev)
        t_graph = time.perf_counter() - t0
        G = a.group
        qt = tiles.QuadTreeTiling({"tx": b["tx"]["pos"], "bd": b["bd"]["pos"]}, max_tile_size=50_000)
        t0 = time.perf_counter()
        ds_q = tiles.TilePredictSet(b, qt, margin=20.0)
        torch.cuda.synchronize()
        t_index_q = time.perf_counter() - t0
        nt = max(1, int(math.ceil(math.sqrt(a.cut_tx / 50_000))))
        lo, hi = ts.tx_pos.min(0) - 1e-3, ts.tx_pos.max(0) + 1e-3
        boxes = tiles.square_tiles(float(lo[0]), float(lo[1]), float(hi[0]), float(hi[1]), nt, nt)
        t0 = time.perf_counter()
        ds_s = tiles.TilePredictSet(b, boxes, margin=20.0, grid=(nt, nt))
        torch.cuda.synchronize()
        t_index_s = time.perf_counter() - t0
        ds_f = tiles.TilePredictSet(b, boxes, margin=20.0)
        run_q, kept_q = cut_pass(ds_q, G)
        run_s, kept_s = cut_pass(ds_s, G)
        ms_q, ms_s = best_ms(run_q, a.reps), best_ms(run_s, a.reps)
        ms_q2, ms_s2 = best_ms(run_q, a.reps), best_ms(run_s, a.reps)      # alternated: the spread of the pair

        def run_f():
            for t in range(len(ds_f)):
                ds_f[t]
        ms_f = best_ms(run_f, max(1, a.reps - 1))
        result["cut"] = {
            "n_tx": a.cut_tx, "n_cells": a.cut_tx // 100, "halo_um": 20.0, "group": G, "host_graph_s": t_graph,
            "quadtree": {"tiles": len(ds_q), "ms": min(ms_q, ms_q2), "ms_runs": [ms_q, ms_q2], "index_build_s": t_index_q,
                         "rows": kept_q[0], "tx_candidates": candidates(ds_q, G),
                         "candidate_ranges": sum(len(s) for s in ds_q._index["spans"])},
            "square_grid": {"tiles": len(ds_s), "ms": min(ms_s, ms_s2), "ms_runs": [ms_s, ms_s2], "index_build_s": t_index_s,
                            "rows": kept_s[0], "tx_candidates": candidates(ds_s, G)},
            "square_subset_fallback": {"tiles": len(ds_f), "ms": ms_f},
        }
        print(json.dumps(result["cut"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(result, f, indent=1)
    print(f"wrote {a.out}")


if __name__ == "__main__":
    main()
