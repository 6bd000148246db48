"""The ring-search kNN (sgb_knn2d_ring: any k <= 1024, any radius up to inf) on Xenium-like density (0.5 points / um^2),
uniform and clustered (~100 points per cluster, sigma 3 um), as scripts/bench_knn.py draws them.

    python scripts/bench_knn_ring.py [--out profiles/bench_knn_ring_b200.json] [--max-n 20000000]

Cases, each CUDA events, best of 3 after one warm-up:

* ``large_k``: k in {64, 256, 1024} at r = 5 um and r = inf over 1M and 20M points, the table only (plan + bin + search).
  The queries are the points themselves, or the first 2^31 / k of them where the [n, k] table would pass 16 GB.
* ``uniform_mode``: setup_prediction_graph(mode='uniform') -- the k nearest transcripts of every centroid, host arrays
  in, CPU edge list out -- for 10k and 200k uniform random centroids over 1M and 20M transcripts, k in {5, 64}.  Timed
  against the method it replaced in the same run: the radius-capped register kernel re-run with a doubling radius until
  every row is full, with a host copy of the points and a count read back per round (it holds k <= 32 only).
* ``small_k``: the ring search against sgb_knn2d at k in {5, 20}, r = 5 um, same inputs, tables compared.

The GPU name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from segger_b200.neighbors import _knn_table, _table_to_coo, knn_table, setup_prediction_graph  # noqa: E402


def points(kind, n, rng):
    side = (n / 0.5) ** 0.5
    if kind == "uniform":
        return rng.uniform(0, side, (n, 2)).astype(np.float32)
    c = rng.uniform(0, side, (max(1, n // 100), 2))
    return (c[rng.integers(0, c.shape[0], n)] + rng.normal(0, 3.0, (n, 2))).astype(np.float32)


def best_ms(fn, reps=3):
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


def best_wall_ms(fn, reps=3):
    """Host clock around host-in / host-out calls that end in a device synchronise."""
    fn()
    best = 1e30
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        best = min(best, (time.perf_counter() - t0) * 1e3)
    return best


def doubling_uniform_graph(points, query, max_k):
    """The uniform-mode search this change replaced: the radius-capped kernel, radius doubled until all rows are full."""
    pts = np.asarray(points, dtype=np.float64)
    n = pts.shape[0]
    k = min(max_k, n)
    span = np.maximum(pts.max(0) - pts.min(0), 1e-9)
    r = float(np.sqrt(4.0 * max(k, 1) * span[0] * span[1] / (np.pi * max(n, 1)))) + 1e-9
    diag = float(np.hypot(*(np.maximum(pts.max(0), query.max(0)) - np.minimum(pts.min(0), query.min(0))))) + 1.0
    rounds = 0
    while True:
        table, count = knn_table(points, max_k, r, query=query)
        rounds += 1
        if r > diag or int((count < k).sum()) == 0:
            break
        r *= 2.0
    with torch.no_grad():
        edge_index, _ = _table_to_coo(table, None, n)
    return edge_index.cpu(), rounds


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_knn_ring_b200.json"))
    ap.add_argument("--max-n", type=int, default=20_000_000)
    a = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    res = {"gpu": q, "density_per_um2": 0.5, "timing": "CUDA events (host clock for uniform_mode), best of 3 after one "
           "warm-up", "large_k": [], "uniform_mode": [], "small_k": []}
    print(json.dumps({"gpu": q}), flush=True)
    rng = np.random.default_rng(0)
    sizes = [n for n in (1_000_000, 20_000_000) if n <= a.max_n]
    for kind in ("uniform", "clustered"):
        for n in sizes:
            pts = points(kind, n, rng)
            dev = torch.from_numpy(pts).cuda()
            for k in (64, 256, 1024):
                nq = min(n, (1 << 31) // k)
                qry = None if nq == n else dev[:nq]
                for r in (5.0, float("inf")):
                    out = {}

                    def run():
                        out["t"] = knn_table(dev, k, r, query=qry)
                    ms = best_ms(run)
                    cnt = out["t"][1]
                    row = dict(kind=kind, n=n, n_query=nq, k=k, r=r, ms=ms, queries_per_s=nq / ms * 1e3,
                               mean_count=float(cnt.double().mean()), full_rows=float((cnt == k).double().mean()))
                    res["large_k"].append(row)
                    print(json.dumps(row), flush=True)
                    del out
            for k in (5, 20):
                t = {}
                ms_reg = best_ms(lambda: t.__setitem__("reg", _knn_table(dev, k, 5.0, None, None, False)))
                ms_ring = best_ms(lambda: t.__setitem__("ring", _knn_table(dev, k, 5.0, None, None, True)))
                same = bool(torch.equal(t["reg"][0], t["ring"][0]) and torch.equal(t["reg"][1], t["ring"][1]))
                row = dict(kind=kind, n=n, k=k, r=5.0, ms_register=ms_reg, ms_ring=ms_ring, ring_over_register=ms_ring / ms_reg,
                           identical=same)
                res["small_k"].append(row)
                print(json.dumps(row), flush=True)
                del t
            del dev
            for m in (10_000, 200_000):
                side = (n / 0.5) ** 0.5
                cen = rng.uniform(0, side, (m, 2))
                for k in (5, 64):
                    out = {}
                    ms_new = best_wall_ms(lambda: out.__setitem__("new", setup_prediction_graph(pts, cen, k, 0, mode="uniform")))
                    row = dict(kind=kind, n_transcripts=n, n_centroids=m, k=k, ms_ring=ms_new, edges=int(out["new"].size(1)))
                    if k <= 32:
                        ms_old = best_wall_ms(lambda: out.__setitem__("old", doubling_uniform_graph(pts, cen, k)))
                        row.update(ms_doubling=ms_old, doubling_rounds=out["old"][1], speedup=ms_old / ms_new,
                                   identical=bool(torch.equal(out["old"][0], out["new"])))
                    else:
                        row.update(ms_doubling=None, note="the doubling search holds k <= 32 only")
                    res["uniform_mode"].append(row)
                    print(json.dumps(row), flush=True)
                    del out
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
