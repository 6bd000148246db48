"""Buffered outlines on the GPU: sgb_polygon_props and the buffered point-in-polygon join against the plain join.

    python scripts/bench_buffered_pip.py [--out profiles/bench_buffered_pip_b200.json] [--max-tx 20000000] [--ratio 0.05]

Workloads: BASELINE configs[1] (1 M synthetic transcripts, 10 k cells) and configs[2] (20 M, 200 k), raw outlines = one
16-gon of radius 6.5 um per synthetic cell (segger_b200.synth), buffer_ratio 0.05 (grows a 6.5 um outline by about
0.33 um, the 5 % the plain-join benchmarks pre-grow their rings by).  Per workload, timed alternately in one run:

* ``props``: ``sgb_polygon_props`` over every ring (area, centroid, box, buffer distance);
* ``buffered``: ``points_in_polygons(tx, Outlines.buffered(ratio))`` (count + fill + sort, device output);
* ``plain``: ``points_in_polygons(tx, PackedPolygons(raw rings))`` on the same rings, unbuffered.

CUDA events, best of --reps after one warm-up; every call includes its one device->host read of the pair count.  Also
reported: the pair counts and the fraction of buffered pairs whose point lies outside the raw ring and within
0.01 |d| of the exact buffered rim -- an upper bound on the pairs where geopandas' buffer (16 chords per quarter
circle, ring simplified by about 1 % of d) could decide differently.  The GPU name and power limit are read in the
same run."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from segger_b200 import _lib  # noqa: E402
from segger_b200._lib import check, ptr, stream_ptr  # noqa: E402
from segger_b200.geometry import Outlines, PackedPolygons, points_in_polygons  # noqa: E402
from segger_b200.synth import synth  # noqa: E402

NV = 16


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


def near_rim_pairs(buf_pairs, plain_pairs, pts, verts, dist, n_poly):
    """Buffered pairs whose point is outside the raw ring and within 0.01 |d| of the grown rim (distance to the ring
    > 0.99 d), counted on the device in fp64 (rings are 16-gons here)."""
    key = lambda e: e[0].long() * n_poly + e[1].long()
    outside = ~torch.isin(key(buf_pairs), key(plain_pairs))
    n = 0
    for s in range(0, buf_pairs.size(1), 1 << 22):
        e = buf_pairs[:, s:s + (1 << 22)][:, outside[s:s + (1 << 22)]]
        p, g = e[0].long(), e[1].long()
        a = verts[g]                                                     # [e, 16, 2]
        b = torch.roll(a, -1, dims=1)
        ab, ap = b - a, pts[p][:, None, :] - a
        t = ((ap * ab).sum(-1) / (ab * ab).sum(-1)).clamp(0.0, 1.0)
        q = ap - t[..., None] * ab
        dmin = q.pow(2).sum(-1).min(1).values.sqrt()
        n += int((dmin > 0.99 * dist[g]).sum())
    return n, int(outside.sum())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_buffered_pip_b200.json"))
    ap.add_argument("--max-tx", type=int, default=20_000_000)
    ap.add_argument("--ratio", type=float, default=0.05)
    ap.add_argument("--reps", type=int, default=10)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_buffered_pip.py measures on a GPU; none found")
    dev = torch.device("cuda")
    lib = _lib.load()
    result = {"gpu": gpu_info(), "ratio": a.ratio, "ring_vertices": NV, "rows": []}
    ang = np.linspace(0, 2 * np.pi, NV, endpoint=False)
    for n_tx, n_cells in ((1_000_000, 10_000), (20_000_000, 200_000)):
        if n_tx > a.max_tx:
            continue
        ts = synth(n_tx, n_cells, seed=0, pred_edges=False)
        pos = torch.from_numpy(ts.tx_pos).to(dev)
        c = ts.bd_pos.astype(np.float64)
        verts = np.stack([c[:, None, 0] + 6.5 * np.cos(ang)[None], c[:, None, 1] + 6.5 * np.sin(ang)[None]], -1).reshape(-1, 2)
        off = np.arange(n_cells + 1, dtype=np.int64) * NV
        outl, plain = Outlines(verts, off), PackedPolygons(verts, off)
        buf = outl.buffered(a.ratio, dev)
        d_verts, d_off = outl.on(dev)
        area = torch.empty(n_cells, dtype=torch.float64, device=dev)
        cen = torch.empty(n_cells, 2, dtype=torch.float64, device=dev)
        box = torch.empty(n_cells, 4, dtype=torch.float64, device=dev)
        dist = torch.empty(n_cells, dtype=torch.float64, device=dev)

        def props():
            check(lib.sgb_polygon_props(ptr(d_verts), ptr(d_off), n_cells, a.ratio, ptr(area), ptr(cen), ptr(box), ptr(dist),
                                        stream_ptr(dev)), "polygon_props")
        out = {}

        def run_buf():
            out["buf"] = points_in_polygons(pos, buf, device=dev, device_output=True)

        def run_plain():
            out["plain"] = points_in_polygons(pos, plain, device=dev, device_output=True)
        runs = {"props": [], "buffered": [], "plain": []}
        for _ in range(2):                                   # alternated: the spread of each pair
            runs["props"].append(best_ms(props, a.reps))
            runs["buffered"].append(best_ms(run_buf, a.reps))
            runs["plain"].append(best_ms(run_plain, a.reps))
        near, outside = near_rim_pairs(out["buf"], out["plain"], pos.double(),
                                       torch.from_numpy(verts).to(dev).view(n_cells, NV, 2), buf.dist, n_cells)
        E = out["buf"].size(1)
        row = dict(n_tx=n_tx, n_outlines=n_cells, props_ms=min(runs["props"]), buffered_ms=min(runs["buffered"]),
                   plain_ms=min(runs["plain"]), ms_runs=runs, buffered_over_plain=min(runs["buffered"]) / min(runs["plain"]),
                   pairs_buffered=E, pairs_plain=int(out["plain"].size(1)), pairs_outside_raw_ring=outside,
                   pairs_within_1pct_of_rim=near, fraction_within_1pct_of_rim=near / max(E, 1),
                   mean_dist_um=float(buf.dist.mean()))
        print(json.dumps(row), flush=True)
        result["rows"].append(row)
        del pos, out, buf, outl
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(result, f, indent=1)
    print(f"wrote {a.out}")


if __name__ == "__main__":
    main()
