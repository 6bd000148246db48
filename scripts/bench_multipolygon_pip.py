"""Outlines with holes and several parts on the GPU: the multi-ring join (sgb_pip_multi_count / _fill) and
sgb_polygon_props_multi, against the one-ring entry points on the same cells.

    python scripts/bench_multipolygon_pip.py [--out profiles/bench_multipolygon_pip_b200.json] [--max-tx 20000000]

Workloads: BASELINE configs[1] (1 M synthetic transcripts, 10 k cells) and configs[2] (20 M, 200 k); per synthetic
cell (segger_b200.synth) a 16-gon cell outline of radius 6.5 um and a 12-gon nucleus of radius 3 um.  Cases, each plain
(already buffered) and buffered on the device at buffer_ratio 0.05:

* ``single_new`` / ``single_old``: the 16-gons as one-ring geometries, through the new entry points (part_off =
  geom_off = 0..M) and through the existing ones (sgb_pip_count / sgb_pip_buffered_count), alternated in one run;
* ``annulus``: the cell ring with the nucleus ring as its hole (the cytoplasm);
* ``two_part``: the cell ring plus a second part, a 12-gon of radius 3 um 10 um away.

CUDA events, best of --reps after one warm-up; every call includes its one device->host read of the pair count; the
buffered cases include nothing of the distance computation (``Outlines.buffered`` is built once per dataset).  Also
timed: ``sgb_polygon_props_multi`` over the annuli.  The GPU name and power limit are read in the same run."""
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


def ngons(c, r, n):
    ang = np.linspace(0, 2 * np.pi, n, endpoint=False)
    return np.stack([c[:, None, 0] + r * np.cos(ang)[None], c[:, None, 1] + r * np.sin(ang)[None]], -1)   # [M, n, 2]


def layouts(c):
    """-> {case: (verts, ring_off, part_off, geom_off)}; part_off / geom_off None = the one-ring layout."""
    M = c.shape[0]
    cell, nuc = ngons(c, 6.5, 16), ngons(c + 0.5, 3.0, 12)
    far = ngons(c + np.array([10.0, 0.0]), 3.0, 12)
    one = np.arange(M + 1, dtype=np.int64)
    two_rings = np.concatenate([cell.reshape(M, -1), nuc.reshape(M, -1)], 1).reshape(-1, 2)
    two_parts = np.concatenate([cell.reshape(M, -1), far.reshape(M, -1)], 1).reshape(-1, 2)
    pair_off = np.zeros(2 * M + 1, dtype=np.int64)
    pair_off[1::2] = np.arange(M) * 28 + 16
    pair_off[2::2] = np.arange(1, M + 1) * 28
    return {
        "single_old": (cell.reshape(-1, 2), one * 16, None, None),
        "single_new": (cell.reshape(-1, 2), one * 16, one, one),
        "annulus": (two_rings, pair_off, one * 2, one),                        # one part of two rings
        "two_part": (two_parts, pair_off, np.arange(2 * M + 1, dtype=np.int64), one * 2),   # two parts of one ring
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_multipolygon_pip_b200.json"))
    ap.add_argument("--max-tx", type=int, default=20_000_000)
    ap.add_argument("--ratio", type=float, default=0.05)
    ap.add_argument("--reps", type=int, default=10)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_multipolygon_pip.py measures on a GPU; none found")
    dev = torch.device("cuda")
    lib = _lib.load()
    result = {"gpu": gpu_info(), "ratio": a.ratio, "cell_vertices": 16, "nucleus_vertices": 12, "rows": []}
    for n_tx, n_cells in ((1_000_000, 10_000), (20_000_000, 200_000)):
        if n_tx > a.max_tx:
            continue
        ts = synth(n_tx, n_cells, seed=0, pred_edges=False)
        pos = torch.from_numpy(ts.tx_pos).to(dev)
        polys = {}
        for case, (verts, ring_off, part_off, geom_off) in layouts(ts.bd_pos.astype(np.float64)).items():
            polys[case, "plain"] = PackedPolygons(verts, ring_off, part_off, geom_off)
            polys[case, "buffered"] = Outlines(verts, ring_off, None, part_off, geom_off).buffered(a.ratio, dev)
        ann = polys["annulus", "buffered"].outlines
        d_ann = ann.on(dev)
        outs = {k: torch.empty(n_cells, w, dtype=torch.float64, device=dev).squeeze(1) for k, w in
                (("area", 1), ("cen", 2), ("box", 4), ("dist", 1))}

        def props():
            check(lib.sgb_polygon_props_multi(*map(ptr, d_ann), n_cells, a.ratio, ptr(outs["area"]), ptr(outs["cen"]),
                                              ptr(outs["box"]), ptr(outs["dist"]), stream_ptr(dev)), "polygon_props_multi")
        pairs = {}

        def runner(key):
            def run():
                pairs[key] = int(points_in_polygons(pos, polys[key], device=dev, device_output=True).size(1))
            return run
        order = [(c, m) for m in ("plain", "buffered") for c in ("single_new", "single_old", "annulus", "two_part")]
        runs = {f"{c}_{m}": [] for c, m in order}
        runs["props_multi"] = []
        for _ in range(3):                                   # alternated: the spread of each case
            for c, m in order:
                runs[f"{c}_{m}"].append(best_ms(runner((c, m)), a.reps))
            runs["props_multi"].append(best_ms(props, a.reps))
        row = dict(n_tx=n_tx, n_outlines=n_cells, ms={k: min(v) for k, v in runs.items()}, ms_runs=runs,
                   pairs={f"{c}_{m}": pairs[c, m] for c, m in order})
        for m in ("plain", "buffered"):
            row[f"single_new_over_old_{m}"] = row["ms"][f"single_new_{m}"] / row["ms"][f"single_old_{m}"]
            assert pairs["single_new", m] == pairs["single_old", m]
        print(json.dumps(row), flush=True)
        result["rows"].append(row)
        del pos, polys, pairs
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(result, f, indent=1)
    print(f"wrote {a.out}")


if __name__ == "__main__":
    main()
