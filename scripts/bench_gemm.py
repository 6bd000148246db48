"""Times and checks the projection GEMMs of the bench workload (cfg2 shapes) on the selected back end.

    SEGGER_B200_TC_KC=4 SEGGER_B200_TC_KC_EXACT=1 python scripts/bench_gemm.py [--rows 1000000]

For every (op, M, N, K): ms per launch (CUDA events, 256 MB L2 flush between launches), effective fp32
TFLOP/s (2MNK / t), achieved GB/s on the compulsory operand traffic, and the error against float64 on a
65k-row sample: max |err| / max |ref| and the mean SIGNED relative error (the round-toward-zero bias).
`gather` is the gene-table forward of ISTEncoder's first projection (y = x w^T + b + table[ids], WM = 1 epilogue).
SEGGER_B200_LIB=<path> times another build of libsegger_b200.so (A/B of two builds: run once per build, alternating)."""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from segger_b200 import ops  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--only", default="", help="comma list of ops to run (fwd, gather, dgrad, wgrad); default all")
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    R = a.rows
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    g = torch.Generator(device="cuda").manual_seed(0)

    def time_it(fn):
        fn(); torch.cuda.synchronize()
        tot = 0.0
        for _ in range(a.reps):
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record()
            torch.cuda.synchronize()
            tot += e0.elapsed_time(e1)
        return tot / a.reps * 1e-3

    rows = []
    shapes = [("gather", R, 384, 128), ("fwd", R, 384, 256), ("fwd", R, 384, 128), ("fwd", 2 * R, 64, 256), ("fwd", 2 * R, 64, 64), ("fwd", R, 64, 128),
              ("dgrad", R, 384, 256), ("dgrad", R, 384, 128), ("dgrad", R, 64, 128), ("dgrad", 2 * R, 64, 64),
              ("wgrad", R, 384, 256), ("wgrad", R, 384, 128), ("wgrad", 2 * R, 64, 256), ("wgrad", R, 64, 128),
              ("wgrad", 2 * R, 64, 64), ("wgrad", R, 256, 128)]
    if a.only:
        shapes = [sh for sh in shapes if sh[0] in a.only.split(",")]
    for op, M, N, K in shapes:
        S = min(M, 65536)
        if op == "fwd":
            # post-GELU-like inputs (mostly positive) are the hard case for a truncating accumulator
            x = torch.nn.functional.gelu(torch.randn(M, K, device=dev, generator=g))
            w = torch.randn(N, K, device=dev, generator=g) / K ** 0.5
            for exact in ((0, 1) if a.only else (0, 1, 2)):
                t = time_it(lambda: ops.linear_fwd(x, w, None, exact=exact))
                y, _ = ops.linear_fwd(x[:S], w, None, exact=exact)
                ref = x[:S].double() @ w.double().t()
                err = float((y.double() - ref).abs().max() / ref.abs().max())
                m = ref.abs() > 0.1 * ref.abs().max()
                bias = float((((y.double() - ref) / ref)[m] * torch.sign(ref[m])).mean())
                rows.append(dict(op=f"fwd exact={exact}", M=M, N=N, K=K, ms=t * 1e3, tflops=2 * M * N * K / t / 1e12,
                                 gbs=4 * (M * K + M * N) / t / 1e9, err=err, signed_bias=bias))
        elif op == "gather":
            n_genes = 500
            x = torch.nn.functional.gelu(torch.randn(M, K, device=dev, generator=g))
            w = torch.randn(N, K, device=dev, generator=g) / K ** 0.5
            b = torch.randn(N, device=dev, generator=g)
            table = torch.randn(n_genes, N, device=dev, generator=g)
            ids = torch.randint(0, n_genes, (M,), device=dev, generator=g)
            t = time_it(lambda: ops.linear_fwd(x, w, b, exact=0, gather=(ids, table)))
            y, _ = ops.linear_fwd(x[:S], w, b, exact=0, gather=(ids[:S], table))
            ref = x[:S].double() @ w.double().t() + b.double() + table.double()[ids[:S]]
            rows.append(dict(op="gather", M=M, N=N, K=K, ms=t * 1e3, tflops=2 * M * N * K / t / 1e12,
                             gbs=4 * (M * K + M * N) / t / 1e9, err=float((y.double() - ref).abs().max() / ref.abs().max())))
        elif op == "dgrad":
            dy = torch.randn(M, N, device=dev, generator=g)
            w = torch.randn(N, K, device=dev, generator=g) / K ** 0.5
            t = time_it(lambda: ops.linear_dgrad(dy, w))
            dx = ops.linear_dgrad(dy[:S], w)
            ref = dy[:S].double() @ w.double()
            rows.append(dict(op="dgrad", M=M, N=N, K=K, ms=t * 1e3, tflops=2 * M * N * K / t / 1e12,
                             gbs=4 * (M * K + M * N) / t / 1e9, err=float((dx.double() - ref).abs().max() / ref.abs().max())))
        else:
            dy = torch.randn(M, N, device=dev, generator=g)
            x = torch.nn.functional.gelu(torch.randn(M, K, device=dev, generator=g))
            t = time_it(lambda: ops.linear_wgrad(dy, x))
            dw, _ = ops.linear_wgrad(dy, x)
            ref = torch.zeros(N, K, dtype=torch.float64, device=dev)
            for i in range(0, M, 1 << 18):
                ref += dy[i:i + (1 << 18)].double().t() @ x[i:i + (1 << 18)].double()
            rows.append(dict(op="wgrad(+colsum)", M=M, N=N, K=K, ms=t * 1e3, tflops=2 * M * N * K / t / 1e12,
                             gbs=4 * (M * K + M * N) / t / 1e9, err=float((dw.double() - ref).abs().max() / ref.abs().max())))
        del_list = [v for v in ("x", "w", "dy") if v in locals()]
    print(f"KC={os.environ.get('SEGGER_B200_TC_KC', '4')} KC_EXACT={os.environ.get('SEGGER_B200_TC_KC_EXACT', '1')} "
          f"TERMS={os.environ.get('SEGGER_B200_TF32_TERMS', 'default')}")
    for r in rows:
        print(f"{r['op']:15s} M={r['M']:8d} N={r['N']:4d} K={r['K']:4d}  {r['ms']:8.3f} ms  {r['tflops']:7.1f} TF/s  {r['gbs']:7.0f} GB/s  "
              f"err {r['err']:.2e}" + (f"  signed bias {r['signed_bias']:+.2e}" if "signed_bias" in r else ""))
    print(json.dumps(rows))


if __name__ == "__main__":
    main()
