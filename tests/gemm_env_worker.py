"""Worker of tests/test_gpu_gemm_matrix.py::test_gemm_env_switch: runs the reduced GEMM matrix (one case per family,
tests/gemm_matrix.py REDUCED) under the SEGGER_B200_GEMM* / SEGGER_B200_TF32_TERMS switches of its environment, with the
same error bounds and the kernel each switch selects checked under torch.profiler.  Prints one JSON line and exits 0
when every case passes."""
import json
import os
import sys
from dataclasses import replace

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from tests.gemm_matrix import REDUCED, Env, case, missing_kernels, profile_case  # noqa: E402


def main():
    e = os.environ
    env = Env(simt=e.get("SEGGER_B200_GEMM", "").lower().startswith("s"), ts=not e.get("SEGGER_B200_GEMM_TS", "").startswith("0"),
              wm_general=e.get("SEGGER_B200_GEMM_WM") == "0",
              pp=int(e["SEGGER_B200_GEMM_PP"]) if e.get("SEGGER_B200_GEMM_PP") in ("0", "1") else None)
    terms4 = e.get("SEGGER_B200_TF32_TERMS") == "4"
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    results, failures = {}, []
    for name in REDUCED:
        c = case(name)
        if terms4 and c.op in ("fwd", "gather"):
            c = replace(c, exact=max(c.exact, 1))          # the fourth product term is used by exact=1 calls only
        chk, first, second, names = profile_case(c)
        results[name] = chk.ratio
        failures += [f"{name}: {f}" for f in chk.failures]
        failures += [f"{name}: {k}: two identical calls differ" for k in first if not torch.equal(first[k], second[k])]
        miss = missing_kernels(c, names, sm, env)
        if miss:
            failures.append(f"{name}: expected {miss}, launched {names}")
    for f in failures:
        print(f, file=sys.stderr)
    vars_ = {k: v for k, v in e.items() if k.startswith("SEGGER_B200_")}
    print(json.dumps({"env": vars_, "ok": not failures, "cases": results}), flush=True)
    sys.exit(1 if failures else 0)


if __name__ == "__main__":
    main()
