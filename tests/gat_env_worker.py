"""Worker of tests/test_gpu_gat_matrix.py::test_gat_env_switch: runs the reduced GATv2 matrix (one case per family,
tests/gat_matrix.py REDUCED; LEGACY under SEGGER_B200_GAT=legacy) under the SEGGER_B200_GAT* switches of its environment,
with the same error bounds and the kernels each switch selects checked under torch.profiler.  Prints one JSON line and
exits 0 when every case passes."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from tests.gat_matrix import LEGACY, REDUCED, Env, case, dispatch_failures, profile_case  # noqa: E402


def main():
    env = Env.from_environ(os.environ)
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    results, failures = {}, []
    for name in (LEGACY if env.legacy else REDUCED):
        c = case(name)
        chk, names = profile_case(c, env=env)
        results[name] = chk.usage
        failures += [f"{name}: {f}" for f in chk.failures + dispatch_failures(c, names, sm, env)]
    for f in failures:
        print(f, file=sys.stderr)
    vars_ = {k: v for k, v in os.environ.items() if k.startswith("SEGGER_B200_")}
    print(json.dumps({"env": vars_, "ok": not failures, "cases": results}), flush=True)
    sys.exit(1 if failures else 0)


if __name__ == "__main__":
    main()
