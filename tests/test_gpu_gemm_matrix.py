"""Every kernel instantiation the projection-GEMM dispatcher can pick, against float64 with a per-element error bound
(tests/gemm_matrix.py), with the kernel that ran checked under torch.profiler.  Prints one JSON line per case with the
worst err / magnitude of each output; GEMM_MATRIX_JSON=<path> also writes them to a file."""
import json
import os
import subprocess
import sys

import pytest
import torch

from tests.gemm_matrix import CASES, DEFAULT_ENV, expected_kernel, missing_kernels, profile_case, result_line

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_RESULTS = {}


def _sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.mark.parametrize("c", CASES, ids=str)
def test_gemm_matrix(c):
    chk, first, second, names = profile_case(c)
    line = result_line(c, chk)
    print(line)
    _RESULTS[c.name] = json.loads(line)
    out = os.environ.get("GEMM_MATRIX_JSON")
    if out:
        with open(out, "w") as f:
            json.dump({"device": torch.cuda.get_device_name(0), "cases": _RESULTS}, f, indent=1)
    assert not chk.failures, chk.failures
    for k in first:
        assert torch.equal(first[k], second[k]), f"{k}: two identical calls differ"
    miss = missing_kernels(c, names, _sm_count(), DEFAULT_ENV)
    assert not miss, (f"expected {expected_kernel(c, _sm_count())}", "launched", names)


ENVS = {"ts0": {"SEGGER_B200_GEMM_TS": "0"}, "wm0": {"SEGGER_B200_GEMM_WM": "0"}, "pp0": {"SEGGER_B200_GEMM_PP": "0"},
        "pp1": {"SEGGER_B200_GEMM_PP": "1"}, "terms4": {"SEGGER_B200_TF32_TERMS": "4"}, "simt": {"SEGGER_B200_GEMM": "simt"}}


@pytest.mark.parametrize("name", list(ENVS))
def test_gemm_env_switch(name):
    """The documented A/B switches are read once per process: each runs the reduced matrix in a fresh interpreter."""
    env = {k: v for k, v in os.environ.items() if not k.startswith("SEGGER_B200_")}
    env.update(ENVS[name])
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "gemm_env_worker.py")], env=env, cwd=ROOT,
                       capture_output=True, text=True, timeout=900)
    print(r.stdout[-4000:], r.stderr[-4000:])
    assert r.returncode == 0
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    res = json.loads(lines[-1])
    assert res["ok"] and res["env"] == ENVS[name] and res["cases"]
