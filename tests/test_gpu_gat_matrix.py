"""Every kernel instantiation the GATv2 attention dispatcher can pick, against float64 with per-element error bounds
(tests/gat_matrix.py), with the kernels that ran checked under torch.profiler.  Prints one JSON line per case with the
worst err / bound of each output; GAT_MATRIX_JSON=<path> also writes them, with the card and its power limit, to a file."""
import json
import os
import subprocess
import sys

import pytest
import torch

from tests.gat_matrix import CASES, DEFAULT_ENV, dispatch_failures, profile_case, result_line, run_raises

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_RESULTS = {}


def _sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip() or None
    except (OSError, subprocess.SubprocessError):
        return None


@pytest.mark.parametrize("c", [c for c in CASES if not c.raises], ids=str)
def test_gat_matrix(c):
    chk, names = profile_case(c)
    line = result_line(c, chk)
    print(line)
    _RESULTS[c.name] = json.loads(line)
    out = os.environ.get("GAT_MATRIX_JSON")
    if out:
        with open(out, "w") as f:
            json.dump({"device": torch.cuda.get_device_name(0), "power_limit": _power_limit(), "cases": _RESULTS}, f,
                      indent=1)
    assert not chk.failures, chk.failures
    miss = dispatch_failures(c, names, _sm_count(), DEFAULT_ENV)
    assert not miss, (miss, names)


@pytest.mark.parametrize("c", [c for c in CASES if c.raises], ids=str)
def test_gat_unsupported_shape_raises(c):
    assert run_raises(c)


ENVS = {"legacy": {"SEGGER_B200_GAT": "legacy"}, "rpw32": {"SEGGER_B200_GAT_RPW": "32"},
        "rpw1": {"SEGGER_B200_GAT_RPW": "1"}, "sort0": {"SEGGER_B200_GAT_SORT": "0"},
        "occ3": {"SEGGER_B200_GAT_DST_OCC": "3"}, "occ4": {"SEGGER_B200_GAT_DST_OCC": "4"},
        "logits0": {"SEGGER_B200_GAT_LOGITS": "0"}, "direct0": {"SEGGER_B200_GAT_DIRECT": "0"}}


@pytest.mark.parametrize("name", list(ENVS))
def test_gat_env_switch(name):
    """The documented A/B switches (RPW and DST_OCC are read once per process): each runs the reduced matrix in a fresh
    interpreter."""
    env = {k: v for k, v in os.environ.items() if not k.startswith("SEGGER_B200_")}
    env.update(ENVS[name])
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "gat_env_worker.py")], env=env, cwd=ROOT,
                       capture_output=True, text=True, timeout=900)
    print(r.stdout[-4000:], r.stderr[-4000:])
    assert r.returncode == 0
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    res = json.loads(lines[-1])
    assert res["ok"] and res["env"] == ENVS[name] and res["cases"]


def test_skipgat_slope_outside_unit_interval_trains():
    """GATv2Conv(negative_slope=1.5): the sub-warp kernels decline the slope, so the tx-belongs-bd conv on a
    unique-source belongs graph (one virtual source per edge) must take the two-pass backward.  Same layer on the
    same edges shuffled (full projection path) -> same outputs and gradients; a training step with dropout runs."""
    from segger_b200 import ops
    from segger_b200.ist_encoder import SkipGAT
    from oracle.ist_encoder_ref import TB, TT
    from tests.util import synth_batch

    torch.manual_seed(1)
    ts, x, edges, pos, bat = synth_batch(3000, 30, seed=6)
    layer = SkipGAT((-1, -1), 64, 2).cuda().eval()
    for conv in layer.conv.convs.values():
        conv.negative_slope = 1.5
    e_tt, e_tb = edges[TT].cuda(), edges[TB].cuda()
    assert bool((e_tb[0][1:] > e_tb[0][:-1]).all())
    perm = torch.randperm(e_tb.size(1), generator=torch.Generator().manual_seed(0)).cuda()
    g = torch.Generator().manual_seed(2)
    x_tx0, x_bd0 = torch.randn(3000, 96, generator=g).cuda(), torch.randn(30, 96, generator=g).cuda()
    go_tx, go_bd = torch.randn(3000, 128, generator=g).cuda(), torch.randn(30, 128, generator=g).cuda()
    res = []
    for tb in (e_tb, e_tb[:, perm].contiguous()):
        ops.CSR_CACHE.clear()
        layer.zero_grad()
        x_tx, x_bd = x_tx0.clone().requires_grad_(), x_bd0.clone().requires_grad_()
        out = layer({"tx": x_tx, "bd": x_bd}, {TT: e_tt, TB: tb})
        ((out["tx"] * go_tx).sum() + (out["bd"] * go_bd).sum()).backward()
        res.append((out["tx"].detach(), out["bd"].detach(), x_tx.grad, x_bd.grad,
                    {n: p.grad.clone() for n, p in layer.named_parameters() if p.grad is not None}))
    for a, b in zip(res[0][:4], res[1][:4]):
        assert float((a - b).abs().max()) <= 1e-5 * float(b.abs().max())
    assert res[0][4].keys() == res[1][4].keys() and len(res[0][4]) == 12
    for n in res[0][4]:
        a, b = res[0][4][n], res[1][4][n]
        assert float((a - b).abs().max()) <= 1e-5 * float(b.abs().max()), n
    layer.train()
    ops.CSR_CACHE.clear()
    layer.zero_grad()
    out = layer({"tx": x_tx0.clone().requires_grad_(), "bd": x_bd0.clone()}, {TT: e_tt, TB: e_tb})
    ((out["tx"] * go_tx).sum() + (out["bd"] * go_bd).sum()).backward()
    assert all(bool(torch.isfinite(p.grad).all()) for p in layer.parameters() if p.grad is not None)
