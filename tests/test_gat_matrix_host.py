"""The GATv2 parity matrix (tests/gat_matrix.py) checked on the host: the cases reach every kernel instantiation the
dispatch mirror can produce on a 148-SM B200 and the edges the kernels are written around, the mirror's sub-warp shape
table agrees with the library's, and the float64 checker rejects plausible subtle kernel bugs."""
import itertools

import pytest
import torch

from tests.gat_matrix import (CASES, DEFAULT_ENV, LEGACY, QUAD_COMBOS, REDUCED, SM_COUNT_B200, VEC_COMBOS, Case, Inputs,
                              Env, check_outputs, chunking, classify, emulate, graph, host_inputs, kernel_set, quad_path,
                              quad_shape, reference, uses_direct, uses_logits, _seed)

SM = SM_COUNT_B200
CS = (7, 16, 32, 50, 64, 96, 100, 128, 200, 256, 300, 512)


def _reachable(env=DEFAULT_ENV):
    keys = set()
    for H, C, slope, layout, g, lg in itertools.product(range(1, 9), CS, (0.2, 1.5), ("plain", "misaligned"),
                                                         ("ragged", "unique"), (True, False)):
        keys |= kernel_set(Case("", H, C, slope=slope, layout=layout, graph=g, logits=lg, alpha=True), SM, env)
    return keys


def test_cases_cover_every_reachable_instantiation():
    reachable = _reachable()
    covered = set().union(*(kernel_set(c, SM) for c in CASES))
    assert sorted(map(str, reachable - covered)) == []
    assert covered <= reachable
    # 12 quad shapes x {fwd, dst without logits, dst LEAN with logits, dst full with logits (one source per edge), src}
    for v, lpr, H in QUAD_COMBOS:
        base = (str(v), str(lpr), str(H))
        for k in (("gatv2_fwd_quad_kernel", base + ("4",)), ("gatv2_bwd_dst_quad_kernel", base + ("4", "3")),
                  ("gatv2_bwd_dst_lg_quad_kernel", base + ("3", "4", "true")),
                  ("gatv2_bwd_dst_lg_quad_kernel", base + ("4", "3", "false")), ("gatv2_bwd_src_quad_kernel", base + ("4",))):
            assert k in covered, k
    for vc in VEC_COMBOS:
        for k in ("gatv2_fwd_vec_kernel", "gatv2_bwd_dst_vec_kernel", "gatv2_bwd_src_vec_kernel"):
            assert (k, tuple(map(str, vc))) in covered
    for tc in (1, 2, 4, 8):
        for k in ("gatv2_fwd_gen_kernel", "gatv2_bwd_dst_gen_kernel", "gatv2_bwd_src_gen_kernel"):
            assert (k, (str(tc),)) in covered
    assert {("colsum_partials_kernel", ()), ("colsum_partials_gen_kernel", ()), ("quad_colsum_kernel", ()),
            ("gatv2_alpha_kernel", ())} <= covered


def test_env_switches_reach_their_forms():
    legacy = set().union(*(kernel_set(c, SM, Env(legacy=True)) for c in map(_case, LEGACY)))
    assert {("gatv2_fwd_vec_kernel", tuple(map(str, vc))) for vc in VEC_COMBOS} <= legacy
    occ4 = set().union(*(kernel_set(c, SM, Env(dst_occ=4)) for c in map(_case, REDUCED)))
    assert any(k[0] == "gatv2_bwd_dst_quad_kernel" and k[1][-1] == "4" for k in occ4)
    assert any(k[0] == "gatv2_bwd_dst_lg_quad_kernel" and k[1][-1] == "true" for k in occ4)
    occ3 = set().union(*(kernel_set(c, SM, Env(dst_occ=3)) for c in map(_case, REDUCED)))
    assert not any(k[0] == "gatv2_bwd_dst_lg_quad_kernel" and k[1][-1] == "true" for k in occ3)
    assert any(uses_direct(c) and uses_logits(c) for c in map(_case, REDUCED))
    assert any(uses_direct(c) and not uses_logits(c) for c in map(_case, REDUCED))


def _case(name):
    return next(c for c in CASES if c.name == name)


def test_case_names_are_unique_and_reduced_sets_exist():
    names = [c.name for c in CASES]
    assert len(names) == len(set(names))
    assert set(REDUCED) <= set(names) and set(LEGACY) <= set(names)


def _degrees(c):
    ei, n_src, n_dst, _ = graph(c, torch.Generator().manual_seed(_seed(c.name)))
    return torch.bincount(ei[1], minlength=n_dst), torch.bincount(ei[0], minlength=n_src)


def test_edges_are_covered():
    live = [c for c in CASES if not c.raises]
    degs = {c.name: _degrees(c) for c in live}
    assert any(int(d.max()) >= 2000 for d, _ in degs.values())
    assert all(bool((d == 0).any()) and bool((d == 1).any()) for c in live if c.graph in ("ragged", "hub")
               for d in [degs[c.name][0]])
    assert any(bool((o == 0).any()) for _, o in degs.values())                      # sources without out-edges
    assert any(c.graph == "empty" and quad_path(c) for c in live) and any(c.graph == "empty" and not quad_path(c) for c in live)
    quad = [c for c in live if quad_path(c) and c.graph != "empty"]
    # a zero-degree row beside rows with edges in one quad group (rows in chunk order: rpw == G, no sort)
    mixed = False
    for c in quad:
        G, rpw, _, _ = chunking(c, c.n_dst)
        d = degs[c.name][0]
        if rpw == G:
            grp = d[: d.numel() // G * G].view(-1, G)
            mixed |= bool(((grp == 0).any(1) & (grp > 0).any(1)).any())
    assert mixed
    # ragged degrees with rpw > G at default settings: the degree sort permutes
    assert any(chunking(c, c.n_dst)[1] > chunking(c, c.n_dst)[0] and c.graph == "ragged" for c in quad)
    assert any(c.n_dst < chunking(c, c.n_dst)[0] for c in quad)
    assert any(c.n_dst % chunking(c, c.n_dst)[0] for c in quad)
    assert any(c.n_dst % chunking(c, c.n_dst)[1] for c in quad if chunking(c, c.n_dst)[1] > chunking(c, c.n_dst)[0])
    # persistent dst grid: a warp owns several chunks, with and without saved logits
    pers = [c for c in quad if chunking(c, c.n_dst)[2] > 4 * chunking(c, c.n_dst)[3]]
    assert {uses_logits(c) for c in pers} == {True, False}
    assert {0.0, 0.2, 1.0, 1.5, -0.1} <= {c.slope for c in live}
    assert any(c.bias == "none" for c in live) and any(c.bias == "big" for c in live)
    assert any(not c.want_pre for c in live) and any(c.gelu and c.backward for c in live)
    drop = {(c.p, c.seed_dev) for c in live}
    assert {(0.2, False), (0.2, True), (0.5, False), (0.5, True)} <= drop
    fam = lambda c: "quad" if quad_path(c) else classify(c.H, c.C, c.layout != "misaligned")[0]  # noqa: E731
    assert {fam(c) for c in live if c.p > 0} == {"quad", "vec", "gen"}
    assert {fam(c) for c in live if c.alpha} == {"quad", "vec", "gen"}
    assert any(c.layout == "slice3f" and quad_path(c) for c in live)
    assert any(c.layout == "misaligned" and quad_shape(c.H, c.C) for c in live)
    assert {(uses_direct(c), uses_logits(c)) for c in live if uses_direct(c)} == {(True, True), (True, False)}
    assert any(c.direct and not uses_direct(c) for c in live)                        # slope outside [0, 1]
    assert {fam(c) for c in live if c.graph == "scripted"} == {"quad", "vec", "gen"}
    assert any(c.raises and c.layout == "plain" for c in CASES) and any(c.raises and c.layout != "plain" for c in CASES)


def test_quad_shape_table_matches_library():
    from segger_b200 import _lib
    lib = _lib.load()
    for H in range(1, 9):
        for C in range(1, 513):
            assert (quad_shape(H, C) is not None) == bool(lib.sgb_gatv2_quad_supported(H, C)), (H, C)


# ---------------------------------------------------------------------------------------------------------------------
# negative controls: the checker rejects plausible subtle bugs on small CPU float64 cases
# ---------------------------------------------------------------------------------------------------------------------
def _control_inputs():
    c = Case("negative_control", 2, 16, n_src=40, n_dst=30, avg=4, slope=0.2)
    ei, n_src, n_dst, x_l, x_r, att, bias, grad_out, rowptr, col, eid = host_inputs(c)
    deg = rowptr[1:] - rowptr[:-1]
    row = torch.repeat_interleave(torch.arange(n_dst), deg)
    for p in range(0, row.numel(), 7):                 # exact zeros of z = x_l + x_r on a few edges
        x_l[col[p], 3] = -x_r[row[p], 3]
    return Inputs(x_l, x_r, att, bias, grad_out, rowptr, col, eid, None, 2, 16, 0.2, 0.0)


def test_checker_accepts_the_rounded_reference():
    inp = _control_inputs()
    vals, bounds = reference(inp)
    chk = check_outputs(emulate(vals), vals, bounds, inp.bias)
    assert not chk.failures, chk.failures


@pytest.mark.parametrize("bug,where", [("drop_edge", "out"), ("att_head", "e_logit"), ("kink", "grad_x_r"),
                                       ("cta_partial", "grad_att"), ("row_scale", "out")])
def test_checker_rejects_subtle_bugs(bug, where):
    inp = _control_inputs()
    z = inp.x_l[inp.col.long()] + inp.x_r[torch.repeat_interleave(torch.arange(30), inp.rowptr[1:] - inp.rowptr[:-1])]
    assert bool((z == 0).any())
    vals, bounds = reference(inp)
    bad, _ = reference(inp, bug=bug)
    chk = check_outputs(emulate(bad), vals, bounds, inp.bias)
    assert any(f.startswith(where) for f in chk.failures), chk.failures
