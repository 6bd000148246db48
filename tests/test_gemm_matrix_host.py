"""Coverage of the projection-GEMM parity matrix (tests/gemm_matrix.py), checked on the host: the cases reach every kernel
instantiation the dispatch mirror can produce on a 148-SM B200, and the edges the kernels are written around."""
import itertools

from tests.gemm_matrix import (BK, CASES, DEFAULT_ENV, REDUCED, SM_COUNT_B200, Case, cdiv, expected_kernel, ts_family,
                               ts_grid)

SM = SM_COUNT_B200
DIMS = (1, 4, 8, 12, 16, 30, 36, 60, 64, 65, 96, 100, 128, 160, 256, 260, 288, 1024, 18944, 18948, 20000)


def _reachable():
    keys = set()
    for M, N, K in itertools.product((1, 255, 256, 4096, 100000), DIMS, DIMS):
        for y_act, out, a_mis in itertools.product(("none", "aligned", "misaligned"), ("plain", "misaligned"), (False, True)):
            keys.add(expected_kernel(Case("", "fwd", M, N, K, act=1 if y_act != "none" else 0, y_act=y_act, out=out,
                                          a_misaligned=a_mis), SM)[0])
        for table, exact in itertools.product(("aligned", "misaligned", "ld_odd"), (0, 2)):
            keys.add(expected_kernel(Case("", "gather", M, N, K, table=table, exact=exact), SM)[0])
        for acc, act, out, a_mis in itertools.product((False, True), (0, 1), ("plain", "misaligned"), (False, True)):
            keys.add(expected_kernel(Case("", "dgrad", M, N, K, accumulate=acc, act=act, out=out, a_misaligned=a_mis), SM)[0])
        for a_mis in (False, True):
            keys.add(expected_kernel(Case("", "wgrad", M, N, K, a_misaligned=a_mis), SM)[0])
    return keys


def test_cases_cover_every_reachable_instantiation():
    reachable = _reachable()
    covered = {expected_kernel(c, SM)[0] for c in CASES}
    assert covered - reachable == set()
    assert sorted(map(str, reachable - covered)) == []
    ts = {k for k in reachable if k[0] == "ts"}
    # 7 (BN, S, B_RES) families; PP fixed by the depth except on BN = 128 streamed (deep, or > 148 n-tiles shallow)
    assert len({k[1:4] for k in ts}) == 7
    assert len(ts) == 32
    assert {k for k in reachable if k[0] == "ss_wgrad"} == {("ss_wgrad", bn, s) for bn in (64, 128) for s in (False, True)}
    assert {("simt", "fwd"), ("simt", "dgrad"), ("simt", "wgrad"), ("skinny", "fwd"), ("skinny", "wgrad"),
            ("rows_gather",)} <= covered


def test_case_names_are_unique_and_reduced_set_exists():
    names = [c.name for c in CASES]
    assert len(names) == len(set(names))
    assert set(REDUCED) <= set(names)


def _ts_cases():
    for c in CASES:
        key = expected_kernel(c, SM)[0]
        if key[0] == "ts":
            out_n, red = (c.N, c.K) if c.op in ("fwd", "gather") else (c.K, c.N)
            yield c, key, out_n, red


def test_edges_are_covered():
    ms = {c.M for c in CASES}
    assert {1, 127, 129} <= ms and any(m % 128 == 1 and m > 129 for m in ms)
    outs = [(c, key, out_n, red) for c, key, out_n, red in _ts_cases()]
    for bn in (64, 128):
        tails = [(out_n % 4) for c, key, out_n, _ in outs if key[1] == bn and out_n % bn]
        assert 0 in tails and any(t != 0 for t in tails), bn                 # N tail with and without N % 4 == 0
    assert {4, 28} <= {red % BK for *_, red in outs}
    # resident-weight families: num_n 3, 5, 7; persistent CTAs looping over a tile count that is not a grid multiple
    res = [ts_grid(c.M, out_n, key[1], True, SM) for c, key, out_n, _ in outs if key[3]]
    assert {3, 5, 7} <= {num_n for _, _, num_n in res}
    assert any(tiles > grid and tiles % grid for tiles, grid, _ in res)
    # alternating epilogue groups: a CTA that owns exactly one tile, and one that owns an odd number >= 3
    owned = set()
    for c, key, out_n, red in outs:
        if key[4]:
            tiles, grid, _ = ts_grid(c.M, out_n, key[1], key[3], SM)
            owned |= {cdiv(tiles - b, grid) for b in range(grid)}
    assert 1 in owned and any(o >= 3 and o % 2 for o in owned)


def test_ts_family_rule():
    assert ts_family(384, 64, SM) == (128, 2, True) and ts_family(384, 128, SM) == (128, 4, True)
    assert ts_family(384, 160, SM) == (128, 4, False) and ts_family(19000, 64, SM) == (128, 4, False)
    assert ts_family(64, 256, SM) == (64, 8, True) and ts_family(64, 288, SM) == (64, 4, False)
    assert expected_kernel(Case("", "fwd", 100, 19000, 64), SM, DEFAULT_ENV)[0] == ("ts", 128, 4, False, False, 0)
