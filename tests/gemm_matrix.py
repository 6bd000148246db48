"""The projection-GEMM parity matrix: a host-side mirror of the dispatch rules of sgb_linear_{fwd,fwd_gather,dgrad,wgrad}
(segger_b200/csrc/sgb_linear*.cu), the cases that reach every kernel instantiation they can pick, and a runner that
checks one case against float64 with a per-element error bound.

Shared by tests/test_gpu_gemm_matrix.py (every case, default settings), tests/test_gemm_matrix_host.py (coverage of the
mirror, no GPU) and tests/gemm_env_worker.py (one case per family under each SEGGER_B200_GEMM* switch).

Error bound.  A tensor-core product sums, per output element, K products split into TF32 halves (x = hi + lo, each half
rounded to nearest; the dropped lo*lo term and the split leave ~2^-22 of |a||b| per product), accumulated inside the
tensor core with truncation over a chunk of 32 or 64 products, then chunk by chunk in registers with round-to-nearest.
Every one of these errors is a fraction of a partial sum of |a_k||b_k|, so

    |c - c_ref| <= tau(K) * (sum_k |a_k| |b_k| + |terms added in the epilogue|),   tau(K) = TAU_C * (K/8 + 16) * 2^-24

elementwise (the magnitude in float64).  TAU_C is calibrated on a B200 (profiles/gemm_matrix_ratios_b200.json): the worst
measured err / magnitude over the matrix sits 4-8x below tau.  A GEMM that loses one split term is off by ~2^-12 of
|a||b| per product, which exceeds tau at shallow depths (K up to a few hundred).  The same bound is
applied to the fp32 SIMT and skinny kernels (round-to-nearest FMAs: well inside it).
"""
from __future__ import annotations

import json
import math
from dataclasses import dataclass, field
from typing import Optional

import torch

BM, BK = 128, 32
SM_COUNT_B200 = 148
TAU_C = 2.0              # calibrated, see the module docstring
TAU_SUM_C = 1.0          # column sums (db): tau_sum(M) = TAU_SUM_C * (M/64 + 16) * 2^-24
EPS_ACT = 2.0 ** -20     # fp32 erf / __expf and the final roundings of an activation or its derivative


def tau(k: int) -> float:
    return TAU_C * (k / 8 + 16) * 2.0 ** -24


def tau_sum(m: int) -> float:
    return TAU_SUM_C * (m / 64 + 16) * 2.0 ** -24


def cdiv(a: int, b: int) -> int:
    return -(-a // b)


# ---------------------------------------------------------------------------------------------------------------------
# dispatch mirror
# ---------------------------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class Env:
    """The process-wide A/B switches (each read once into a static by the library)."""
    simt: bool = False          # SEGGER_B200_GEMM=simt
    ts: bool = True             # SEGGER_B200_GEMM_TS=0 -> False
    wm_general: bool = False    # SEGGER_B200_GEMM_WM=0 -> True
    pp: Optional[int] = None    # SEGGER_B200_GEMM_PP=0|1

    def variables(self) -> dict:
        v = {}
        if self.simt:
            v["SEGGER_B200_GEMM"] = "simt"
        if not self.ts:
            v["SEGGER_B200_GEMM_TS"] = "0"
        if self.wm_general:
            v["SEGGER_B200_GEMM_WM"] = "0"
        if self.pp is not None:
            v["SEGGER_B200_GEMM_PP"] = str(self.pp)
        return v


DEFAULT_ENV = Env()


@dataclass(frozen=True)
class Case:
    """One call.  Shapes use the C ABI's names: fwd / gather x[M,K] w[N,K] -> y[M,N]; dgrad dy[M,N] w[N,K] -> dx[M,K];
    wgrad dy[M,N] x[M,K] -> dw[N,K], db[N]."""
    name: str
    op: str                       # fwd | gather | dgrad | wgrad
    M: int
    N: int
    K: int
    bias: bool = True             # fwd / gather
    act: int = 0                  # fwd: y_act = act(y);  dgrad: act' applied with act_pre
    y_act: str = "none"           # fwd: none | aligned | misaligned
    out: str = "plain"            # y / dx / dw view: plain | strided (aligned, ld > width) | misaligned
    a_misaligned: bool = False    # x (fwd) / dy (dgrad, wgrad) as a column slice at a 4-byte offset
    ids: str = "int64"            # gather: int32 | int64
    table: str = "aligned"        # gather: aligned | misaligned | ld_odd
    accumulate: bool = False      # dgrad / wgrad
    act_pre: str = "aligned"      # dgrad with act != 0: aligned | misaligned
    want_db: bool = True          # wgrad
    exact: int = 0                # fwd / gather
    scaled: bool = True           # rows / columns scaled by 2^[-40, 40], a few zeroed

    def __str__(self):
        return self.name


def _out_width(c: Case) -> int:
    return {"fwd": c.N, "gather": c.N, "dgrad": c.K, "wgrad": c.K}[c.op]


def _vec(misaligned: bool, ld: int) -> bool:
    return not misaligned and ld % 4 == 0


def _views(c: Case):
    """(A operand vector-loadable, output vector-storable, y_act vector-storable, table vector-loadable)."""
    red = {"fwd": c.K, "gather": c.K, "dgrad": c.N, "wgrad": c.N}[c.op]
    a_ld = red + 1 if c.a_misaligned else red
    w = _out_width(c)
    out_ld = w + 8 if c.out == "strided" else (w + 1 if c.out == "misaligned" else w)
    a_vec = _vec(c.a_misaligned, a_ld)
    out_vec = _vec(c.out == "misaligned", out_ld)
    ya_vec = c.y_act == "aligned" and c.N % 4 == 0 if c.y_act != "none" else None
    tab_ld = {"aligned": c.N, "misaligned": c.N + 1, "ld_odd": c.N + 3}[c.table]
    tab_vec = _vec(c.table == "misaligned", tab_ld)
    return a_vec, out_vec, ya_vec, tab_vec


def ts_family(out_n: int, red_k: int, sm: int):
    """run_packed: (BN, S, B_RES) of the TS kernel for output width out_n and reduction depth red_k."""
    bn = 64 if out_n <= 64 else 128
    num_n, num_ks = cdiv(out_n, bn), cdiv(red_k, BK)
    if bn == 128:
        if num_ks <= 4 and num_n <= sm:
            return 128, (2 if num_ks <= 2 else 4), True
        return 128, 4, False
    if num_ks <= 8 and num_n <= sm:
        return 64, (2 if num_ks <= 2 else 4 if num_ks <= 4 else 8), True
    return 64, 4, False


def ts_grid(M: int, out_n: int, bn: int, b_res: bool, sm: int):
    """launch_ts_wm: (tiles, grid, num_n)."""
    num_n = cdiv(out_n, bn)
    tiles = cdiv(M, BM) * num_n
    grid = min(tiles, sm)
    if b_res:
        grid = grid // num_n * num_n
        if grid < num_n:
            grid = num_n if num_n < tiles else tiles
    return tiles, grid, num_n


def _packed(c: Case, out_n: int, red_k: int, wm: int, sm: int, env: Env):
    bn = 64 if out_n <= 64 else 128
    if not env.ts:
        s = 3 if bn == 128 else 4
        return ("ss_fwd", bn), [("pack_b_kernel", (bn,)), ("gemm_tf32x3_kernel", (bn, False, False, True, s))]
    BN, S, b_res = ts_family(out_n, red_k, sm)
    pp = (env.pp == 1) if env.pp is not None else cdiv(red_k, BK) >= 3
    if env.wm_general:
        wm = 4
    return ("ts", BN, S, b_res, pp, wm), [("pack_b_kernel", (bn,)), ("gemm_tf32x3_ts_kernel", (BN, S, b_res, pp, wm))]


def _skinny_fwd_ok(c: Case, a_vec, out_vec, ya_vec) -> bool:
    return (c.M >= 4096 and 4 <= c.K <= 16 and c.K % 4 == 0 and 4 <= c.N <= 256 and c.N % 4 == 0 and a_vec and out_vec
            and ya_vec is not False)


def _simt_fwd(c: Case):
    return ("simt", "fwd"), [("sgemm_kernel", (128 if c.N > 64 else 64, True, True))]


def expected_kernel(c: Case, sm: int = SM_COUNT_B200, env: Env = DEFAULT_ENV):
    """(coverage key, [(kernel base name, template arguments)] that must launch) for case c."""
    a_vec, out_vec, ya_vec, tab_vec = _views(c)
    tc = not env.simt
    k4 = lambda k: min(k // 4, 4)  # noqa: E731  skinny kernels: switch (K / 4) {1, 2, 3, default 4}
    if c.op in ("fwd", "gather"):
        tc_ok = tc and c.M >= 1 and c.N >= 8 and c.K >= 8 and c.K % 4 == 0 and a_vec
        ya = None if c.op == "gather" else ya_vec
        skinny = _skinny_fwd_ok(c, a_vec, out_vec, ya)
        if c.op == "gather" and c.exact != 2 and tc_ok and not skinny:
            vec_c = out_vec and c.N % 4 == 0
            wm = 1 if (vec_c and tab_vec) else 4
            return _packed(c, c.N, c.K, wm, sm, env)
        if skinny:
            key, ks = ("skinny", "fwd"), [("skinny_fwd_kernel", (k4(c.K),))]
        elif c.exact != 2 and tc_ok:
            vec_c = out_vec and c.N % 4 == 0
            wm = 4 if not vec_c else (0 if ya is None else (2 if ya else 4))
            key, ks = _packed(c, c.N, c.K, wm, sm, env)
        else:
            key, ks = _simt_fwd(c)
        if c.op == "gather":
            return ("rows_gather",), ks + [("rows_gather_add_kernel", ("int" if c.ids == "int32" else "long",))]
        return key, ks
    if c.op == "dgrad":
        if tc and c.M >= 1 and c.K >= 8 and c.N >= 8 and c.N % 4 == 0 and a_vec:
            vec_c = out_vec and c.K % 4 == 0
            wm = 4 if (not vec_c or c.act or c.accumulate) else 0
            return _packed(c, c.K, c.N, wm, sm, env)
        return ("simt", "dgrad"), [("sgemm_kernel", (128 if c.K > 64 else 64, True, False))]
    # wgrad (x is always aligned here; only dy may be misaligned)
    M, N, K = c.M, c.N, c.K
    if M >= 4096 and 4 <= K <= 16 and K % 4 == 0 and 1 <= N <= 256:
        vec = (N & (N - 1)) == 0 and 4 <= N <= 128 and a_vec
        return ("skinny", "wgrad"), [("skinny_wgrad_vec_kernel" if vec else "skinny_wgrad_kernel", (k4(K),)),
                                     ("skinny_wgrad_reduce_kernel", ())]
    if tc and M >= 256 and N >= 8 and K >= 8 and N % 4 == 0 and K % 4 == 0 and a_vec:
        splits = tc_wgrad_splits(M, N, K, sm)
        bn = 64 if K <= 64 else 128
        ks = [("gemm_tf32x3_kernel", (bn, True, True, False, 3 if bn == 128 else 4))]
        if splits > 1:
            ks.append(("tc_splitk_reduce_kernel", ()))
            if c.want_db:
                ks.append(("tc_colsum_reduce_kernel", ()))
        return ("ss_wgrad", bn, splits > 1), ks
    ks = [("sgemm_kernel", (128 if K > 64 else 64, False, False))]
    if simt_wgrad_splits(M, N, K, sm) > 1:
        ks.append(("splitk_reduce_kernel", ()))
    if c.want_db:
        ks += [("colsum_stage1_kernel", ()), ("colsum_stage2_kernel", ())]
    return ("simt", "wgrad"), ks


def tc_wgrad_splits(M: int, N: int, K: int, sm: int) -> int:
    """tc_wgrad_splits + the trim in tc_linear_wgrad (every split owns at least one k-stage)."""
    bn = 64 if K <= 64 else 128
    s = max(1, min(sm // (cdiv(N, BM) * cdiv(K, bn)), cdiv(M, 8 * BK)))
    kps = cdiv(cdiv(M, s), BK) * BK
    while s > 1 and (s - 1) * kps >= M:
        s -= 1
    return s


def simt_wgrad_splits(M: int, N: int, K: int, sm: int) -> int:
    tiles = cdiv(N, BM) * cdiv(K, 128 if K > 64 else 64)
    s = (sm * 2 + tiles - 1) // tiles
    return max(1, min(s, cdiv(max(M, 1), 4 * BK), 512))


# ---------------------------------------------------------------------------------------------------------------------
# the matrix
# ---------------------------------------------------------------------------------------------------------------------
GELU, SILU = 1, 2
F, G, D, W = "fwd", "gather", "dgrad", "wgrad"

CASES = [
    # --- TS (128, 2, resident), PP off ------------------------------------------------------------------------------
    Case("ts128r2_wm0", F, 20000, 384, 36),                                     # num_n 3, 471 tiles on 147 CTAs
    Case("ts128r2_wm1_ntail", G, 777, 100, 60, ids="int32"),                   # N % 128 = 100, table ld == N
    Case("ts128r2_wm1_int64_nobias", G, 4096, 72, 40, bias=False),
    Case("ts128r2_wm2", F, 129, 640, 64, act=GELU, y_act="aligned"),           # num_n 5
    Case("ts128r2_wm4_ntail4", F, 127, 130, 40, act=SILU, y_act="aligned"),    # N % 4 != 0
    Case("ts128r2_wm4_tab_ld", G, 1000, 200, 64, table="ld_odd"),
    Case("ts128r2_m1", F, 1, 136, 12),
    # --- TS (128, 4, resident), PP on --------------------------------------------------------------------------------
    Case("ts128r4_wm0_pp1tile", F, 4097, 896, 100, bias=False),               # num_n 7; 231 tiles: CTAs own 1 or 2
    Case("ts128r4_wm1", G, 5000, 384, 128),
    Case("ts128r4_wm2", F, 3000, 200, 92, act=GELU, y_act="aligned"),         # K % 32 = 28, N tail
    Case("ts128r4_wm4_yact_mis", F, 2000, 256, 96, act=SILU, y_act="misaligned"),
    Case("ts128r4_wm4_dgrad", D, 1000, 96, 256, accumulate=True, act=GELU),
    Case("ts128r4_wm0_exact1", F, 513, 384, 128, exact=1, out="strided"),
    # --- TS (128, 4, streamed) ---------------------------------------------------------------------------------------
    Case("ts128s_pp_wm0_odd", F, 20001, 384, 260),                             # 471 tiles on 148 CTAs: 3 or 4 each
    Case("ts128s_pp_wm1", G, 4096, 384, 300, ids="int32"),
    Case("ts128s_pp_wm2", F, 1000, 260, 160, act=SILU, y_act="aligned", bias=False),
    Case("ts128s_pp_wm4_ymis", F, 1000, 384, 256, act=GELU, y_act="aligned", out="misaligned"),
    Case("ts128s_pp_wm4_dgrad_none", D, 2000, 512, 384, accumulate=True),
    Case("ts128s_nopp_wm0", F, 128, 19000, 64),                                # 149 n-tiles, N % 128 = 56
    Case("ts128s_nopp_wm1", G, 130, 19200, 32),
    Case("ts128s_nopp_wm2", F, 64, 19004, 60, act=GELU, y_act="aligned"),
    Case("ts128s_nopp_wm4_dgrad", D, 200, 64, 19000, accumulate=True, act=SILU),
    # --- TS (64, 2, resident), PP off --------------------------------------------------------------------------------
    Case("ts64r2_wm0_m1", F, 1, 64, 8),
    Case("ts64r2_wm1_n36", G, 2000, 36, 28),                                   # N % 64 = 36
    Case("ts64r2_wm2", F, 129, 48, 64, act=SILU, y_act="aligned"),
    Case("ts64r2_wm4_dgrad_ktail", D, 5000, 32, 37),                           # dx width 37
    # --- TS (64, 4, resident), PP on ---------------------------------------------------------------------------------
    Case("ts64r4_wm0_dgrad", D, 10000, 100, 64),                               # plain dgrad writes with WM 0
    Case("ts64r4_wm1", G, 1000, 64, 96),
    Case("ts64r4_wm2", F, 300, 60, 128, act=GELU, y_act="aligned"),
    Case("ts64r4_wm4_ntail4", F, 127, 50, 68, act=SILU, y_act="aligned"),
    # --- TS (64, 8, resident), PP on ---------------------------------------------------------------------------------
    Case("ts64r8_wm0_odd", F, 37889, 64, 256),                                 # 297 tiles: CTA 0 owns 3
    Case("ts64r8_wm1", G, 3000, 64, 200, ids="int32"),
    Case("ts64r8_wm2", F, 500, 40, 220, act=SILU, y_act="aligned"),
    Case("ts64r8_wm4_dgrad_pre_mis", D, 3000, 160, 64, accumulate=True, act=GELU, act_pre="misaligned"),
    # --- TS (64, 4, streamed), PP on ---------------------------------------------------------------------------------
    Case("ts64s_wm0", F, 5000, 64, 292),
    Case("ts64s_wm1_strided", G, 2049, 64, 512, out="strided"),
    Case("ts64s_wm2", F, 700, 24, 1024, act=GELU, y_act="aligned"),
    Case("ts64s_wm4_tab_mis", G, 1500, 64, 300, table="misaligned", ids="int32"),
    Case("ts64s_wm4_dgrad", D, 3000, 512, 48, act=SILU),
    # --- dgrad epilogue order: (dy W [+ dx]) * act'(pre) -------------------------------------------------------------
    Case("dgrad_acc_gelu", D, 1500, 384, 128, accumulate=True, act=GELU),
    Case("dgrad_acc_silu_pre_mis", D, 1500, 384, 128, accumulate=True, act=SILU, act_pre="misaligned"),
    Case("dgrad_acc_none", D, 1500, 384, 128, accumulate=True),
    Case("dgrad_gelu", D, 1500, 384, 128, act=GELU),
    Case("dgrad_dx_strided", D, 777, 256, 128, out="strided", accumulate=True),
    # --- SS wgrad ------------------------------------------------------------------------------------------------------
    Case("ss128_split1_m256", W, 256, 200, 100, accumulate=True, out="strided"),
    Case("ss128_split1_80tiles", W, 4096, 1280, 1024),
    Case("ss64_split1_m256", W, 256, 96, 64, want_db=False),
    Case("ss128_splitk", W, 20000, 256, 128, accumulate=True),
    Case("ss64_splitk", W, 50001, 64, 36, accumulate=True, out="strided"),
    Case("ss64_splitk_nodb", W, 3000, 384, 60, want_db=False),
    # --- SIMT ----------------------------------------------------------------------------------------------------------
    Case("simt_fwd_k30", F, 100, 50, 30, act=GELU, y_act="aligned"),
    Case("simt_fwd_xmis", F, 3000, 130, 64, a_misaligned=True, act=SILU, y_act="misaligned"),
    Case("simt_fwd_exact2", F, 1000, 384, 256, exact=2, out="misaligned"),
    Case("simt_dgrad_dymis", D, 1000, 65, 70, a_misaligned=True, accumulate=True, act=GELU),
    Case("simt_dgrad_n_tail", D, 129, 66, 64),
    Case("simt_wgrad_m200", W, 200, 96, 128, accumulate=True),
    Case("simt_wgrad_k30", W, 3000, 64, 30),
    Case("simt_wgrad_dymis", W, 1000, 40, 48, a_misaligned=True, accumulate=True, out="strided"),
    # --- skinny (K <= 16) ----------------------------------------------------------------------------------------------
    Case("skinny_fwd", F, 8193, 100, 12, act=SILU, y_act="aligned"),
    Case("skinny_wgrad_vec", W, 8192, 64, 16, accumulate=True),
    Case("skinny_wgrad", W, 5000, 100, 8, out="strided"),
    # --- gather through the SIMT / skinny forward + rows_gather_add ---------------------------------------------------
    Case("rows_gather_exact2", G, 1000, 100, 64, exact=2),
    Case("rows_gather_skinny", G, 5000, 64, 16, ids="int32"),
]

# one case per family for the A/B switches (tests/gemm_env_worker.py)
REDUCED = ["ts128r2_wm2", "ts128r4_wm1", "ts128s_pp_wm0_odd", "ts128s_nopp_wm0", "ts64r2_wm1_n36", "ts64r4_wm0_dgrad",
           "ts64r8_wm4_dgrad_pre_mis", "ts64s_wm2", "ss128_split1_m256", "ss64_splitk", "simt_fwd_k30", "skinny_fwd",
           "rows_gather_exact2"]


def case(name: str) -> Case:
    return next(c for c in CASES if c.name == name)


# ---------------------------------------------------------------------------------------------------------------------
# runner
# ---------------------------------------------------------------------------------------------------------------------
SENTINEL = -12345.5


def _rand(shape, g, dev):
    """Random signs, magnitudes >= 2^-8 (so that 2^-40 scaling keeps every split half normal)."""
    v = torch.randn(shape, generator=g, dtype=torch.float32)
    v = torch.where(v.abs() < 2.0 ** -8, torch.copysign(torch.full_like(v, 2.0 ** -8), v), v)
    return v.to(dev)


def _scales(n, g, dev, scaled):
    """Per-index factors 2^s, s in [-40, 40], with a few indices zeroed."""
    if not scaled:
        return torch.ones(n, device=dev)
    s = torch.randint(-40, 41, (n,), generator=g).double()
    f = torch.pow(2.0, s).float()
    if n >= 3:
        f[torch.randperm(n, generator=g)[: max(1, n // 97)]] = 0.0
    return f.to(dev)


def _keep(n, g, dev, scaled):
    """1 for most indices, 0 for a few (all-zero rows / columns)."""
    return (_scales(n, g, dev, scaled) != 0).float()


def _buffer(rows, cols, kind, dev, fill=SENTINEL):
    """A [rows, cols] view of a sentinel-filled buffer: plain (the buffer itself), strided (ld = cols + 8, aligned) or
    misaligned (4-byte offset, ld = cols + 1)."""
    if kind == "plain":
        buf = torch.full((rows, cols), fill, device=dev)
        return buf, buf
    pad, off = (8, 4) if kind == "strided" else (1, 1)
    buf = torch.full((rows, cols + pad), fill, device=dev)
    return buf, buf[:, off:off + cols]


def _act64(v, act):
    if act == GELU:
        return torch.nn.functional.gelu(v)
    if act == SILU:
        return torch.nn.functional.silu(v)
    return v


def _dact64(v, act):
    if act == GELU:
        cdf = 0.5 * (1 + torch.erf(v / math.sqrt(2)))
        return cdf + v * torch.exp(-0.5 * v * v) / math.sqrt(2 * math.pi)
    if act == SILU:
        s = torch.sigmoid(v)
        return s * (1 + v * (1 - s))
    return torch.ones_like(v)


@dataclass
class Check:
    """Worst err / magnitude and worst err / bound of each output of a case."""
    ratio: dict = field(default_factory=dict)
    usage: dict = field(default_factory=dict)
    failures: list = field(default_factory=list)

    def add(self, what, got, ref, mag, bound):
        got = got.double()
        err = (got - ref).abs()
        bad = ~(err <= bound)                   # NaN fails too
        nz = mag > 0
        self.ratio[what] = float((err[nz] / mag[nz]).max()) if bool(nz.any()) else 0.0
        pos = bound > 0
        self.usage[what] = float((err[pos] / bound[pos]).max()) if bool(pos.any()) else 0.0
        if bool(bad.any()):
            i = int(bad.flatten().nonzero()[0])
            self.failures.append(f"{what}: {int(bad.sum())} elements out of bound; first flat index {i}: "
                                 f"got {got.flatten()[i].item()!r} ref {ref.flatten()[i].item()!r} "
                                 f"bound {bound.flatten()[i].item():.3e}")

    def untouched(self, what, buf, view, before):
        """Everything of buf outside view still holds `before`."""
        mask = torch.ones_like(buf, dtype=torch.bool)
        mask_view = mask.as_strided(view.shape, view.stride(), view.storage_offset() - buf.storage_offset())
        mask_view.fill_(False)
        if not torch.equal(buf[mask], before[mask]):
            self.failures.append(f"{what}: the call wrote outside the output view")


def run_case(c: Case, dev="cuda", seed=None):
    """Runs c twice; returns (Check, outputs of the first call, outputs of the second).  Inputs are seeded by the
    case's name."""
    from segger_b200 import ops

    seed = seed if seed is not None else sum(ord(ch) * (i + 1) for i, ch in enumerate(c.name))
    g = torch.Generator().manual_seed(seed)
    chk = Check()
    M, N, K = c.M, c.N, c.K

    def a_operand(rows, cols):
        if c.a_misaligned:
            buf = torch.zeros(rows, cols + 1, device=dev)
            return buf[:, 1:]
        return torch.empty(rows, cols, device=dev)

    if c.op in ("fwd", "gather"):
        x = a_operand(M, K)
        x.copy_(_rand((M, K), g, dev) * _scales(M, g, dev, c.scaled)[:, None] * _keep(K, g, dev, c.scaled)[None, :])
        wsc = _scales(N, g, dev, c.scaled)
        w = _rand((N, K), g, dev) * wsc[:, None]
        b = _rand((N,), g, dev) * torch.where(wsc > 0, wsc, torch.ones_like(wsc)) if c.bias else None
        ref = x.double() @ w.double().t()
        mag = x.double().abs() @ w.double().abs().t()
        if b is not None:
            ref += b.double()
            mag += b.double().abs()
        gather = None
        if c.op == "gather":
            n_rows = 37
            ids = torch.randint(0, n_rows, (M,), generator=g).to(dev)      # repeated, unsorted
            ids = ids.to(torch.int32) if c.ids == "int32" else ids
            tsc = torch.pow(2.0, torch.randint(-20, 21, (n_rows,), generator=g).double()).float().to(dev) if c.scaled else torch.ones(n_rows, device=dev)
            tvals = _rand((n_rows, N), g, dev) * tsc[:, None]
            if c.table == "aligned":
                table = tvals.clone()
            else:
                pad, off = (1, 1) if c.table == "misaligned" else (3, 0)
                tbuf = torch.zeros(n_rows, N + pad, device=dev)
                table = tbuf[:, off:off + N]
                table.copy_(tvals)
            gather = (ids, table)
            tg = table.double()[ids.long()]
            ref += tg
            mag += tg.abs()
        bound = tau(K) * mag

        def call():
            ybuf, y = _buffer(M, N, c.out, dev)
            yabuf, ya = (_buffer(M, N, "plain" if c.y_act == "aligned" else "misaligned", dev)
                         if c.y_act != "none" else (None, None))
            ops.linear_fwd(x, w, b, c.act, y=y, y_act=ya, exact=c.exact, gather=gather)
            return {"y": (ybuf, y), **({"y_act": (yabuf, ya)} if ya is not None else {})}

        outs = call(), call()
        ybuf, y = outs[0]["y"]
        chk.add("y", y, ref, mag, bound)
        chk.untouched("y", ybuf, y, torch.full_like(ybuf, SENTINEL))
        if "y_act" in outs[0]:
            yabuf, ya = outs[0]["y_act"]
            aref = _act64(ref, c.act)
            chk.add("y_act", ya, aref, mag, _dact64(ref, c.act).abs() * bound + EPS_ACT * (aref.abs() + ref.abs()))
            chk.untouched("y_act", yabuf, ya, torch.full_like(yabuf, SENTINEL))
    elif c.op == "dgrad":
        dy = a_operand(M, N)
        msc, ksc = _scales(M, g, dev, c.scaled), _scales(K, g, dev, c.scaled)
        dy.copy_(_rand((M, N), g, dev) * msc[:, None])
        w = _rand((N, K), g, dev) * ksc[None, :] * _keep(N, g, dev, c.scaled)[:, None]
        v = dy.double() @ w.double()
        mag = dy.double().abs() @ w.double().abs()
        old = None
        if c.accumulate:
            old = _rand((M, K), g, dev) * (msc[:, None] * ksc[None, :]) * math.sqrt(N)
            v += old.double()
            mag += old.double().abs()
        pre = None
        if c.act:
            pre = torch.empty(M, K, device=dev) if c.act_pre == "aligned" else torch.zeros(M, K + 1, device=dev)[:, 1:]
            pre.copy_(torch.randn(M, K, generator=g) * 2)
            d = _dact64(pre.double(), c.act)
            ref = v * d
            bound = d.abs() * tau(N) * mag + EPS_ACT * (1 + pre.double().abs()) * v.abs()
        else:
            ref, bound = v, tau(N) * mag

        def call():
            fill = SENTINEL
            buf, dx = _buffer(M, K, c.out, dev, fill)
            if old is not None:
                dx.copy_(old)
            before = buf.clone()
            ops.linear_dgrad(dy, w, dx=dx, accumulate=c.accumulate, act=c.act, act_pre=pre)
            return {"dx": (buf, dx, before)}

        outs = call(), call()
        buf, dx, before = outs[0]["dx"]
        chk.add("dx", dx, ref, mag, bound)
        chk.untouched("dx", buf, dx, before)
    else:
        dy = a_operand(M, N)
        nsc, ksc = _scales(N, g, dev, c.scaled), _scales(K, g, dev, c.scaled)
        rsc = _keep(M, g, dev, c.scaled)                                      # a few all-zero rows
        dy.copy_(_rand((M, N), g, dev) * nsc[None, :] * rsc[:, None])
        x = _rand((M, K), g, dev) * ksc[None, :]
        ref = dy.double().t() @ x.double()
        mag = dy.double().abs().t() @ x.double().abs()
        dbref = dy.double().sum(0)
        dbmag = dy.double().abs().sum(0)
        old = oldb = None
        if c.accumulate:
            old = _rand((N, K), g, dev) * (nsc[:, None] * ksc[None, :]) * math.sqrt(M)
            oldb = _rand((N,), g, dev) * nsc * math.sqrt(M)
            ref += old.double()
            mag += old.double().abs()
            dbref += oldb.double()
            dbmag += oldb.double().abs()

        def call():
            buf, dw = _buffer(N, K, c.out, dev)
            db = torch.full((N,), SENTINEL, device=dev) if c.want_db else None
            if old is not None:
                dw.copy_(old)
                if db is not None:
                    db.copy_(oldb)
            before = buf.clone()
            ops.linear_wgrad(dy, x, dw=dw, db=db, want_db=c.want_db, accumulate=c.accumulate)
            return {"dw": (buf, dw, before), **({"db": (db, db, db)} if db is not None else {})}

        outs = call(), call()
        buf, dw, before = outs[0]["dw"]
        chk.add("dw", dw, ref, mag, tau(M) * mag)
        chk.untouched("dw", buf, dw, before)
        if c.want_db:
            db = outs[0]["db"][1]
            chk.add("db", db, dbref, dbmag, tau_sum(M) * dbmag)
    first = {k: v[0] for k, v in outs[0].items()}
    second = {k: v[0] for k, v in outs[1].items()}
    return chk, first, second


def launched_kernels(names):
    """Parse profiler kernel names ('void ns::kern<128, 4, false, true, 1>(ns::P)') into {(base, (args, ...))}."""
    import re
    out = set()
    for n in names:
        m = re.search(r"([A-Za-z_]\w*)(?:<([^<>]*)>)?\(", n)
        if m:
            args = tuple(a.strip() for a in m.group(2).split(",")) if m.group(2) else ()
            out.add((m.group(1), args))
    return out


def fmt_args(args) -> tuple:
    return tuple(str(a).lower() if isinstance(a, bool) else str(a) for a in args)


def missing_kernels(c: Case, names, sm: int, env: Env = DEFAULT_ENV):
    """Expected (base, args) of case c not found among the launched kernel names."""
    got = launched_kernels(names)
    _, want = expected_kernel(c, sm, env)
    return [(b, fmt_args(a)) for b, a in want if (b, fmt_args(a)) not in got]


def profile_case(c: Case, dev="cuda"):
    """run_case under torch.profiler (CUDA activity): (Check, first outputs, second outputs, kernel names)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = run_case(c, dev)
        torch.cuda.synchronize()
    names = sorted({e.name for e in prof.events()})
    return (*res, names)


def result_line(c: Case, chk: Check) -> str:
    return json.dumps({"case": c.name, "op": c.op, "M": c.M, "N": c.N, "K": c.K, "ratio": chk.ratio, "usage": chk.usage})
