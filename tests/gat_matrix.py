"""The GATv2 attention parity matrix: a host-side mirror of the dispatch rules of sgb_gatv2_fwd / sgb_gatv2_bwd /
sgb_gatv2_alpha (segger_b200/csrc/sgb_gatv2.cu `classify`, sgb_gatv2_quad.cu `quad_shape` / `pick_rpw` / `quad_dst_lean`
/ `quad_dst_minb`, ops._quad_path and the `direct` rule of ops.gatv2_bwd), the cases that reach every kernel
instantiation they can pick, a float64 reference of the same operation with per-element error bounds, and a runner.

Shared by tests/test_gpu_gat_matrix.py (every case, default settings), tests/test_gat_matrix_host.py (coverage of the
mirror and negative controls of the checker, no GPU) and tests/gat_env_worker.py (one case per family under each
SEGGER_B200_GAT* switch).

Error bounds (u = 2^-24, every magnitude below is the float64 "twin" of the quantity: the same formula on |values|).
The reference takes the kernel's own fp32 inputs, so z = x_l + x_r has the sign of the kernel's rounded sum and the
LeakyReLU kink needs no allow-list.
  * logit of edge e, head h:   tau(C) * sum_c |att| |lrelu z|                                      =: lerr_e
  * softmax of row i:          rel_i = 2 max_e lerr_e + EXP_C u (max_e |l_e - m_i| + kTau + 1) + DEG_C u (deg_i + 16)
    (the worst logit error moves every weight by twice itself; __expf loses ~u per unit of its argument, and the
    lazy-max forward lets the argument reach kTau = 12 above the true maximum; the sums and rescales lose ~u per edge)
  * out:                       rel_i * sum_e alpha_e k_e |x_l[j]|  +  2u (that sum + |bias|)
  * stat_max + log(stat_den):  2 rel_i + 2u (|lse| + 1) against the row's log-sum-exp
  * alpha (pre-dropout):       alpha_e (lerr_e + 2 rel_i)
  * delta_e = alpha_e (k_e g_i.x_l[j] - c_i),  c_i = g_i.(out_i - bias),  g = grad_out (* GELU'(out) when fused, whose
    fp32 error e_g = 2^-20 |grad_out| (1 + |GELU'|) is absolute: 1 + erf cancels for negative arguments):
                               Ddelta_e = alpha_e (lerr_e + 2 rel_i) (k_e |g.x| + |c_i|) + alpha_e tau(C)
                                          (k_e sum|g||x_l[j]| + sum|g| (|out| + |bias|)) + alpha_e (the same sums of e_g)
  * grad_x_r, grad_x_l:        sum_e Ddelta_e |lrelu'(z)| |att| (+ the alpha' g term for grad_x_l)
                               + tau_sum(degree) * sum_e |each term|
  * grad_att / grad_bias:      sum_e Ddelta_e |lrelu z| + tau_sum(E) sum_e |delta_e lrelu z|;  tau_sum(n_dst) sum_i |g_i|
                               + sum_i e_g
  * every bound also gets FLOOR = 2^-100: fp32 flushes what float64 keeps below 2^-126.
The constants are calibrated on a B200 (profiles/gat_matrix_ratios_b200.json, DESIGN "GATv2 parity matrix").
"""
from __future__ import annotations

import contextlib
import json
import math
from dataclasses import dataclass, field
from typing import Optional

import torch

from tests.gemm_matrix import fmt_args, launched_kernels

SM_COUNT_B200 = 148
U = 2.0 ** -24
KTAU = 12.0
TAU_C = 2.0          # logits: tau(C) = TAU_C (C/8 + 16) u
TAU_SUM_C = 2.0      # ordered sums over edges / rows: tau_sum(n) = TAU_SUM_C (n/64 + 16) u
EXP_C = 8.0
DEG_C = 4.0
EPS_ACT = 2.0 ** -20  # fp32 erf and the roundings of GELU or its derivative
FLOOR = 2.0 ** -100   # added to every bound: fp32 flushes what fp64 keeps below 2^-126 (e^-94 weights, GELU' of -1e3)
SENTINEL = -12345.5
DEN_EMPTY = float(torch.tensor(1e-16, dtype=torch.float32))   # stat_den of a row without edges


def tau(c: int) -> float:
    return TAU_C * (c / 8 + 16) * U


def tau_sum(n):
    return TAU_SUM_C * (n / 64 + 16) * U


def cdiv(a: int, b: int) -> int:
    return -(-a // b)


# ---------------------------------------------------------------------------------------------------------------------
# dispatch mirror
# ---------------------------------------------------------------------------------------------------------------------
QUAD_COMBOS = [(4, 8, 1), (4, 8, 2), (4, 8, 4), (3, 8, 3), (3, 8, 1), (2, 8, 1), (2, 8, 2), (2, 32, 1), (2, 32, 2),
               (4, 32, 1), (4, 32, 2), (4, 32, 4)]                         # SGB_QUAD_COMBOS: (V, LPR, H)
VEC_COMBOS = [(1, 8), (1, 16), (1, 32), (2, 8), (2, 16), (2, 32), (2, 64), (3, 32), (4, 16), (4, 32), (4, 64),
              (4, 128)]                                                     # SGB_VEC_COMBOS: (VEC, CV)
D_FWD, D_DST, D_DST_LEAN, D_SRC = 4, 4, 3, 4


@dataclass(frozen=True)
class Env:
    """The SEGGER_B200_GAT* switches.  RPW and DST_OCC are cached in statics by the library: fresh process only."""
    legacy: bool = False        # SEGGER_B200_GAT=legacy
    rpw: int = 0                # SEGGER_B200_GAT_RPW
    sort: bool = True           # SEGGER_B200_GAT_SORT=0 -> False
    dst_occ: int = 0            # SEGGER_B200_GAT_DST_OCC=3|4
    logits: bool = True         # SEGGER_B200_GAT_LOGITS=0 -> False
    direct: bool = True         # SEGGER_B200_GAT_DIRECT=0 -> False

    def variables(self) -> dict:
        v = {}
        if self.legacy:
            v["SEGGER_B200_GAT"] = "legacy"
        if self.rpw:
            v["SEGGER_B200_GAT_RPW"] = str(self.rpw)
        if not self.sort:
            v["SEGGER_B200_GAT_SORT"] = "0"
        if self.dst_occ:
            v["SEGGER_B200_GAT_DST_OCC"] = str(self.dst_occ)
        if not self.logits:
            v["SEGGER_B200_GAT_LOGITS"] = "0"
        if not self.direct:
            v["SEGGER_B200_GAT_DIRECT"] = "0"
        return v

    @staticmethod
    def from_environ(e) -> "Env":
        occ = e.get("SEGGER_B200_GAT_DST_OCC")
        return Env(legacy=e.get("SEGGER_B200_GAT", "").startswith("l"), rpw=int(e.get("SEGGER_B200_GAT_RPW", "0") or 0),
                   sort=not e.get("SEGGER_B200_GAT_SORT", "").startswith("0"),
                   dst_occ=int(occ) if occ in ("3", "4") else 0,
                   logits=e.get("SEGGER_B200_GAT_LOGITS", "1") != "0", direct=e.get("SEGGER_B200_GAT_DIRECT", "1") != "0")


DEFAULT_ENV = Env()


def quad_shape(H: int, C: int):
    """(V, LPR) of the sub-warp kernels for (H, C), or None."""
    F = H * C
    for lpr in (8, 32):
        if F % (4 * lpr) or C % (4 * lpr):
            continue
        v = F // (4 * lpr)
        if v > 4 or v % H:
            continue
        if (v, lpr, H) in QUAD_COMBOS:
            return v, lpr
    return None


def classify(H: int, C: int, aligned: bool):
    """("vec", VEC, CV) | ("gen", TC) | None (unsupported)."""
    F = H * C
    if aligned and F % 128 == 0 and C % 4 == 0 and (F // 128, C // 4) in VEC_COMBOS:
        return "vec", F // 128, C // 4
    if C <= 256:
        return "gen", (1 if C <= 32 else 2 if C <= 64 else 4 if C <= 128 else 8)
    return None


def pick_rpw(n_rows: int, G: int, sm: int, forced: int = 0) -> int:
    rpw = n_rows // (sm * 16 * 6)
    rpw = max(G, rpw // G * G)
    rpw = min(rpw, 32)
    if G == 1 and rpw > 8:
        rpw = 8
    if forced > 0:
        rpw = min(32, max(G, forced // G * G))
    return rpw


def quad_dst_blocks(n_dst: int, rpw: int, per_sm: int, sm: int) -> int:
    return min(cdiv(cdiv(max(n_dst, 1), rpw), 4), sm * per_sm)


@dataclass(frozen=True)
class Case:
    """One forward (+ backward, + alpha) call of ops.gatv2_fwd / gatv2_bwd / gatv2_alpha."""
    name: str
    H: int
    C: int
    graph: str = "ragged"       # ragged | hub | unique (one source per edge) | scripted | empty
    n_src: int = 300
    n_dst: int = 200
    avg: int = 6                # mean in-degree (ragged / hub / unique)
    slope: float = 0.2
    p: float = 0.0              # dropout (training) probability
    seed_dev: bool = False      # dropout seed partly from a device word (ops.device_seed)
    bias: str = "rand"          # rand | none | big (|bias| ~ 1e3 x the aggregate)
    want_pre: bool = True
    gelu: bool = False          # forward also writes GELU(out); backward fuses GELU'
    layout: str = "plain"       # plain | slice3f (x_l / x_r / outputs: column slices of [N, 3F]) | misaligned
    logits: bool = True         # gatv2_fwd(want_logits=True): saved-logit backward where the sub-warp kernels apply
    inputs: str = "scaled"      # scaled (per-column 2^[-6, 6]) | scripted (x_r = 0, x_l[j] = t_j, att = 1/C)
    backward: bool = True
    alpha: bool = False
    raises: bool = False        # unsupported shape: gatv2_fwd must raise

    def __str__(self):
        return self.name

    @property
    def direct(self) -> bool:
        return self.graph == "unique"


def _aligned(c: Case) -> bool:
    return c.layout != "misaligned"


def quad_path(c: Case, env: Env = DEFAULT_ENV) -> bool:
    """ops._quad_path: the library runs the sub-warp kernels."""
    return _aligned(c) and not env.legacy and 0.0 <= c.slope <= 1.0 and quad_shape(c.H, c.C) is not None


def n_edges(c: Case) -> int:
    return {"empty": 0, "scripted": 8 * c.n_dst}.get(c.graph, -1)


def uses_logits(c: Case, env: Env = DEFAULT_ENV) -> bool:
    """gatv2_fwd asks for e_logit (and gatv2_bwd passes it on)."""
    return c.logits and env.logits and c.graph != "empty" and c.n_dst > 0 and quad_path(c, env)


def uses_direct(c: Case, env: Env = DEFAULT_ENV) -> bool:
    """ops.gatv2_bwd's one-source-per-edge form: src_rowptr = NULL, the dst pass writes grad_x_l."""
    return c.direct and env.direct and c.n_dst > 0 and quad_path(c, env)


def expected_kernels(c: Case, sm: int = SM_COUNT_B200, env: Env = DEFAULT_ENV):
    """{"fwd" | "bwd" | "alpha": [(kernel base name, template arguments)]} launched by case c, in launch order.
    None for a case that must raise."""
    H, C = c.H, c.C
    cls = classify(H, C, _aligned(c))
    if cls is None:
        return None
    out = {}
    if quad_path(c, env):
        v, lpr = quad_shape(H, C)
        out["fwd"] = [("gatv2_fwd_quad_kernel", (v, lpr, H, D_FWD))]
        if c.backward:
            direct = uses_direct(c, env)
            if uses_logits(c, env):
                lean = env.dst_occ == 4 or (env.dst_occ != 3 and not direct)
                dst = (("gatv2_bwd_dst_lg_quad_kernel", (v, lpr, H, D_DST_LEAN, 4, True)) if lean else
                       ("gatv2_bwd_dst_lg_quad_kernel", (v, lpr, H, D_DST, 3, False)))
            else:
                dst = ("gatv2_bwd_dst_quad_kernel", (v, lpr, H, D_DST, 4 if env.dst_occ == 4 else 3))
            out["bwd"] = [dst, ("quad_colsum_kernel", ())]
            if not direct:
                out["bwd"].append(("gatv2_bwd_src_quad_kernel", (v, lpr, H, D_SRC)))
    elif cls[0] == "vec":
        vc = cls[1:]
        out["fwd"] = [("gatv2_fwd_vec_kernel", vc)]
        if c.backward:
            out["bwd"] = [("gatv2_bwd_dst_vec_kernel", vc), ("colsum_partials_kernel", ()), ("gatv2_bwd_src_vec_kernel", vc)]
    else:
        tc = (cls[1],)
        out["fwd"] = [("gatv2_fwd_gen_kernel", tc)]
        if c.backward:
            out["bwd"] = [("gatv2_bwd_dst_gen_kernel", tc), ("colsum_partials_gen_kernel", ()), ("gatv2_bwd_src_gen_kernel", tc)]
    if c.alpha and n_edges(c) != 0:
        out["alpha"] = [("gatv2_alpha_kernel", ())]
    return out


def kernel_set(c: Case, sm: int = SM_COUNT_B200, env: Env = DEFAULT_ENV) -> set:
    ks = expected_kernels(c, sm, env)
    return set() if ks is None else {(b, fmt_args(a)) for v in ks.values() for b, a in v}


def chunking(c: Case, n_dst: int, sm: int = SM_COUNT_B200, env: Env = DEFAULT_ENV):
    """(G, rpw, number of chunks, dst-pass CTAs) of the sub-warp path for n_dst rows."""
    v, lpr = quad_shape(c.H, c.C)
    G = 32 // lpr
    rpw = pick_rpw(n_dst, G, sm, env.rpw)
    lean = uses_logits(c, env) and (env.dst_occ == 4 or (env.dst_occ != 3 and not uses_direct(c, env)))
    nb = quad_dst_blocks(n_dst, rpw, 4 if (lean or env.dst_occ == 4) else 3, sm)
    return G, rpw, cdiv(n_dst, rpw), nb


# ---------------------------------------------------------------------------------------------------------------------
# the matrix
# ---------------------------------------------------------------------------------------------------------------------
def _quad_cases():
    """Every (H, C) of SGB_QUAD_COMBOS x {no saved logits, saved logits (LEAN dst pass), one source per edge with saved
    logits (full dst pass)}, spread over slopes, dropout, bias, GELU and layouts."""
    shapes = [(1, 128), (2, 64), (4, 32), (3, 32), (1, 96), (1, 64), (2, 32), (1, 256), (2, 128), (1, 512), (2, 256),
              (4, 128)]
    slopes = (0.2, 0.0, 1.0)
    cases = []
    for i, (H, C) in enumerate(shapes):
        s = slopes[i % 3]
        tag = f"q{H}x{C}"
        cases += [
            Case(f"{tag}_nolg", H, C, slope=s, logits=False, bias=("none", "rand", "big")[i % 3], gelu=i % 2 == 0,
                 p=(0.0, 0.2, 0.5)[i % 3], seed_dev=i % 4 == 1, alpha=i % 3 == 0),
            Case(f"{tag}_lg", H, C, slope=s, n_src=200, n_dst=200, graph="hub" if i % 4 == 0 else "ragged",
                 layout="slice3f" if i % 2 else "plain", gelu=i % 2 == 1, p=(0.2, 0.0)[i % 2], seed_dev=i % 3 == 0,
                 bias=("rand", "big", "none")[i % 3]),
            Case(f"{tag}_direct_lg", H, C, graph="unique", slope=s, n_src=2000, n_dst=150, gelu=i % 2 == 0,
                 p=(0.0, 0.5)[i % 2], alpha=i % 5 == 0),
        ]
    return cases


# vec combos: 8 reached only when the sub-warp kernels decline the slope, 4 at default settings
_VEC = [((4, 32), 1.5), ((2, 64), -0.1), ((1, 128), 1.5), ((2, 128), -0.1), ((1, 256), 1.5), ((4, 128), -0.1),
        ((2, 256), 1.5), ((1, 512), -0.1), ((8, 32), 0.2), ((4, 64), 0.2), ((3, 128), 0.2), ((8, 64), 0.2)]

CASES = _quad_cases() + [
    Case(f"vec{H}x{C}_s{s}", H, C, slope=s, gelu=i % 2 == 0, p=0.5 if i % 3 == 0 else 0.0, seed_dev=i % 6 == 0,
         bias="none" if i % 4 == 3 else "rand", alpha=i % 4 == 0, graph="hub" if i == 5 else "ragged")
    for i, ((H, C), s) in enumerate(_VEC)
] + [
    # generic kernels: gen<1|2|4|8>, a misaligned quad shape (falls to gen, no logits, no error)
    Case("gen1_5x7", 5, 7, p=0.2, seed_dev=True, alpha=True),
    Case("gen2_2x50", 2, 50, gelu=True, bias="big"),
    Case("gen4_1x100", 1, 100, slope=-0.1, alpha=True),
    Case("gen8_1x200", 1, 200, p=0.5, bias="none"),
    Case("gen4_1x96_slope", 1, 96, slope=1.5),
    Case("gen1_3x32_slope", 3, 32, slope=-0.1, graph="hub"),
    Case("gen2_misaligned_2x64", 2, 64, layout="misaligned", p=0.2),
    Case("gen4_misaligned_4x128", 4, 128, layout="misaligned", gelu=True),
    # unsupported shapes (C > 256 off the vector path) must raise
    Case("unsupported_1x300", 1, 300, raises=True, backward=False),
    Case("unsupported_2x512", 2, 512, raises=True, backward=False),
    Case("unsupported_1x512_misaligned", 1, 512, layout="misaligned", raises=True, backward=False),
    # edges of the sub-warp chunking
    Case("q2x64_big_sorted", 2, 64, n_src=60000, n_dst=120_001, avg=4),                # rpw 8 > G: the sort permutes
    Case("q2x64_persistent", 2, 64, n_src=30000, n_dst=40_003, avg=4, logits=False),   # warps own several chunks
    Case("q2x64_persistent_lg", 2, 64, n_src=30000, n_dst=40_003, avg=4),
    Case("q1x128_ndst3", 1, 128, n_src=50, n_dst=3, avg=20),                             # n_dst < G
    Case("q4x32_ndst_odd", 4, 32, n_src=500, n_dst=1001, logits=False),                  # not a multiple of G
    Case("q2x64_empty", 2, 64, graph="empty", alpha=True),
    Case("vec4x32_empty", 4, 32, graph="empty", slope=1.5),
    Case("gen1_empty", 5, 7, graph="empty"),
    Case("q2x64_direct_nolg", 2, 64, graph="unique", n_src=2000, n_dst=150, logits=False, p=0.2),
    Case("q2x64_direct_slope", 2, 64, graph="unique", n_src=2000, n_dst=150, slope=1.5),  # declines to vec, two-pass
    Case("q2x64_act_only", 2, 64, gelu=True, want_pre=False, backward=False),
    # scripted logits: repeated rescales, a first logit 80 above the rest, all equal, quads that disagree
    Case("q2x64_scripted", 2, 64, graph="scripted", n_dst=64, alpha=True),
    Case("q1x128_scripted_nolg", 1, 128, graph="scripted", n_dst=64, logits=False, p=0.2),
    Case("vec2x64_scripted", 2, 64, graph="scripted", n_dst=64, slope=1.5),
    Case("gen2x50_scripted", 2, 50, graph="scripted", n_dst=64),
]

# one case per family for the switches (tests/gat_env_worker.py)
REDUCED = ["q2x64_lg", "q4x32_nolg", "q2x128_direct_lg", "q2x64_direct_nolg", "q2x64_persistent_lg", "q2x64_scripted",
           "vec4x32_s1.5", "gen1_5x7"]
# SEGGER_B200_GAT=legacy: all 12 vector combos at slope 0.2 (the quad shapes fall to the vector / generic kernels)
LEGACY = [f"q{H}x{C}_nolg" for H, C in [(1, 128), (2, 64), (4, 32), (1, 256), (2, 128), (1, 512), (2, 256), (4, 128)]] + \
    ["vec8x32_s0.2", "vec4x64_s0.2", "vec3x128_s0.2", "vec8x64_s0.2", "q1x64_nolg"]


def case(name: str) -> Case:
    return next(c for c in CASES if c.name == name)


# ---------------------------------------------------------------------------------------------------------------------
# inputs
# ---------------------------------------------------------------------------------------------------------------------
def _seed(name: str) -> int:
    return sum(ord(ch) * (i + 1) for i, ch in enumerate(name))


# scripted logit rows (8 edges each): repeated rescales, first 80 above the rest, all equal, falling
SCRIPTS = [[0.0, 13.0, 26.5, 40.0, 53.5, 67.0, 80.5, 94.0],
           [80.0, 0.0, -1.0, 0.5, 1.0, -2.0, 0.25, 0.0],
           [5.0] * 8,
           [3.0, 2.0, 1.0, 0.0, -1.0, -2.0, -3.0, -4.0]]


def graph(c: Case, g: torch.Generator):
    """(edge_index [2, E] int64, n_src, n_dst, t) on the host; t = scripted logit per source (scripted graphs)."""
    n_src, n_dst = c.n_src, c.n_dst
    t = None
    if c.graph == "empty":
        return torch.zeros(2, 0, dtype=torch.long), n_src, n_dst, t
    if c.graph == "scripted":
        E = 8 * n_dst
        t = torch.tensor([SCRIPTS[(i // 1) % 4][k] for i in range(n_dst) for k in range(8)], dtype=torch.float64)
        return torch.stack([torch.arange(E), torch.arange(E) // 8]), E, n_dst, t
    if c.graph == "unique":
        E = min(n_src, n_dst * c.avg)
        src = torch.sort(torch.randperm(n_src, generator=g)[:E]).values
        dst = torch.randint(0, n_dst, (E,), generator=g)
        return torch.stack([src, dst]), n_src, n_dst, t
    deg = torch.randint(0, 2 * c.avg + 1, (n_dst,), generator=g)
    deg[torch.randperm(n_dst, generator=g)[: max(1, n_dst // 10)]] = 0    # isolated destinations
    if n_dst > 2:
        deg[1] = 1
        deg[2] = max(int(deg[2]), 2)
    if c.graph == "hub":
        deg[n_dst // 2] = 2500
    dst = torch.repeat_interleave(torch.arange(n_dst), deg)
    used = max(1, n_src - n_src // 10)                                     # the last tenth of the sources: no out-edge
    src = torch.randint(0, used, (dst.numel(),), generator=g)
    perm = torch.randperm(dst.numel(), generator=g)                        # edge ids != CSR positions
    return torch.stack([src[perm], dst[perm]]), n_src, n_dst, t


@dataclass
class Inputs:
    x_l: torch.Tensor
    x_r: torch.Tensor
    att: torch.Tensor
    bias: Optional[torch.Tensor]
    grad_out: torch.Tensor
    rowptr: torch.Tensor
    col: torch.Tensor
    eid: torch.Tensor
    keep: Optional[torch.Tensor]      # [E, H] keep mask in original edge order (training), else None
    H: int
    C: int
    slope: float
    p: float


def host_inputs(c: Case, dev="cpu"):
    """Seeded inputs as plain contiguous fp32 tensors, and the dst-CSR arrays (as build_csr makes them)."""
    g = torch.Generator().manual_seed(_seed(c.name))
    ei, n_src, n_dst, t = graph(c, g)
    H, C, F = c.H, c.C, c.H * c.C
    n_l = ei.size(1) if c.direct else n_src
    if c.inputs == "scripted" or c.graph == "scripted":
        x_l = t[:, None].float().expand(n_l, F).contiguous()
        x_r = torch.zeros(n_dst, F)
        att = torch.full((H, C), 1.0 / C)
        cs = torch.ones(F)
    else:
        cs = torch.pow(2.0, torch.randint(-6, 7, (F,), generator=g).double()).float()
        x_l = torch.randn(n_l, F, generator=g) * cs
        x_r = torch.randn(n_dst, F, generator=g) * cs
        att = (torch.randn(F, generator=g) * (2.0 / math.sqrt(C)) / cs).view(H, C)
    bias = None
    if c.bias == "rand":
        bias = torch.randn(F, generator=g) * cs * 0.5
    elif c.bias == "big":
        bias = torch.randn(F, generator=g) * cs * 1000.0
    rs = torch.pow(2.0, torch.randint(-4, 5, (n_dst,), generator=g).double()).float()
    grad_out = torch.randn(n_dst, F, generator=g) * rs[:, None]
    # dst-CSR (stable by destination), and for the one-source-per-edge form col = edge id
    src, dst = ei[0], ei[1]
    order = torch.argsort(dst, stable=True)
    rowptr = torch.zeros(n_dst + 1, dtype=torch.long)
    rowptr[1:] = torch.bincount(dst, minlength=n_dst).cumsum(0)
    col = order.clone() if c.direct else src[order]
    return ei, n_src, n_dst, x_l.to(dev), x_r.to(dev), att.to(dev), (bias.to(dev) if bias is not None else None), \
        grad_out.to(dev), rowptr.to(dev), col.to(dev), order.to(dev)


# ---------------------------------------------------------------------------------------------------------------------
# float64 reference with per-element bounds
# ---------------------------------------------------------------------------------------------------------------------
def _seg_max(vals, row, n):
    out = torch.full((n,) + vals.shape[1:], -math.inf, dtype=vals.dtype, device=vals.device)
    return out.scatter_reduce(0, row.view(-1, *([1] * (vals.dim() - 1))).expand_as(vals), vals, "amax")


def _add(idx, vals, n):
    return torch.zeros((n,) + vals.shape[1:], dtype=vals.dtype, device=vals.device).index_add_(0, idx, vals)


def _gelu_grad(v):
    cdf = 0.5 * (1 + torch.erf(v / math.sqrt(2)))
    return cdf + v * torch.exp(-0.5 * v * v) / math.sqrt(2 * math.pi)


def reference(inp: Inputs, out32=None, gelu=False, bug=None):
    """float64 reference of forward, backward and alpha from the fp32 inputs, with bounds.  ``out32``: the forward
    output the backward is given (the kernel's; the reference's own rounded to fp32 when None).  ``bug`` injects one
    plausible kernel mistake (negative controls): drop_edge | att_head | kink | cta_partial | row_scale.
    -> (values, bounds), dicts keyed like the kernel outputs."""
    H, C, s = inp.H, inp.C, inp.slope
    rowptr, col, eid = inp.rowptr.long(), inp.col.long(), inp.eid.long()
    n_dst = rowptr.numel() - 1
    n_src = inp.x_l.size(0)
    deg = rowptr[1:] - rowptr[:-1]
    row = torch.repeat_interleave(torch.arange(n_dst, device=rowptr.device), deg)
    E = row.numel()
    xl = inp.x_l.double().reshape(n_src, H, C)
    xr = inp.x_r.double().reshape(n_dst, H, C)
    at = inp.att.double().reshape(H, C)
    b = inp.bias.double().reshape(H, C) if inp.bias is not None else torch.zeros(H, C, dtype=torch.float64, device=xl.device)
    ks = torch.ones(E, H, dtype=torch.float64, device=xl.device)
    if inp.keep is not None:
        ks = inp.keep[eid].double() / (1.0 - inp.p)
    live = torch.ones(E, dtype=torch.float64, device=xl.device)
    if bug == "drop_edge":                                # the second edge of the first row with degree >= 2
        i0 = int(torch.nonzero(deg >= 2)[0])
        live[int(rowptr[i0]) + 1] = 0.0
    at_used = at.roll(1, 0) if bug == "att_head" else at

    z = xl[col] + xr[row]
    pos = (z >= 0) if bug == "kink" else (z > 0)
    sel = torch.where(pos, torch.ones_like(z), torch.full_like(z, s))
    lz = torch.where(z > 0, z, s * z)
    lg = (at_used * lz).sum(-1)
    lmag = (at.abs() * lz.abs()).sum(-1)
    lerr = tau(C) * lmag
    lg_m = torch.where(live[:, None] > 0, lg, torch.full_like(lg, -math.inf))
    m = _seg_max(lg_m, row, n_dst)
    mrow = torch.where(torch.isfinite(m), m, torch.zeros_like(m))
    ex = torch.exp(lg_m - mrow[row])
    den = _add(row, ex, n_dst)
    alpha = ex / torch.where(den > 0, den, torch.ones_like(den))[row]
    lse = mrow + torch.log(torch.where(den > 0, den, torch.ones_like(den)))
    w = alpha * ks
    outv = _add(row, w[..., None] * xl[col], n_dst) + b
    if bug == "row_scale":
        i0 = int(torch.nonzero(deg >= 1)[0])
        outv[i0] = (outv[i0] - b) * (1 + 2.0 ** -12) + b
    outmag = _add(row, w[..., None] * xl[col].abs(), n_dst)

    dlm = _seg_max(torch.where(live[:, None] > 0, mrow[row] - lg, torch.zeros_like(lg)), row, n_dst)
    dlm = torch.where(torch.isfinite(dlm), dlm, torch.zeros_like(dlm))
    lerr_row = _seg_max(lerr, row, n_dst)
    lerr_row = torch.where(torch.isfinite(lerr_row), lerr_row, torch.zeros_like(lerr_row))
    rel = 2 * lerr_row + EXP_C * U * (dlm + KTAU + 1) + DEG_C * U * (deg[:, None].double() + 16)
    vals = {"out": outv.reshape(n_dst, H * C), "e_logit": lg, "lse": lse, "alpha": alpha}
    bounds = {"out": (rel[..., None] * outmag + 2 * U * (outmag + b.abs())).reshape(n_dst, H * C), "e_logit": lerr,
              "lse": 2 * rel + 2 * U * (lse.abs() + 1), "alpha": alpha * (lerr + 2 * rel[row])}
    if gelu:
        o = vals["out"]
        vals["out_act"] = torch.nn.functional.gelu(o)
        bounds["out_act"] = _gelu_grad(o).abs() * bounds["out"] + EPS_ACT * (vals["out_act"].abs() + o.abs())

    # backward, given out32 (what the kernel's backward reads)
    if out32 is None:
        out32 = vals["out"].float()
    ob = out32.double().reshape(n_dst, H, C)
    g = inp.grad_out.double().reshape(n_dst, H, C)
    ge = torch.zeros_like(g)            # error of the fp32 g = grad_out * GELU'(out): absolute, 1 + erf cancels
    if gelu:
        gp = _gelu_grad(ob)
        ge = EPS_ACT * g.abs() * (1 + gp.abs())
        g = g * gp
    c_i = (g * (ob - b)).sum(-1)
    cmag = (g.abs() * (ob.abs() + b.abs())).sum(-1)
    d_e = (g[row] * xl[col]).sum(-1)
    dmag = (g[row].abs() * xl[col].abs()).sum(-1)
    delta = alpha * (ks * d_e - c_i[row])
    relA = lerr + 2 * rel[row]
    Dm = alpha * relA * (ks * d_e.abs() + c_i[row].abs()) + alpha * tau(C) * (ks * dmag + cmag[row]) + alpha * (
        ks * (ge[row] * xl[col].abs()).sum(-1) + (ge * (ob.abs() + b.abs())).sum(-1)[row])
    dz = delta[..., None] * sel * at
    dz_b = Dm[..., None] * sel.abs() * at.abs()
    ag = w[..., None] * g[row]
    ag_b = (w * (relA + 2 * U))[..., None] * g[row].abs() + w[..., None] * ge[row]
    outdeg = torch.bincount(col, minlength=n_src)
    gxr = _add(row, dz, n_dst)
    gxl = _add(col, dz + ag, n_src)
    gatt_terms = delta[..., None] * lz
    if bug == "cta_partial":                             # the rows of one 4-warp CTA chunk left out of grad_att
        r0 = n_dst // 3
        keep_rows = ~((row >= r0) & (row < r0 + 16))
        gatt = (gatt_terms * keep_rows[:, None, None]).sum(0)
    else:
        gatt = gatt_terms.sum(0)
    vals.update({
        "grad_x_r": gxr.reshape(n_dst, H * C), "grad_x_l": gxl.reshape(n_src, H * C),
        "grad_att": gatt.reshape(H * C), "grad_bias": g.sum(0).reshape(H * C)})
    bounds.update({
        "grad_x_r": (_add(row, dz_b, n_dst) + tau_sum(deg.double())[:, None, None] * _add(row, dz.abs(), n_dst)).reshape(n_dst, H * C),
        "grad_x_l": (_add(col, dz_b + ag_b, n_src)
                     + tau_sum(outdeg.double())[:, None, None] * _add(col, dz.abs() + ag.abs(), n_src)).reshape(n_src, H * C),
        "grad_att": ((Dm[..., None] * lz.abs()).sum(0) + tau_sum(E) * gatt_terms.abs().sum(0)).reshape(H * C),
        "grad_bias": (tau_sum(n_dst) * g.abs().sum(0) + ge.sum(0)).reshape(H * C)})
    bounds = {k: v + FLOOR for k, v in bounds.items()}
    vals["_deg"] = deg
    vals["_m"] = mrow
    vals["_den"] = torch.where(den > 0, den, torch.full_like(den, DEN_EMPTY))
    vals["_outdeg"] = outdeg
    vals["_eid"] = eid
    return vals, bounds


def emulate(vals: dict) -> dict:
    """The reference's values rounded to fp32 and laid out like the kernels' outputs (for the negative controls)."""
    got = {k: vals[k].float() for k in ("out", "e_logit", "grad_x_r", "grad_x_l", "grad_att", "grad_bias")}
    got["stat_max"], got["stat_den"] = vals["_m"].float(), vals["_den"].float()
    a = torch.empty_like(vals["alpha"])
    a[vals["_eid"]] = vals["alpha"]
    got["alpha"] = a.float()
    return got


# ---------------------------------------------------------------------------------------------------------------------
# checker
# ---------------------------------------------------------------------------------------------------------------------
@dataclass
class Check:
    usage: dict = field(default_factory=dict)      # worst err / bound per output
    failures: list = field(default_factory=list)

    def add(self, what, got, ref, bound):
        got = got.double()
        err = (got - ref).abs()
        bad = ~(err <= bound)                       # NaN and the sentinel fail too
        pos = bound > 0
        self.usage[what] = max(self.usage.get(what, 0.0), float((err[pos] / bound[pos]).max()) if bool(pos.any()) else 0.0)
        if bool(bad.any()):
            i = int(bad.flatten().nonzero()[0])
            self.failures.append(f"{what}: {int(bad.sum())} of {bad.numel()} elements out of bound; first flat index {i}: "
                                 f"got {got.flatten()[i].item()!r} ref {ref.flatten()[i].item()!r} "
                                 f"bound {bound.flatten()[i].item():.3e}")

    def exact(self, what, ok: bool):
        if not ok:
            self.failures.append(what)


def check_outputs(got: dict, vals: dict, bounds: dict, bias, chk: Optional[Check] = None) -> Check:
    """Every output of `got` (the kernel's) against the reference: per-element bounds, plus the exact rules for rows
    without edges (out == bias, stat_max == 0, stat_den == 1e-16, gradients exactly 0)."""
    chk = chk or Check()
    deg, outdeg = vals["_deg"], vals["_outdeg"]
    iso = deg == 0
    for k in ("out", "out_act", "e_logit", "grad_x_r", "grad_x_l", "grad_att", "grad_bias"):
        if got.get(k) is not None:
            chk.add(k, got[k], vals[k], bounds[k])
    if got.get("stat_max") is not None:
        sm, sd = got["stat_max"].double(), got["stat_den"].double()
        has = ~iso
        lse = sm + torch.log(sd.clamp_min(1e-300))
        chk.add("lse", lse[has], vals["lse"][has], bounds["lse"][has])
        chk.exact("stat of rows without edges", bool((got["stat_max"][iso] == 0).all()) and
                  bool((got["stat_den"][iso] == DEN_EMPTY).all()))
    if got.get("alpha") is not None:
        a = torch.empty_like(vals["alpha"])
        a[vals["_eid"]] = vals["alpha"]
        ab = torch.empty_like(bounds["alpha"])
        ab[vals["_eid"]] = bounds["alpha"]
        chk.add("alpha", got["alpha"], a, ab)
    if got.get("out") is not None and bool(iso.any()):
        F = got["out"].size(1)
        b = bias.reshape(1, F) if bias is not None else torch.zeros(1, F, device=got["out"].device)
        chk.exact("out of rows without edges != bias", bool((got["out"][iso] == b).all()))
    if got.get("grad_x_r") is not None:
        chk.exact("grad_x_r of rows without edges != 0", bool((got["grad_x_r"][iso] == 0).all()))
    if got.get("grad_x_l") is not None:
        chk.exact("grad_x_l of sources without out-edges != 0", bool((got["grad_x_l"][outdeg == 0] == 0).all()))
    return chk


def untouched(chk: Check, what, buf, view):
    """Everything of buf outside view still holds the sentinel."""
    mask = torch.ones_like(buf, dtype=torch.bool)
    mask.as_strided(view.shape, view.stride(), view.storage_offset() - buf.storage_offset()).fill_(False)
    if not bool((buf[mask] == SENTINEL).all()):
        chk.failures.append(f"{what}: the call wrote outside the output view")


@contextlib.contextmanager
def sentinel_alloc():
    """Inside the block every float tensor torch.empty returns holds SENTINEL and every byte buffer 0xff (NaN as
    floats): an output element the kernels forget to write, or workspace they read before writing, shows."""
    real = torch.empty

    def empty(*a, **k):
        t = real(*a, **k)
        if t.is_floating_point():
            t.fill_(SENTINEL)
        elif t.dtype == torch.uint8:
            t.fill_(255)
        return t

    torch.empty = empty
    try:
        yield
    finally:
        torch.empty = real


# ---------------------------------------------------------------------------------------------------------------------
# runner
# ---------------------------------------------------------------------------------------------------------------------
def _view(x, layout, width_mult=3, col=0):
    """A copy of x as plain, as the column slice `col` of an [N, 3F] buffer, or at a 4-byte offset with ld % 4 == 3."""
    n, F = x.shape
    if layout == "slice3f":
        buf = torch.zeros(n, width_mult * F, device=x.device)
        v = buf[:, col * F:(col + 1) * F]
    elif layout == "misaligned":
        buf = torch.zeros(n, F + 3, device=x.device)
        v = buf[:, 1:F + 1]
    else:
        v = torch.empty_like(x)
    v.copy_(x)
    return v


def run_case(c: Case, dev="cuda", env: Env = DEFAULT_ENV):
    """Runs c twice under the switches env describes.  -> (Check, outputs of the first call, outputs of the second)."""
    from segger_b200 import ops

    ei, n_src, n_dst, x_l, x_r, att, bias, grad_out, rowptr, col, eid = host_inputs(c, dev)
    H, C, F = c.H, c.C, c.H * c.C
    csr = ops.build_csr(ei.to(dev), n_src, n_dst)
    if c.direct:
        assert csr.sources_unique_increasing()
        csr = csr.per_edge_sources()
    assert torch.equal(csr.rowptr.long(), rowptr) and torch.equal(csr.col.long(), col) and torch.equal(csr.eid.long(), eid)
    if c.layout == "slice3f":
        assert x_l.size(0) == x_r.size(0)
        y = torch.zeros(x_l.size(0), 3 * F, device=dev)
        y[:, :F], y[:, F:2 * F] = x_l, x_r
        xl_v, xr_v = y[:, :F], y[:, F:2 * F]
    else:
        xl_v, xr_v = _view(x_l, c.layout), _view(x_r, c.layout)
    training = c.p > 0
    seed = 0
    word = None
    if training:
        seed = 0x1234567 + _seed(c.name)
        if c.seed_dev:
            word = torch.tensor([0x5DEECE66D + _seed(c.name)], dtype=torch.int64, device=dev)
            seed = (seed, word)
    keep = ops.dropout_keep_mask(seed, csr.E, H, c.p, dev) if training else None
    inp = Inputs(x_l, x_r, att, bias, grad_out, rowptr, col, eid, keep, H, C, c.slope, c.p)
    chk = Check()

    def call():
        res, views = {}, {}
        with sentinel_alloc():
            out = None
            if c.layout == "slice3f" and c.want_pre:
                obuf = torch.empty(n_dst, 2 * F, device=dev)
                out = obuf[:, F:]
                views["out"] = (obuf, out)
            r = ops.gatv2_fwd(xl_v, xr_v, att, bias, csr, H, C, c.slope, c.p, training, seed, c.gelu, out=out,
                              want_pre=c.want_pre, want_logits=True if c.logits else None)
            res["out"], res["out_act"], res["stat_max"], res["stat_den"], res["e_logit"] = r
            if c.backward:
                gl = gr = None
                if c.layout == "slice3f":
                    G = torch.empty(x_l.size(0), 3 * F, device=dev)
                    gl, gr = G[:, :F], G[:, F:2 * F]
                    views["grad"] = (G, G[:, :2 * F])
                gl, gr, ga, gb = ops.gatv2_bwd(xl_v, xr_v, att, bias, res["out"], grad_out, c.gelu, csr, H, C, c.slope,
                                               c.p, training, seed, res["stat_max"], res["stat_den"], grad_x_l=gl,
                                               grad_x_r=gr, e_logit=res["e_logit"])
                res.update(grad_x_l=gl, grad_x_r=gr, grad_att=ga, grad_bias=gb)
            if c.alpha:
                res["alpha"] = ops.gatv2_alpha(xl_v, xr_v, att, csr, H, C, c.slope, res["stat_max"], res["stat_den"])
        torch.cuda.synchronize()
        return {k: (v.clone() if v is not None else None) for k, v in res.items()}, views

    first, views = call()
    second, _ = call()
    vals, bounds = reference(inp, first["out"] if first["out"] is not None else None, c.gelu)
    if uses_logits(c, env):
        chk.exact("e_logit missing on the sub-warp path", first["e_logit"] is not None)
    else:
        chk.exact("e_logit offered outside the sub-warp path", first["e_logit"] is None)
    if not c.want_pre:
        chk.exact("want_pre=False returned out", first["out"] is None)
    check_outputs(first, vals, bounds, bias, chk)
    for k, (buf, v) in views.items():
        untouched(chk, k, buf, v)
    for k in first:
        if first[k] is not None and not torch.equal(first[k], second[k]):
            chk.failures.append(f"{k}: two identical calls differ")
    return chk, first, second


def gat_names(names):
    """The GATv2 kernels among profiler kernel names."""
    return {k for k in launched_kernels(names) if k[0].startswith("gatv2_") or "colsum" in k[0]}


def profile_case(c: Case, dev="cuda", env: Env = DEFAULT_ENV):
    """run_case under torch.profiler (CUDA activity): (Check, kernel names)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        chk, _, _ = run_case(c, dev, env)
        torch.cuda.synchronize()
    names = sorted({e.name for e in prof.events()})
    return chk, names


def dispatch_failures(c: Case, names, sm: int, env: Env = DEFAULT_ENV):
    """The GATv2 kernels launched must be exactly those the mirror predicts."""
    want = kernel_set(c, sm, env)
    got = gat_names(names)
    return [] if got == want else [f"expected {sorted(want)}, launched {sorted(got)}"]


def run_raises(c: Case, dev="cuda"):
    """An unsupported shape: gatv2_fwd raises and names the shape."""
    from segger_b200 import ops
    ei, n_src, n_dst, x_l, x_r, att, bias, *_ = host_inputs(c, dev)
    csr = ops.build_csr(ei.to(dev), n_src, n_dst)
    xl_v, xr_v = _view(x_l, c.layout), _view(x_r, c.layout)
    try:
        ops.gatv2_fwd(xl_v, xr_v, att, bias, csr, c.H, c.C, c.slope, 0.0, False, 0, False)
    except Exception as e:          # noqa: BLE001
        return f"H={c.H} C={c.C}" in str(e)
    return False


def result_line(c: Case, chk: Check) -> str:
    return json.dumps({"case": c.name, "H": c.H, "C": c.C, "usage": chk.usage})

