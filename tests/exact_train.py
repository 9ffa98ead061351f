"""Inputs, references and error bounds for the training-time scorer tests (tests/test_gpu_train_exact.py and the
CPU premise test tests/test_train_exact_cpu.py).

Field components (csrc/train.cu: ``field_components_fwd/bwd_docs/bwd_q``) are tested on inputs where fp32 is EXACT
in any summation order: query and doc coordinates are integers in [-3, 3], the upstream gradient G holds integers in
[-2, 2] and the temperature is a power of two.  Every product and every partial sum is then a multiple of 1/T with a
magnitude below 2^24, so the forward, ``ddocs`` and the fp32-atomic ``dq`` all have one correct answer: the float64
contraction cast to fp32 (for bf16 / f16 inputs, cast once more to that dtype, as the autograd Function returns
``.to(dtype)``).  G has whole zero query lanes and whole zero (doc, field) columns next to nonzero ones, so the
``cb == 0`` skip of ``bwd_docs`` runs beside queries it must not skip.

The field mixture (``mixture_weights/apply`` in csrc/aux_kernels.cu, ``mixture_bwd`` in csrc/train.cu) involves expf
and a division, so it is compared with float64 under the per-element bound of ``mixture_bounds``.
"""
from __future__ import annotations

import math
from typing import Dict, List, NamedTuple, Optional

import torch

U = 2.0 ** -24                          # fp32 unit roundoff
EXP_ULP = 4                             # expf (CUDA: 2 ulp) and a vectorised CPU exp, with room
DIV_ULP = 2                             # one division, or a reciprocal and a multiply
TINY = 2.0 ** -125                      # absolute error of a weight that under-flows (with or without flush-to-zero)


def gamma(n: int) -> float:
    """gamma_n = n u / (1 - n u): the relative bound of a sum of n products in fp32, in any order."""
    return n * U / (1 - n * U)


# ---------------------------------------------------------------------------------------------------------------------
# Field components: exact-arithmetic cases
# ---------------------------------------------------------------------------------------------------------------------

class Case(NamedTuple):
    B: int                  # queries (kTrQTile = 32 per tile)
    E: int                  # embedding size (128-float chunks + a (E % 128) / 4-lane tail, E <= 1024)
    F: int                  # fields (<= MFAR_MAX_FIELDS = 64)
    P: int                  # docs [P,F,E], or P groups of Neg docs [P,F,Neg,E]
    Neg: Optional[int]      # None: [N,F,E] layout; else [P,F,Neg,E] with doc n = p*Neg + s
    grads: str              # "q", "d" or "both"
    dtype: str              # "f32", "bf16", "f16"
    T: float                # temperature, a power of two

    @property
    def N(self) -> int:
        return self.P * (self.Neg or 1)

    @property
    def rows(self) -> int:
        return self.N * self.F


DTYPES = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}

# Axis values and why (each appears at least once, next to non-trivial values of the other axes):
#   B      1, 31, 32, 33, 64, 65, 192          query tile of 32: lane == query, partial last tile, several tiles
#   E      4, 124, 128, 132, 512, 764, 768, 1020, 1024
#                                               tail only, 31-lane tail, exact chunks, chunk + 1-lane tail, 8 chunks
#   F      1, 2, 3, 22, 44, 63, 64            up to MFAR_MAX_FIELDS
#   layout [N,F,E]; [P,F,Neg,E] with Neg in 1, 2, 3, 5
#   rows   N*F in 1, 15, 16, 17, 4736 (= 296*16), 4737, >= 50000
#                                               bwd_q slicing: below one 16-row stage, exactly 2*148 slices, one more
#                                               row, many rows per CTA
#   grads  q, d, both                           dq / ddocs null paths of mfar_field_components_bwd
#   dtype  f32; bf16 and f16                    .float() in, .to(dtype) out
#   T      1, 0.5, 0.125
_BS = (1, 31, 32, 33, 64, 65, 192)
_ES = (4, 124, 128, 132, 512, 764, 768, 1020, 1024)
_FS = (1, 2, 3, 22, 44, 63, 64)
_NEGS = (None, 1, 2, 3, 5)
_PS = (1, 2, 5, 9)
_GRADS = ("both", "q", "d")
_TS = (1.0, 0.5, 0.125)

# the N*F row counts of bwd_q's slicing, each with a non-trivial B / E / layout
ROW_CASES: List[Case] = [
    Case(1, 768, 1, 1, None, "d", "f32", 0.125),           # rows 1
    Case(33, 132, 1, 1, 1, "both", "f32", 0.5),            # rows 1, two query tiles
    Case(65, 764, 3, 5, None, "both", "f32", 0.125),       # rows 15
    Case(31, 124, 1, 5, 3, "both", "f32", 0.5),            # rows 15, Neg 3
    Case(33, 132, 2, 4, 2, "both", "f32", 0.5),            # rows 16
    Case(64, 1020, 1, 17, None, "both", "f32", 1.0),       # rows 17
    Case(32, 512, 1, 17, 1, "q", "f32", 0.125),            # rows 17
    Case(192, 768, 64, 37, 2, "both", "f32", 0.125),       # rows 4736 = 296*16
    Case(33, 1024, 2, 2368, None, "q", "f32", 0.5),        # rows 4736, max E
    Case(65, 132, 3, 1579, None, "both", "f32", 1.0),      # rows 4737
    Case(31, 1020, 3, 1579, 1, "q", "f32", 0.125),         # rows 4737, 31-lane tail
    Case(33, 132, 44, 1137, None, "both", "f32", 0.5),     # rows 50028
    Case(65, 128, 22, 455, 5, "both", "f32", 0.125),       # rows 50050, Neg 5
]

# a cyclic cover of B x E x F x layout x grads x T on small doc counts (the moduli 7, 9, 7, 5, 3, 3 interleave)
CYCLE_CASES: List[Case] = [
    Case(_BS[i % 7], _ES[i % 9], _FS[(3 * i + i // 7) % 7], _PS[i % 4], _NEGS[i % 5], _GRADS[(i // 9) % 3],
         "f32", _TS[(i // 7) % 3])
    for i in range(63)
]

DTYPE_CASES: List[Case] = [
    Case(33, 132, 3, 5, 2, "both", "bf16", 0.5),
    Case(65, 768, 22, 3, None, "q", "bf16", 0.125),
    Case(31, 1024, 2, 4, 3, "both", "f16", 1.0),
    Case(64, 4, 64, 2, None, "d", "f16", 0.125),
]

COMPONENT_CASES: List[Case] = ROW_CASES + CYCLE_CASES + DTYPE_CASES


def case_id(c: Case) -> str:
    lay = "NFE" if c.Neg is None else f"Neg{c.Neg}"
    return f"B{c.B}_E{c.E}_F{c.F}_P{c.P}_{lay}_{c.grads}_{c.dtype}_T{c.T:g}"


def component_inputs(c: Case, device="cpu"):
    """q [B,E], docs [P,F,E] or [P,F,Neg,E] (integers in [-3,3]) and G [B,N,F] (integers in [-2,2] with zero query
    lanes and zero (doc, field) columns), all float64, seeded by the case."""
    g = torch.Generator().manual_seed(_seed(c))
    q = torch.randint(-3, 4, (c.B, c.E), generator=g).double()
    shape = (c.P, c.F, c.E) if c.Neg is None else (c.P, c.F, c.Neg, c.E)
    docs = torch.randint(-3, 4, shape, generator=g).double()
    G = torch.randint(-2, 3, (c.B, c.N, c.F), generator=g).double()
    G[torch.arange(c.B) % 7 == 3] = 0                                       # whole zero query lanes
    G.view(c.B, c.rows)[:, torch.arange(c.rows) % 5 == 2] = 0               # whole zero (doc, field) columns
    return q.to(device), docs.to(device), G.to(device)


def _seed(c: Case) -> int:
    return (c.B * 1000003 + c.E * 10007 + c.F * 101 + c.P * 13 + (c.Neg or 0)) % (2 ** 31)


def docs_as_nfe(docs: torch.Tensor) -> torch.Tensor:
    """[N,F,E] view of either layout, doc n = p*Neg + s (losses.py:186)."""
    if docs.dim() == 3:
        return docs
    P, F, Neg, E = docs.shape
    return docs.permute(0, 2, 1, 3).reshape(P * Neg, F, E)


def components_reference(q, docs, G, T):
    """float64 comp [B,N,F], dq [B,E] and ddocs (docs' layout) of comp = <q, doc> / T with upstream gradient G."""
    d = docs_as_nfe(docs)
    comp = torch.einsum("be,nfe->bnf", q, d) / T
    dq = torch.einsum("bnf,nfe->be", G, d) / T
    dd = torch.einsum("bnf,be->nfe", G, q) / T
    if docs.dim() == 4:
        P, F, Neg, E = docs.shape
        dd = dd.reshape(P, Neg, F, E).permute(0, 2, 1, 3).contiguous()
    return comp, dq, dd


def components_magnitudes(q, docs, G, T):
    """Sum of |terms| of every output element of ``components_reference``: a bound on every partial sum."""
    return components_reference(q.abs(), docs.abs(), G.abs(), T)


# ---------------------------------------------------------------------------------------------------------------------
# Field mixture: float64 reference and per-element fp32 error bounds
# ---------------------------------------------------------------------------------------------------------------------

def mixture_reference(x, q, W, query_cond: bool, g) -> Dict[str, torch.Tensor]:
    """float64 forward and backward of out[b,s] = sum_f softmax(logits)[b,f] x[b,s,f] with upstream gradient g[b,s].
    logits = q @ W ([B,F]) when query_cond, else W^T ([1,F], one row for every b, as the kernels use it)."""
    x, W, g = x.double(), W.double(), g.double()
    q = q.double() if query_cond else None
    logits = q @ W if query_cond else W.t()
    w = torch.softmax(logits, dim=1)
    out = (w[:, None, :] * x).sum(-1)
    dwt = torch.einsum("bs,bsf->bf", g, x)
    dlogit = w * (dwt - (w * dwt).sum(1, keepdim=True))
    r = {"logits": logits, "w": w, "out": out, "dx": g[:, :, None] * w[:, None, :], "dwt": dwt, "dlogit": dlogit}
    if query_cond:
        r["dW"], r["dq"] = q.t() @ dlogit, dlogit @ W.t()
    else:
        r["dW"] = dlogit.sum(0)[:, None]
    return r


def mixture_bounds(x, q, W, query_cond: bool, g) -> Dict[str, torch.Tensor]:
    """Per-element bounds on |fp32 - exact| of every value of ``mixture_reference``, from standard fp32 error analysis
    (u = 2^-24, gamma_n = n u / (1 - n u); inputs x, q, W, g are fp32 values, so they carry no error).

    forward
      logit  l_bf = sum_e q_be W_ef                |dl| <= gamma_E sum_e |q_be W_ef|          (0 without query_cond)
      weight w_f = exp(l_f - m) / sum_g exp(l_g - m)
             the exp argument is off by  a_f = dl_f + max_g dl_g + u |l_f - m|  (the subtraction's rounding), so
             e_f has relative error  r_f = (1 + expm1(a_f)) (1 + EXP_ULP u) - 1;  the sum of F positive terms
             rs = (1 + max_f r_f) (1 + gamma_F) - 1;  the division  rho_f = (1 + r_f)(1 + DIV_ULP u) / (1 - rs) - 1
             |dw_f| <= rho_f w_f + TINY      (TINY: a weight that under-flows)
      out    out_bs = sum_f w_f x_bsf            |dout| <= sum_f |x| dw_f + gamma_F sum_f (w_f + dw_f) |x|
    backward (csrc/train.cu mixture_bwd_kernel / mixture_bwd_params_kernel, and the same formulas in autograd)
      dx     g_bs w_f: one rounding of the computed weight (checked bit for bit elsewhere)
      dwt_f  = sum_s g_bs x_bsf                  e_dwt = gamma_S sum_s |g x|
      dot    = sum_f w_f dwt_f                   e_dot = sum_f [dw_f (|dwt_f| + e_dwt_f) + w_f e_dwt_f]
                                                         + gamma_F sum_f (w_f + dw_f)(|dwt_f| + e_dwt_f)
      diff_f = dwt_f - dot                       e_diff = (e_dwt_f + e_dot)(1 + u) + u |diff_f|
      dlogit = w_f diff_f                        e_dl = dw_f (|diff| + e_diff) + w_f e_diff + u (w + dw)(|diff| + e_diff)
      dW     sum_b q_be dlogit_bf                |q|^T e_dl + gamma_B |q|^T (|dlogit| + e_dl)
             (no query_cond: sum_b dlogit_bf     sum_b e_dl + gamma_B sum_b (|dlogit| + e_dl))
      dq     sum_f dlogit_bf W_ef                e_dl |W|^T + gamma_F (|dlogit| + e_dl) |W|^T
    Every bound is a worst case over summation orders, so it holds for the CUDA kernels and for torch CPU fp32 alike
    (tests/test_train_exact_cpu.py checks the latter)."""
    r = mixture_reference(x, q, W, query_cond, g)
    x, W, g = x.double(), W.double(), g.double()
    B, S, F = x.shape
    if query_cond:
        qd = q.double()
        dl = gamma(qd.shape[1]) * (qd.abs() @ W.abs())
    else:
        dl = torch.zeros_like(r["logits"])
    lg, w = r["logits"], r["w"]
    m = lg.max(1, keepdim=True).values
    a = dl + dl.max(1, keepdim=True).values + U * (lg - m).abs()
    rf = (1 + torch.expm1(a)) * (1 + EXP_ULP * U) - 1
    rs = (1 + rf.max(1, keepdim=True).values) * (1 + gamma(F)) - 1
    rho = (1 + rf) * (1 + DIV_ULP * U) / (1 - rs) - 1
    dw = rho * w + TINY
    ax = x.abs()
    b = {"w": dw,
         "out": (dw[:, None, :] * ax).sum(-1) + gamma(F) * ((w + dw)[:, None, :] * ax).sum(-1)}
    dwt = r["dwt"]
    e_dwt = gamma(S) * torch.einsum("bs,bsf->bf", g.abs(), ax)
    hdwt = dwt.abs() + e_dwt
    e_dot = (dw * hdwt + w * e_dwt).sum(1, keepdim=True) + gamma(F) * ((w + dw) * hdwt).sum(1, keepdim=True)
    diff = dwt - (w * dwt).sum(1, keepdim=True)
    e_diff = (e_dwt + e_dot) * (1 + U) + U * diff.abs()
    hdiff = diff.abs() + e_diff
    e_dl = dw * hdiff + w * e_diff + U * (w + dw) * hdiff
    hdl = r["dlogit"].abs() + e_dl
    b["dlogit"] = e_dl
    if query_cond:
        aq = qd.abs()
        b["dW"] = aq.t() @ e_dl + gamma(B) * (aq.t() @ hdl)
        b["dq"] = e_dl @ W.abs().t() + gamma(F) * (hdl @ W.abs().t())
    else:
        b["dW"] = (e_dl.sum(0) + gamma(B) * hdl.sum(0))[:, None]
    return {k: v * (1 + 2.0 ** -20) + TINY for k, v in b.items()}     # room for float64's own rounding


def mixture_inputs(B: int, S: int, F: int, E: int, query_cond: bool, seed: int):
    """fp32 x [B,S,F], q [B,E], W ([E,F] or [F,1]) and g [B,S] with logits spread over about +-60, so some weights
    are near one-hot and some are tiny."""
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(B, S, F, generator=gen)
    q = torch.randn(B, E, generator=gen)
    if query_cond:
        W = torch.randn(E, F, generator=gen) * (25.0 / math.sqrt(E))
    else:
        W = (torch.rand(F, 1, generator=gen) * 120.0 - 60.0)
    g = torch.randn(B, S, generator=gen)
    return x, q, W, g


# (F, S, B, E, query_cond, requires-grad subset of "xqW"): every F with each S, B and E; 256 % F != 0 for 3, 7, 33, 44,
# 63; the second lane pass of the softmax for F > 32; S*F below and above one 256-thread sweep
_MIX_FS = (1, 2, 3, 7, 31, 32, 33, 44, 63, 64)
_MIX_SS = (1, 37, 1000)
_MIX_BS = (1, 5, 64)
_MIX_ES = (4, 100, 768)
_SUBSETS = ("x", "q", "W", "xq", "xW", "qW", "xqW")
MIXTURE_CASES = [(F, _MIX_SS[(i + j) % 3], _MIX_BS[(i + 2 * j) % 3], _MIX_ES[(2 * i + j) % 3], (i + j) % 2 == 0,
                  _SUBSETS[(3 * i + j) % 7])
                 for i, F in enumerate(_MIX_FS) for j in range(3)]


def mixture_case_id(c) -> str:
    F, S, B, E, qc, req = c
    return f"F{F}_S{S}_B{B}_E{E}_{'qc' if qc else 'static'}_{req}"


# ---------------------------------------------------------------------------------------------------------------------
# Losses: per-element bar against float64
# ---------------------------------------------------------------------------------------------------------------------

def row_bar(cpu32, f64: torch.Tensor) -> torch.Tensor:
    """Allowed |cuda - f64| per element: 4 |cpu_fp32 - f64| + 2^-20 max |f64| over the element's row (last axis).
    ``cpu32`` is one fp32 CPU result or several in different summation orders; the largest deviation counts, so one
    order that happens to land on the float64 value does not make the bar vanish."""
    f64 = f64.double().cpu()
    runs = cpu32 if isinstance(cpu32, (list, tuple)) else [cpu32]
    dev = torch.stack([(r.double().cpu() - f64).abs() for r in runs]).amax(0)
    rowmax = f64.abs() if f64.dim() == 0 else f64.abs().amax(dim=-1, keepdim=True)
    return 4 * dev + 2.0 ** -20 * rowmax


def spread_rows(t: torch.Tensor, gen: torch.Generator) -> torch.Tensor:
    """Scale every E-row of a [P,F,E] or [P,F,Neg,E] tensor by 2^k, k uniform in [-8, 8] per (p, f)."""
    k = torch.randint(-8, 9, t.shape[:2], generator=gen).double()
    return t * torch.pow(2.0, k).to(t.dtype).view(*t.shape[:2], *([1] * (t.dim() - 2)))
