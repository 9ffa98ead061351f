"""Inputs whose mixture scores are EXACT in fp32 whatever the summation order, and their closed-form top-k.

Doc coordinates are small integers (0..255, exact in bf16); a query puts the coefficients +-2^16, +-2^8, +-1 (exact in
bf16) on the three coordinates of ONE group, so doc n scores ``sum(coef * coord)``, an integer below 2^22 in magnitude.
Every partial sum of such products is an integer below 2^24 and therefore exact in fp32 on CUDA cores and in the
tensor cores' fp32 accumulator alike; mixture weights of exactly 1/F (F in {1, 2, 4}) only move the binary point.
The correct top-k is then the (score desc, doc id asc) order of integers - no tolerance, no near-tie rule - and an
answer that differs in one id inside a tie group is wrong.

Every pattern is tied or ordered in a way that stresses one part of the top-k machinery (tests/test_gpu_topk_exact.py):
``n`` ascending / descending (sign), ``mod128/127/129`` (one member of each tie group per tile, aligned and not),
``div37/div1000`` (runs of duplicates across tiles, CTAs, shard cuts), ``planted`` (fewer than 100 distinct winners
above a tied floor), ``perm`` (control: distinct scores in random order), ``zero_sign`` (docs that cancel to +0 and
all-zero docs in one tie group) and ``equal`` (the zero query: every doc ties).
"""
from __future__ import annotations

from typing import List, Tuple

import numpy as np

PATTERNS = ("n", "mod128", "mod127", "mod129", "div37", "div1000", "planted", "perm", "zero_sign", "equal")
COMBOS: List[Tuple[str, int]] = [(p, s) for p in PATTERNS for s in (1, -1)]   # (pattern, query sign)
GROUPS = [p for p in PATTERNS if p != "equal"]                                  # patterns that own a coordinate group
MAX_SCORE = 1 << 22
LEVELS = (65536, 256, 1)


def pattern_values(name: str, N: int) -> np.ndarray:
    """int64 [N] value v(n) >= 0 of a three-level pattern (score = sign * v)."""
    n = np.arange(N, dtype=np.int64)
    if name == "n":
        v = n
    elif name.startswith("mod"):
        v = n % int(name[3:])
    elif name.startswith("div"):
        v = n // int(name[3:])
    elif name == "planted":                             # a few distinct winners above a floor of N - P zeros
        rng = np.random.default_rng(1000 + N)
        P = min(40, N // 4)
        v = np.zeros(N, dtype=np.int64)
        v[rng.choice(N, P, replace=False)] = 1 + rng.permutation(P)
    elif name == "perm":
        v = np.random.default_rng(2000 + N).permutation(N).astype(np.int64)
    else:
        raise ValueError(name)
    if N > MAX_SCORE or v.max(initial=0) >= MAX_SCORE:
        raise ValueError(f"pattern {name} at N={N} leaves the exact range")
    return v


def pattern_terms(name: str, N: int) -> List[Tuple[int, np.ndarray]]:
    """[(query coefficient, doc coordinates uint8 [N])] of a pattern's group (empty for ``equal``)."""
    if name == "equal":
        return []
    if name == "zero_sign":                             # query (+1, -1): n%3==0 (c,c) -> +0, n%3==1 (0,0), n%3==2 (0,c) -> -c
        n = np.arange(N, dtype=np.int64)
        c = 1 + (n // 3) % 255
        return [(1, np.where(n % 3 == 0, c, 0).astype(np.uint8)), (-1, np.where(n % 3 != 1, c, 0).astype(np.uint8))]
    v = pattern_values(name, N)
    return [(65536, (v >> 16).astype(np.uint8)), (256, ((v >> 8) & 255).astype(np.uint8)), (1, (v & 255).astype(np.uint8))]


def dense_scores(name: str, sign: int, N: int) -> np.ndarray:
    """int64 [N]: what every doc scores under the query (pattern, sign) - the closed form."""
    out = np.zeros(N, dtype=np.int64)
    for coef, x in pattern_terms(name, N):
        out += sign * coef * x.astype(np.int64)
    return out


def group_positions(g: int, dim: int) -> Tuple[int, int, int]:
    """Coordinates of group g: with dim >= 768 in three different 64-wide K blocks, the last one always in the LAST
    block, so a dropped, duplicated or reordered K block changes the answer."""
    if dim == 64:
        return g, 16 + g, 32 + g
    if dim < 768:
        raise ValueError("groups are laid out for dim 64 or >= 768")
    return 64 * (g % 12) + 10 + g // 12, 64 * ((g + 4) % 12) + 30 + g // 12, dim - 64 + 40 + g


def doc_matrix(N: int, dim: int, lo: int = 0, hi: int = None) -> np.ndarray:
    """uint8 [hi-lo, dim] coordinates of docs [lo, hi) (every group filled)."""
    hi = N if hi is None else hi
    out = np.zeros((hi - lo, dim), dtype=np.uint8)
    for g, name in enumerate(GROUPS):
        pos = group_positions(g, dim)
        terms = pattern_terms(name, N)
        slots = (pos[0], pos[2]) if len(terms) == 2 else pos     # zero_sign: first and last-block coordinate
        for p, (_, x) in zip(slots, terms):
            out[:, p] = x[lo:hi]
    return out


def query_vector(name: str, sign: int, dim: int) -> np.ndarray:
    q = np.zeros(dim, dtype=np.float32)
    if name == "equal":
        return q
    g = GROUPS.index(name)
    pos = group_positions(g, dim)
    terms = pattern_terms(name, 4)
    slots = (pos[0], pos[2]) if len(terms) == 2 else pos
    for p, (coef, _) in zip(slots, terms):
        q[p] = sign * coef
    return q


def topk_order(scores: np.ndarray, k: int) -> np.ndarray:
    """Local rows of the top k of int64 scores under (score desc, row asc) - argpartition on one composite int64 key."""
    N = scores.shape[0]
    k = min(k, N)
    assert np.abs(scores).max(initial=0) < (1 << 30) and N < (1 << 31)
    comp = (-(scores.astype(np.int64)) + (1 << 30)) * (1 << 31) + np.arange(N, dtype=np.int64)
    part = np.argpartition(comp, k - 1)[:k] if k < N else np.arange(N)
    return part[np.argsort(comp[part], kind="stable")]
