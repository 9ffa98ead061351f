"""Non-finite scores with a closed-form answer: the inputs of tests/exact_topk.py plus NaN and infinities planted on
coordinates that no pattern group uses.

Docs keep their small-integer pattern coordinates (exact_topk.doc_matrix), so every finite score is still an exact
integer.  On top of that, reserved coordinates carry
  ``nan``    bf16 NaN of both signs (and two payloads) at a few docs: those docs score NaN under every query
             (0 * NaN = NaN);
  ``few``    bf16 +inf at fewer than 100 docs;
  ``many``   bf16 +inf at n % 29 == 3 (N < 100k) or n % 97 == 3: more than 128 docs, on every tile stride and inside
             the threshold-seeding prefix;
  ``almost`` bf16 +inf at every doc but ~40 (only in the corpora built with ``almost=True``).
A query puts a coefficient of +1, -1 or 0 on each +inf coordinate, so the same docs score +inf, -inf or NaN
(0 * inf) depending on the query, and +inf + -inf where sets overlap.  The expected score of a (doc, query) pair is the
IEEE evaluation of the same formula in float64 (``dense_values``); its class does not depend on the summation order.
The expected ranking is ``mfar_oracle.rank_rows``: NaN > +inf > finite desc > -inf, lower doc id first in a class.
"""
from __future__ import annotations

import itertools
from typing import Dict, Tuple

import numpy as np

import exact_topk as X

BF16_INF = 0x7F80
BF16_NANS = (0x7FC0, 0xFFC0, 0x7F81, 0xFF81)          # +NaN, -NaN, and both signs with another payload
PLANTS = ("few", "many", "almost")                    # +inf coordinates, in query-coefficient order
COEFS = list(itertools.product((1, -1, 0), repeat=2))  # (few, many) coefficients of a query
NEG_NAN_F32 = np.array([0xFFC00001], dtype=np.uint32).view(np.float32)[0]


def reserved(dim: int) -> Dict[str, int]:
    """Coordinates of the planted values: offsets 50..58 of a 64-wide K block, which no pattern group uses (groups sit
    at offsets 0..48), spread over different K blocks (the ``many`` one in the last)."""
    if dim == 64:
        return dict(nan=50, few=52, many=54, almost=56, big=58)
    assert dim >= 768
    return dict(nan=64 * 2 + 50, few=64 * 5 + 52, many=dim - 64 + 54, almost=56, big=64 * 7 + 58)


def plant_sets(N: int) -> Dict[str, np.ndarray]:
    """bool [N] masks of the planted docs."""
    n = np.arange(N)
    nan = np.zeros(N, dtype=bool)
    nan[[0, 130, N // 2, N - 1]] = True                 # first tile, second tile, the middle, the last doc
    few = np.zeros(N, dtype=bool)
    few[np.unique(np.linspace(1, N - 2, 24).astype(np.int64))] = True
    few[5] = True
    many = n % (29 if N < 100_000 else 97) == 3
    almost = n % max(2, N // 40) != 1
    return dict(nan=nan, few=few, many=many, almost=almost)


def nan_bits(N: int) -> np.ndarray:
    """uint16 [N]: the bf16 NaN planted at each ``nan`` doc (the i-th one takes BF16_NANS[i % 4]), 0 elsewhere."""
    at = np.nonzero(plant_sets(N)["nan"])[0]
    out = np.zeros(N, dtype=np.uint16)
    out[at] = np.array(BF16_NANS, dtype=np.uint16)[np.arange(at.size) % len(BF16_NANS)]
    return out


def plant_columns(N: int, dim: int, almost: bool, lo: int = 0, hi: int = None) -> Dict[int, np.ndarray]:
    """{coordinate: int16 bf16 bit patterns [hi-lo]} to overwrite in the packed rows of docs [lo, hi) (0 = bf16 +0)."""
    hi = N if hi is None else hi
    S, pos = plant_sets(N), reserved(dim)
    cols = {}
    cols[pos["nan"]] = nan_bits(N)[lo:hi]
    for name in PLANTS:
        if name == "almost" and not almost:
            continue
        cols[pos[name]] = np.where(S[name], BF16_INF, 0)[lo:hi]
    return {p: v.astype(np.uint16).view(np.int16) for p, v in cols.items()}


def query_vector(combo: Tuple[str, int], coefs: Tuple[int, ...], dim: int) -> np.ndarray:
    """exact_topk's query of (pattern, sign) plus the coefficients on the ``few``, ``many`` (and ``almost``) coords."""
    q = X.query_vector(*combo, dim)
    pos = reserved(dim)
    for name, c in zip(PLANTS, coefs):
        q[pos[name]] = c
    return q


def dense_values(combo, coefs, N: int, almost: bool) -> np.ndarray:
    """float64 [N]: the dot product of every doc with the query, evaluated in IEEE float64 (closed form)."""
    v = X.dense_scores(*combo, N).astype(np.float64)
    S = plant_sets(N)
    with np.errstate(invalid="ignore"):
        v = v + np.where(S["nan"], np.nan, 0.0)
        names = PLANTS if almost else PLANTS[:2]
        assert len(coefs) == len(names), "a corpus with the almost-all plant needs three coefficients"
        for name, c in zip(names, coefs):
            v = v + np.where(S[name], c * np.inf, 0.0)
    return v


def classes(x: np.ndarray) -> np.ndarray:
    """int8 class of every value: 3 NaN, 2 +inf, 1 finite, 0 -inf."""
    x = np.asarray(x, dtype=np.float64)
    return np.where(np.isnan(x), 3, np.where(x == np.inf, 2, np.where(x == -np.inf, 0, 1))).astype(np.int8)


def brute_force_order(s: np.ndarray, k: int) -> np.ndarray:
    """Rows of the top k by a float64 sort on (class desc, value desc, row asc) - the rule spelled out, O(N log N)."""
    x = np.asarray(s, dtype=np.float64)
    cls = classes(x)
    val = np.where(cls == 1, x, 0.0)
    return np.lexsort((np.arange(x.shape[0]), -val, -cls))[:k]
