"""Float64 restatement of the filtered top-k (DESIGN §4.5) and bitmap rows built with ``safe_docs_bitmap``.

``filtered_topk`` ranks each query's ELIGIBLE docs under the kernels' rule (``mfar_oracle.rank_rows``: NaN > +inf >
finite descending > -inf, the lower doc id first inside a class) and pads a query with fewer than k eligible docs with
(-inf, -1).  Scores are given in float64 and rounded to fp32 once, the type the kernels report.
"""
from __future__ import annotations

from typing import Sequence, Tuple

import numpy as np

import mfar_oracle as O
from mfar_b200.data.bm25 import safe_docs_bitmap


def bitmap_rows(eligible: np.ndarray, doc_id_base: int) -> np.ndarray:
    """uint32 [R, W] rows of a filter over GLOBAL doc ids from bool [R, N] eligibility of local docs 0..N-1 (W covers
    doc_id_base + N).  Every row is one ``safe_docs_bitmap``."""
    eligible = np.atleast_2d(eligible)
    total = doc_id_base + eligible.shape[1]
    return np.stack([safe_docs_bitmap(np.flatnonzero(e) + doc_id_base, total) for e in eligible])


def eligible_from_bits(bits: np.ndarray, doc_id_base: int, n_docs: int) -> np.ndarray:
    """bool [R, n_docs]: the bits of global docs [doc_id_base, doc_id_base + n_docs) of uint32 rows [R, W]."""
    bits = np.atleast_2d(np.asarray(bits).view(np.uint32))
    ids = doc_id_base + np.arange(n_docs, dtype=np.int64)
    return ((bits[:, ids >> 5] >> (ids & 31).astype(np.uint32)) & 1).astype(bool)


def filtered_topk(scores: np.ndarray, eligible: np.ndarray, k: int, doc_id_base: int = 0
                  ) -> Tuple[np.ndarray, np.ndarray]:
    """(fp32 [Q, k], int64 [Q, k]): the top k of each row of ``scores`` [Q, N] among the docs whose ``eligible`` bit is
    set ([N] shared or [Q, N] per query), ids global, missing slots (-inf, -1)."""
    s = np.asarray(scores, dtype=np.float64).astype(np.float32)
    Q, N = s.shape
    el = np.broadcast_to(np.atleast_2d(eligible), (Q, N))
    out_s = np.full((Q, k), -np.inf, dtype=np.float32)
    out_i = np.full((Q, k), -1, dtype=np.int64)
    for q in range(Q):
        idx = np.flatnonzero(el[q])
        if idx.size == 0:
            continue
        sel = idx[O.rank_rows(s[q, idx], k)]          # idx ascending: the subset's row order is the doc id order
        out_s[q, :sel.size] = s[q, sel]
        out_i[q, :sel.size] = sel + doc_id_base
    return out_s, out_i


def unfiltered_rank(scores: np.ndarray, k: int) -> Sequence[np.ndarray]:
    """Local rows of each row's unfiltered top k (the ids a filter can leave out on purpose)."""
    return [O.rank_rows(np.asarray(r, dtype=np.float64).astype(np.float32), k) for r in np.atleast_2d(scores)]
