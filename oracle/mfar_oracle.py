"""CPU oracle for mFAR's multi-field scoring + retrieval hot path.

TEST INFRASTRUCTURE ONLY.  Nothing in the product package imports this file; only
``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl
reference`` legs may call it, and there only as the checker / CPU baseline.

It is a fresh restatement (torch CPU, fp32) of the reference algorithm.  Every function
cites the reference file:line it follows (paths relative to the upstream repo root).

Parity pinning: the reference ships no tests, golden vectors or fixtures for this path
(SURVEY.md section 4 / 8c), so the oracle is pinned against outputs of the reference's
own classes (DenseFlatIndex, BM25sSparseIndex.score_batch, LinearWeights, MemoryMapDict)
executed in the build container.  ``oracle/make_golden.py`` is the generating script,
``tests/golden/*.npz`` the committed vectors, ``tests/test_oracle_golden.py`` the check.
BM25 arithmetic itself (third-party ``bm25s`` 0.1.10, not vendored, not installed) is NOT
restated: per-field BM25 score vectors are inputs to this path -> "BM25 parity unpinned".

Two modes (SURVEY.md section 0):
  * ``exhaustive``     - the reference's formulas applied to all N docs (graded mode)
  * ``union_rescore``  - the faithful ``trec_eval_step`` pipeline:
                         per-field top-k -> union -> rescore -> mask -> mixture -> top-k
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch


# --------------------------------------------------------------------------------------
# Field mixture                                           mfar/modeling/weighting.py:17-29
# --------------------------------------------------------------------------------------
def mixture_weights(q_emb: Optional[torch.Tensor], W: torch.Tensor, query_cond: bool) -> torch.Tensor:
    """softmax over fields of ``q @ W`` (query-conditioned, weighting.py:25) or of ``W^T``
    (weighting.py:27; W is [F, 1] there, contrastive.py:285).  Returns [Q, F] or [1, F]."""
    if query_cond:
        logits = q_emb.float() @ W.float()            # [Q, E] @ [E, F]
    else:
        logits = W.float().transpose(1, 0)            # [1, F]
    return torch.softmax(logits, dim=1)               # weighting.py:28


def linear_weights_forward(x: torch.Tensor, q_emb: Optional[torch.Tensor], W: torch.Tensor,
                           query_cond: bool) -> torch.Tensor:
    """``LinearWeights.forward`` (weighting.py:17-29): sum_f softmax_f * x[..., f].
    x is [B, S, F] (or [S, F], which broadcasts to [1, S] exactly as in trec_eval_step)."""
    w = mixture_weights(q_emb, W, query_cond)
    return torch.sum(w.unsqueeze(1) * x, dim=-1)      # weighting.py:29


# --------------------------------------------------------------------------------------
# Dense flat index                                            mfar/data/index.py:181-232
# --------------------------------------------------------------------------------------
def dense_retrieve_batch(q_vecs: torch.Tensor, vectors: torch.Tensor, top_k: int,
                         vector_batch_size: int = 1048576) -> Tuple[torch.Tensor, torch.Tensor]:
    """``DenseFlatIndex.retrieve_batch`` (index.py:181-222).

    Chunked ``q @ V^T`` merged into a running top-k that starts as (score 0.0, row 0)
    (index.py:192-193) - so when fewer than k rows score above 0 the result contains
    (0.0, row 0) entries, exactly like the reference.  Returns (scores [Q,k], rows [Q,k]),
    sorted descending (index.py:203-209)."""
    q = q_vecs.float()
    Q = q.shape[0]
    top_scores = torch.zeros((Q, top_k), dtype=torch.float32)
    top_rows = torch.zeros((Q, top_k), dtype=torch.int64)
    n = vectors.shape[0]
    for lb in range(0, n, vector_batch_size):
        ub = min(n, lb + vector_batch_size)
        s = torch.matmul(q, vectors[lb:ub].float().t())                       # index.py:197
        comb_s = torch.cat([top_scores, s], dim=1)                            # index.py:198
        comb_i = torch.cat([top_rows, torch.arange(lb, ub).unsqueeze(0).expand(Q, -1)], dim=1)
        cs, ci = torch.topk(comb_s, top_k, dim=1, largest=True, sorted=True)  # index.py:203
        top_rows = comb_i[torch.arange(Q).unsqueeze(1), ci]                   # index.py:211
        top_scores = cs[:, :top_k]
    return top_scores, top_rows


def dense_score_batch(q_vecs: torch.Tensor, vectors: torch.Tensor, rows: Sequence[int]) -> torch.Tensor:
    """``DenseFlatIndex.score_batch`` (index.py:227-232): gather candidate rows, ``q @ V_c^T``.
    Returns [Q, C] fp32."""
    idx = torch.as_tensor(list(rows), dtype=torch.int64)
    return torch.matmul(q_vecs.float(), vectors[idx].float().t())             # index.py:230-231


# --------------------------------------------------------------------------------------
# Sparse (BM25) index as an input provider                    mfar/data/index.py:95-118
# --------------------------------------------------------------------------------------
def sparse_retrieve_batch(score_vecs: torch.Tensor, top_k: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """``BM25sSparseIndex.retrieve_batch`` (index.py:95-103) given the full-corpus score
    vectors ``get_scores`` would return (index.py:72-76): top-k rows by score, descending.
    (bm25s' own top-k tie order is unpinned.)"""
    s, i = torch.topk(score_vecs.float(), top_k, dim=1, largest=True, sorted=True)
    return s, i


def sparse_score_batch(score_vecs: torch.Tensor, rows: Sequence[int]) -> torch.Tensor:
    """``BM25sSparseIndex.score_batch`` (index.py:111-118): gather candidate columns from
    the per-query full-corpus score vectors; unknown keys (row == -1) score 0 (112-117)."""
    idx = torch.as_tensor(list(rows), dtype=torch.int64)
    out = score_vecs.float()[:, idx.clamp(min=0)].clone()
    out[:, idx < 0] = 0.0
    return out


# --------------------------------------------------------------------------------------
# Exhaustive mode (graded): reference formulas over all N docs
# --------------------------------------------------------------------------------------
def exhaustive_scores(q_vecs: torch.Tensor, dense_fields: Sequence[torch.Tensor],
                      sparse_scores: Optional[torch.Tensor], weights: torch.Tensor,
                      mask: Optional[torch.Tensor] = None, doc_chunk: int = 65536,
                      normalize: bool = False) -> torch.Tensor:
    """Mixture score of every doc: ``sum_f w[q,f] * mask[f] * s_f[q,n]`` with
    s_f = q . v_f for dense fields (index.py:197 / 231) followed by the sparse fields'
    precomputed scores (index.py:114-117), field order dense-then-sparse (schema.py:130-134),
    mask applied to the per-field scores before the mixture and NOT renormalised
    (contrastive.py:686 then weighting.py:28-29).

    q_vecs [Q,d]; dense_fields: F_d tensors [N,d]; sparse_scores [Q,F_s,N] or None;
    weights [Q,F] or [1,F] (already softmaxed).  With ``normalize`` (cosine: the encoder ends in
    ``Normalize()``, modeling/util.py:50-51) queries and doc rows first go through
    ``normalize_rows_bf16``.  Returns [Q, N] fp32."""
    if normalize:
        q_vecs = torch.from_numpy(normalize_rows_bf16(q_vecs))
        dense_fields = [torch.from_numpy(normalize_rows_bf16(f)) for f in dense_fields]
    Q = q_vecs.shape[0]
    Fd = len(dense_fields)
    Fs = 0 if sparse_scores is None else sparse_scores.shape[1]
    N = dense_fields[0].shape[0] if Fd else sparse_scores.shape[2]
    w = weights.float().expand(Q, Fd + Fs)
    if mask is not None:
        w = w * mask.float().reshape(1, -1)
    q = q_vecs.float()
    out = torch.zeros((Q, N), dtype=torch.float32)
    for lb in range(0, N, doc_chunk):
        ub = min(N, lb + doc_chunk)
        acc = torch.zeros((Q, ub - lb), dtype=torch.float32)
        for f in range(Fd):
            acc += w[:, f:f + 1] * torch.matmul(q, dense_fields[f][lb:ub].float().t())
        for j in range(Fs):
            acc += w[:, Fd + j:Fd + j + 1] * sparse_scores[:, j, lb:ub].float()
        out[:, lb:ub] = acc
    return out


NAN_ORDERED = 0xFFC00000          # csrc/common.cuh kNanOrdered: the one score word of every NaN, above +inf's


def ordered_words(scores: np.ndarray) -> np.ndarray:
    """uint64 score words of the device key (csrc/common.cuh ``float_to_ordered``): unsigned order == the rank order
    NaN (any sign or payload) > +inf > finite (desc) > -inf.  -0.0 is folded into +0.0 first (one zero, as in
    ``torch.topk``; the kernels' sums never produce -0.0)."""
    with np.errstate(invalid="ignore"):
        f = np.asarray(scores, dtype=np.float32) + np.float32(0.0)
    u = f.view(np.uint32).astype(np.uint64)
    o = np.where((u & np.uint64(0x80000000)) != 0, (~u) & np.uint64(0xFFFFFFFF), u | np.uint64(0x80000000))
    return np.where(np.isnan(f), np.uint64(NAN_ORDERED), o)


def rank_rows(scores: np.ndarray, k: int) -> np.ndarray:
    """Rows of the top k of one fp32 score row under the kernels' rule: NaN (every NaN one value) > +inf > finite
    scores descending > -inf, the lower row first inside a class - ``torch.topk``'s order (NaN counts as the largest
    value) with the tie order made explicit.  Ranks the composite uint64 (score word, ~row) key, the device's own."""
    N = int(np.asarray(scores).shape[0])
    k = min(k, N)
    assert N < (1 << 32)
    key = (ordered_words(scores) << np.uint64(32)) | (~np.arange(N, dtype=np.uint64) & np.uint64(0xFFFFFFFF))
    part = np.argpartition(key, N - k)[N - k:] if k < N else np.arange(N)
    return part[np.argsort(key[part])[::-1]]


def topk_sorted(scores: torch.Tensor, k: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """``torch.topk(k)`` (contrastive.py:696) with the tie order made explicit: NaN > +inf > finite scores
    descending > -inf, then row ascending (``rank_rows``; torch leaves tie order unspecified)."""
    s = scores.float().numpy()
    Q, N = s.shape
    k = min(k, N)
    out_s = np.empty((Q, k), dtype=np.float32)
    out_i = np.empty((Q, k), dtype=np.int64)
    for qi in range(Q):
        sel = rank_rows(s[qi], k)
        out_i[qi] = sel
        out_s[qi] = s[qi][sel]
    return torch.from_numpy(out_s), torch.from_numpy(out_i)


def exhaustive_topk(q_vecs, dense_fields, sparse_scores, weights, mask=None, k: int = 100,
                    doc_chunk: int = 65536) -> Tuple[torch.Tensor, torch.Tensor]:
    """Exhaustive multi-field top-k: ``exhaustive_scores`` then ``topk_sorted``."""
    return topk_sorted(exhaustive_scores(q_vecs, dense_fields, sparse_scores, weights, mask, doc_chunk), k)


# --------------------------------------------------------------------------------------
# Faithful pipeline                                  mfar/modeling/contrastive.py:669-704
# --------------------------------------------------------------------------------------
def union_rescore(q_vecs: torch.Tensor, dense_fields: Sequence[torch.Tensor],
                  sparse_scores: Optional[torch.Tensor], q_emb: Optional[torch.Tensor],
                  W: torch.Tensor, query_cond: bool, mask: Optional[torch.Tensor] = None,
                  k: int = 100, vector_batch_size: int = 1048576
                  ) -> Tuple[List[torch.Tensor], List[List[int]]]:
    """``RetrievalTrainingModule.trec_eval_step`` (contrastive.py:669-704) with the text
    encoder factored out (query vectors are inputs).

    A. per-field ``retrieve_batch(top_k=k)``                       (672-674)
    B. per query: union of the F id sets                            (676-679)
    C. per query, per field: ``score_batch`` on the union          (681-683)
    D. stack [F,U] * mask [F,1]                                     (685-686)
    E. ``mixture_of_fields_layer(all_tens.t(), x_encoded)`` -> [1,U] (694)
    F. ``torch.topk(k)``                                            (696)
    The union is ordered by ascending row here (the reference iterates a Python set of
    string ids, whose order only matters for exact ties).  Returns per query
    (values [k], rows [k])."""
    Q = q_vecs.shape[0]
    Fd = len(dense_fields)
    Fs = 0 if sparse_scores is None else sparse_scores.shape[1]
    F = Fd + Fs
    mask_t = torch.ones(F, 1) if mask is None else mask.float().reshape(F, 1)
    hits = []
    for f in range(Fd):
        hits.append(dense_retrieve_batch(q_vecs, dense_fields[f], k, vector_batch_size)[1])
    for j in range(Fs):
        hits.append(sparse_retrieve_batch(sparse_scores[:, j, :], k)[1])
    out_vals, out_rows = [], []
    for i in range(Q):
        union = sorted(set().union(*[set(h[i].tolist()) for h in hits]))
        new_hits = []
        for f in range(Fd):
            new_hits.append(dense_score_batch(q_vecs[i:i + 1], dense_fields[f], union))
        for j in range(Fs):
            new_hits.append(sparse_score_batch(sparse_scores[i:i + 1, j, :], union))
        all_tens = torch.stack(new_hits, dim=0).squeeze(1)          # [F, U]
        all_tens = all_tens * mask_t
        qe = None if q_emb is None else q_emb[i:i + 1]
        scores = linear_weights_forward(all_tens.t(), qe, W, query_cond)   # [1, U]
        if scores.shape[1] < k:      # torch.topk (contrastive.py:696) raises when the union is smaller than k
            raise RuntimeError("selected index k out of range")
        vals, idx = topk_sorted(scores, k)
        out_vals.append(vals[0])
        out_rows.append([union[j] for j in idx[0].tolist()])
    return out_vals, out_rows


# --------------------------------------------------------------------------------------
# bf16 rounding shared by tests / bench (the kernel and the oracle consume the SAME
# bf16-rounded tensors - SURVEY.md section 7 "Parity definition")
# --------------------------------------------------------------------------------------
def round_bf16(x: torch.Tensor) -> torch.Tensor:
    return x.to(torch.bfloat16).to(torch.float32)


# --------------------------------------------------------------------------------------
# Cosine: L2 normalisation rounded once to bf16                modeling/util.py:50-51
# --------------------------------------------------------------------------------------
NORM_EPS = float(np.float32(1e-12))     # F.normalize's eps as it acts on an fp32 tensor
BF16_MIN_EXP = -133                     # exponent of the bf16 subnormal spacing


def round_bf16_rne(y) -> np.ndarray:
    """float64 -> the nearest bf16 value (ties to even), as float64: ONE rounding, including bf16 subnormals
    (spacing 2^-133) and overflow to +-inf.  Signs of zeros are kept.  (torch's float64 -> bf16 cast may round twice
    through fp32, so it is not used here.)"""
    y = np.asarray(y, dtype=np.float64)
    _, e = np.frexp(y)                                  # |y| = m 2^e, 0.5 <= m < 1: 8 significant bits -> 2^(e-8)
    q = np.maximum(e - 8, BF16_MIN_EXP)
    with np.errstate(over="ignore"):
        r = np.ldexp(np.rint(np.ldexp(y, -q)), q)       # the scaling is exact; rint rounds half to even
    big = np.abs(r) >= 2.0 ** 128                       # past the largest bf16 (1 - 2^-8) 2^128
    return np.where(big, np.copysign(np.inf, y), r)


def normalize_rows_bf16(x) -> np.ndarray:
    """The cosine contract of ``PackedCorpus(normalize=True)`` for docs and queries alike: every row, taken exactly into
    float64, is divided by ``max(||x||_2, float32(1e-12))`` in float64 and rounded ONCE to nearest-even bf16.  An
    all-zero row stays zero and keeps the signs of its zeros.  x: [n, d] fp32 / bf16 / f16 (tensor or array).
    Returns float32 [n, d] holding bf16 values exactly."""
    if torch.is_tensor(x):
        x = x.detach().cpu().double().numpy()
    x = np.asarray(x, dtype=np.float64)
    norm = np.sqrt(np.sum(x * x, axis=1, keepdims=True))   # squares of fp32 values are exact in float64
    y = x / np.maximum(norm, NORM_EPS)
    return round_bf16_rne(y).astype(np.float32)
