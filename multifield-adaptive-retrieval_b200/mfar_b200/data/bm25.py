"""Device-resident BM25 index: stands where ``bm25s.BM25`` stands in the reference
(``BM25sSparseIndex``, mfar/data/index.py:39-157; ``bm25s.BM25(method="lucene", k1=1.2, b=0.75)``, index.py:138).

The score matrix (token-major CSC, fp32) lives in HBM; ``get_scores`` / ``retrieve`` and the fused hybrid search
(``MultiFieldRetriever.search(sparse_tokens=...)``) run the postings scatter-add kernel of ``csrc/bm25.cu`` through
the C ABI.  Index construction from token ids is done on the device too (sort / run-length plumbing in torch, the
BM25 arithmetic in ``mfar_bm25_build_scores``).  Nothing here computes on the CPU except text tokenisation.

bm25s (0.1.10) is a third-party dependency of the reference that is not available in this image: formulas, the
tokeniser defaults and the on-disk file names follow its published behaviour - BM25 parity is unpinned.
"""
from __future__ import annotations

import ctypes
import json
import os
import re
from typing import Dict, List, Optional, Sequence, Tuple, Union

import numpy as np
import torch

from .. import _native as nv

# bm25s "en" stop words (Lucene's default English set)
STOPWORDS_EN = ("a", "an", "and", "are", "as", "at", "be", "but", "by", "for", "if", "in", "into", "is", "it", "no",
                "not", "of", "on", "or", "such", "that", "the", "their", "then", "there", "these", "they", "this",
                "to", "was", "will", "with")
_TOKEN_RE = re.compile(r"(?u)\b\w\w+\b")


def tokenize(texts: Union[str, Sequence[str]], stopwords: Union[str, Sequence[str], None] = "en",
             stemmer: Optional[object] = None) -> List[List[str]]:
    """``bm25s.tokenize(texts, stopwords=..., stemmer=..., return_ids=False)`` (index.py:64,139): lower-case,
    ``\\b\\w\\w+\\b`` tokens, stop words dropped, optional stemmer (an object with ``stemWords`` or a callable that maps a
    token list to a token list, as bm25s calls it)."""
    if isinstance(texts, str):
        texts = [texts]
    stop = set(STOPWORDS_EN if stopwords in ("en", "english", True) else (stopwords or ()))
    out = []
    for text in texts:
        toks = [t for t in _TOKEN_RE.findall(text.lower()) if t not in stop]
        if stemmer is not None:
            # bm25s' contract: a PyStemmer-like object, or a callable applied to the WHOLE token list
            toks = list(stemmer.stemWords(toks)) if hasattr(stemmer, "stemWords") else list(stemmer(toks))
        out.append(toks)
    return out


def tokens_to_ids(vocab_dict: Optional[Dict[str, int]], query_tokens: Sequence) -> List[int]:
    """bm25s ``get_tokens_ids``: str tokens are looked up and dropped when absent from the vocabulary (repeats are
    kept); integer tokens are taken as vocabulary ids."""
    if len(query_tokens) and isinstance(query_tokens[0], str):
        vd = vocab_dict or {}
        return [vd[t] for t in query_tokens if t in vd]
    return [int(t) for t in query_tokens]


def token_entries(vocab_dicts: Sequence[Optional[Dict[str, int]]],
                  tokens_per_field: Sequence[Sequence[Sequence]]) -> np.ndarray:
    """tokens_per_field[j][q] = token list (str or vocabulary ids) of query q for sparse field j
    -> int32 [n_entries, 3] rows (query row, field, token id), one per token occurrence, sorted by query row - the
    batch format of ``mfar_score_topk_bm25`` / ``mfar_bm25_scores`` (any order is accepted there; query-major order
    is the fast one)."""
    if len(tokens_per_field) != len(vocab_dicts):
        raise ValueError(f"need token lists for {len(vocab_dicts)} sparse fields, got {len(tokens_per_field)}")
    n_q = {len(per_query) for per_query in tokens_per_field}
    if len(n_q) > 1:
        raise ValueError(f"sparse fields disagree on the number of queries: {sorted(n_q)}")
    # query-major order: the scatter kernel walks the entries' postings in this order, so the slice of the fp32
    # score rows being accumulated at any moment is a few queries' rows (L2-resident) instead of all Q rows
    rows = []
    for q in range(n_q.pop() if n_q else 0):
        for j, vd in enumerate(vocab_dicts):
            ids = tokens_to_ids(vd, tokens_per_field[j][q])
            if ids:
                a = np.empty((len(ids), 3), dtype=np.int32)
                a[:, 0], a[:, 1], a[:, 2] = q, j, ids
                rows.append(a)
    return np.concatenate(rows) if rows else np.zeros((0, 3), dtype=np.int32)


def safe_docs_bitmap(safe_docs, n_docs_total: int) -> np.ndarray:
    """uint32 bitmap over global doc ids (bit d set <=> d in ``safe_docs``) - the membership test of
    ``get_scores_sparse`` (index.py:82-83) in the form ``mfar_sparse_coo_count/write`` take.  Ids outside
    ``[0, n_docs_total)`` can never be hit by a score row and are dropped."""
    bits = np.zeros((int(n_docs_total) + 31) // 32, dtype=np.uint32)
    ids = np.fromiter((int(d) for d in safe_docs), dtype=np.int64)
    ids = ids[(ids >= 0) & (ids < n_docs_total)]
    np.bitwise_or.at(bits, ids >> 5, (np.uint32(1) << (ids & 31).astype(np.uint32)))
    return bits


def rows_to_coo(scores: torch.Tensor, n_docs: int, safe_bits: Optional[torch.Tensor] = None,
                qids: Optional[torch.Tensor] = None, doc_id_base: int = 0,
                vals_dtype: torch.dtype = torch.float16) -> Tuple[torch.Tensor, torch.Tensor]:
    """Dense score rows fp32 [Q, ld] (device) -> the pairs ``precompute_score_for_field`` writes
    (precompute_bm25s_scores.py:19-27): keys int32 [nnz,2] = (qid, doc), vals [nnz] = np.float16(score), entries
    != 0 whose doc is in the safe set, ordered (query row, doc).  Two device passes (count + scan, write) and ONE
    host read of nnz in between; see csrc/sparse_coo.cu."""
    nv.require_device(scores, "scores")
    if scores.dtype != torch.float32 or scores.dim() != 2 or scores.stride(1) != 1:
        raise ValueError("scores must be fp32 [Q, ld] with unit column stride")
    if vals_dtype not in (torch.float16, torch.float32):
        raise ValueError("vals_dtype must be float16 (the reference's file dtype) or float32")
    Q, ld = scores.shape[0], scores.stride(0)
    dev = scores.device
    if safe_bits is not None:
        nv.require_device(safe_bits, "safe_bits")
        if safe_bits.dtype not in (torch.int32, torch.uint32) or safe_bits.numel() * 32 < doc_id_base + n_docs:
            raise ValueError("safe_bits must be a 32-bit bitmap covering every global doc id of this shard")
    if qids is not None:
        qids = qids.to(dev, torch.int32).contiguous()
        if qids.numel() != Q:
            raise ValueError(f"need {Q} query ids, got {qids.numel()}")
    lib = nv.lib()
    offs = torch.empty(lib.mfar_sparse_coo_offsets_len(Q, n_docs), dtype=torch.int64, device=dev)
    nv.check(lib.mfar_sparse_coo_count(nv.ptr(scores), ld, Q, n_docs, nv.ptr(safe_bits), doc_id_base, nv.ptr(offs),
                                       nv.stream()), "sparse_coo_count")
    nnz = int(offs[-1].item())
    keys = torch.empty((nnz, 2), dtype=torch.int32, device=dev)
    vals = torch.empty((nnz,), dtype=vals_dtype, device=dev)
    if nnz:
        nv.check(lib.mfar_sparse_coo_write(nv.ptr(scores), ld, Q, n_docs, nv.ptr(safe_bits), nv.ptr(qids), doc_id_base,
                                           nv.ptr(offs), nv.ptr(keys), nv.ptr(vals),
                                           nv.F16 if vals_dtype == torch.float16 else nv.F32, nv.stream()),
                 "sparse_coo_write")
    return keys, vals


class DeviceBM25:
    """``bm25s.BM25`` with the score matrix in HBM.

    Attributes mirror bm25s: ``vocab_dict`` (token -> id), ``scores`` (dict of data / indices / indptr /
    num_docs, here device tensors), ``k1``, ``b``, ``method``.  ``doc_base``/``num_docs`` describe the doc-range
    shard this instance holds (rows are local); idf and the average length are always whole-corpus statistics."""

    def __init__(self, k1: float = 1.2, b: float = 0.75, method: str = "lucene", device="cuda"):
        if method != "lucene":
            raise ValueError("only method='lucene' is implemented (the one the reference uses, index.py:138)")
        self.k1, self.b, self.method = float(k1), float(b), method
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("DeviceBM25 (mfar_b200) runs on a CUDA sm_100 device only; there is no CPU path")
        self.vocab_dict: Dict[str, int] = {}
        self.scores: Dict[str, object] = {}
        self.doc_base = 0
        self._plan: Optional[torch.Tensor] = None
        self.last_launches = 0

    # ------------------------------------------------------------------ construction
    @property
    def num_docs(self) -> int:
        return int(self.scores["num_docs"])

    @property
    def n_vocab(self) -> int:
        return int(self.scores["indptr"].numel() - 1)

    def _set(self, data, indices, indptr, num_docs: int, doc_base: int = 0) -> "DeviceBM25":
        dev = self.device

        def dev_tensor(a, dtype):
            if isinstance(a, np.ndarray) and not a.flags.writeable:    # np.load(mmap_mode="r"): copy before wrapping
                a = np.array(a)
            return torch.as_tensor(a).to(dev, dtype).contiguous()
        self.scores = {
            "data": dev_tensor(data, torch.float32),
            "indices": dev_tensor(indices, torch.int32),
            "indptr": dev_tensor(indptr, torch.int64),
            "num_docs": int(num_docs),
        }
        self.doc_base = int(doc_base)
        return self

    @classmethod
    def from_csc(cls, data, indices, indptr, num_docs: int, vocab_dict: Optional[Dict[str, int]] = None,
                 k1: float = 1.2, b: float = 0.75, device="cuda",
                 doc_range: Optional[Tuple[int, int]] = None) -> "DeviceBM25":
        """Adopt a bm25s score matrix (``BM25.scores``: data fp32, indices int32, indptr) - optionally only the
        postings of docs ``[lo, hi)`` (doc-range sharding; rows are rebased to lo)."""
        self = cls(k1, b, "lucene", device)
        self.vocab_dict = dict(vocab_dict or {})
        self._set(data, indices, indptr, num_docs)
        return self.shard(*doc_range) if doc_range is not None else self

    def index(self, corpus_tokens, vocab: Optional[Dict[str, int]] = None) -> "DeviceBM25":
        """``BM25.index(tokens)`` (index.py:140).  ``corpus_tokens``: list of token lists (str -> the vocabulary is
        built in first-seen order) or of token-id lists together with ``vocab`` (or an int vocabulary size)."""
        if len(corpus_tokens) and len(corpus_tokens) and any(len(d) and isinstance(d[0], str) for d in corpus_tokens):
            vd: Dict[str, int] = {}
            ids = [[vd.setdefault(t, len(vd)) for t in doc] for doc in corpus_tokens]
            self.vocab_dict, n_vocab = vd, len(vd)
        else:
            ids = corpus_tokens
            if isinstance(vocab, dict):
                self.vocab_dict, n_vocab = dict(vocab), len(vocab)
            else:
                n_vocab = int(vocab) if vocab is not None else (max((max(d) for d in ids if len(d)), default=-1) + 1)
                self.vocab_dict = {}
        lens = np.fromiter((len(d) for d in ids), dtype=np.int64, count=len(ids))
        flat = np.fromiter((t for d in ids for t in d), dtype=np.int64, count=int(lens.sum()))
        return self.index_flat(torch.from_numpy(flat), torch.from_numpy(lens), n_vocab)

    def index_flat(self, token_ids: torch.Tensor, doc_lens: torch.Tensor, n_vocab: int) -> "DeviceBM25":
        """Index a corpus given as one flat token-id tensor [T] plus per-doc token counts [N] (host or device)."""
        dev = self.device
        tok = token_ids.to(dev, torch.int64)
        lens = doc_lens.to(dev, torch.int64)
        n_docs = int(lens.numel())
        if n_docs == 0 or int(lens.sum().item()) == 0:
            raise ValueError("cannot index an empty corpus")
        doc = torch.repeat_interleave(torch.arange(n_docs, device=dev), lens)
        key = tok * n_docs + doc                                   # token-major, doc-minor: the CSC order
        uniq, tf = torch.unique(key, return_counts=True)           # sorted: postings in (token, doc) order
        p_tok = torch.div(uniq, n_docs, rounding_mode="floor")
        p_doc = uniq - p_tok * n_docs
        df = torch.bincount(p_tok, minlength=n_vocab)
        indptr = torch.zeros(n_vocab + 1, dtype=torch.int64, device=dev)
        indptr[1:] = torch.cumsum(df, 0)
        l_avg = float(lens.double().mean().item())
        data = torch.empty(uniq.numel(), dtype=torch.float32, device=dev)
        p_tok32, p_doc32, tf32 = p_tok.int().contiguous(), p_doc.int().contiguous(), tf.int().contiguous()
        df32, len32 = df.int().contiguous(), lens.int().contiguous()
        nv.check(nv.lib().mfar_bm25_build_scores(nv.ptr(p_tok32), nv.ptr(p_doc32), nv.ptr(tf32), uniq.numel(),
                                                 nv.ptr(df32), nv.ptr(len32), n_docs, l_avg, self.k1, self.b,
                                                 nv.ptr(data), nv.stream()), "bm25_build_scores")
        return self._set(data, p_doc32, indptr, n_docs)

    def shard(self, lo: int, hi: int) -> "DeviceBM25":
        """A new index holding the postings of docs [lo, hi) of this one, rows rebased to lo."""
        s = self.scores
        keep = (s["indices"] >= lo) & (s["indices"] < hi)
        c = torch.zeros(keep.numel() + 1, dtype=torch.int64, device=self.device)
        c[1:] = torch.cumsum(keep, 0)
        out = DeviceBM25(self.k1, self.b, self.method, self.device)
        out.vocab_dict = self.vocab_dict
        out._set(s["data"][keep], s["indices"][keep] - lo, c[s["indptr"]], hi - lo, self.doc_base + lo)
        return out

    # ------------------------------------------------------------------ bm25s on-disk layout (index.py:147-157)
    _FILES = {"data": "data.csc.index.npy", "indices": "indices.csc.index.npy", "indptr": "indptr.csc.index.npy"}

    def save(self, save_dir: str) -> None:
        os.makedirs(save_dir, exist_ok=True)
        for k, fn in self._FILES.items():
            arr = self.scores[k].cpu().numpy()
            np.save(os.path.join(save_dir, fn), arr.astype(np.int32) if k == "indptr" and arr[-1] < 2**31 else arr)
        with open(os.path.join(save_dir, "vocab.index.json"), "w") as f:
            json.dump(self.vocab_dict, f)
        with open(os.path.join(save_dir, "params.index.json"), "w") as f:
            json.dump({"k1": self.k1, "b": self.b, "delta": 0.5, "method": self.method, "idf_method": self.method,
                       "dtype": "float32", "int_dtype": "int32", "num_docs": self.num_docs, "version": "0.1.10"}, f)

    @classmethod
    def load(cls, save_dir: str, mmap: bool = False, device="cuda",
             doc_range: Optional[Tuple[int, int]] = None) -> "DeviceBM25":
        with open(os.path.join(save_dir, "params.index.json")) as f:
            params = json.load(f)
        with open(os.path.join(save_dir, "vocab.index.json")) as f:
            vocab = json.load(f)
        arrs = {k: np.load(os.path.join(save_dir, fn), mmap_mode="r" if mmap else None) for k, fn in cls._FILES.items()}
        if params.get("method", "lucene") != "lucene":
            raise ValueError("only method='lucene' indices are supported")
        return cls.from_csc(np.asarray(arrs["data"]), np.asarray(arrs["indices"]), np.asarray(arrs["indptr"]),
                            int(params["num_docs"]), vocab, params.get("k1", 1.2), params.get("b", 0.75), device,
                            doc_range)

    # ------------------------------------------------------------------ scoring
    def get_tokens_ids(self, query_tokens: Sequence[str]) -> List[int]:
        """bm25s ``get_tokens_ids``: tokens that are not in the vocabulary are dropped; repeats are kept."""
        return tokens_to_ids(self.vocab_dict, list(query_tokens))

    def get_scores_batch(self, queries_tokens: Sequence[Sequence]) -> torch.Tensor:
        """fp32 [Q, num_docs] on the device: row q = ``get_scores(queries_tokens[q])``."""
        fs = BM25FieldSet([self])
        ent = fs.entries([queries_tokens])
        return fs.field_scores(ent, len(queries_tokens))[:, 0, : self.num_docs]

    def get_scores(self, query_tokens_single: Sequence) -> np.ndarray:
        """``BM25.get_scores`` (index.py:75): fp32 [num_docs] numpy vector."""
        if not isinstance(query_tokens_single, (list, tuple)):
            raise ValueError("The query_tokens must be a list of tokens.")
        return self.get_scores_batch([query_tokens_single])[0].cpu().numpy()

    def retrieve(self, query_tokens: Sequence[Sequence], k: int = 10, **_ignored) -> Tuple[np.ndarray, np.ndarray]:
        """``BM25.retrieve(query_tokens, k=...)`` (index.py:92,99): (doc rows [Q,k], scores [Q,k]) as numpy,
        sorted descending (ties: ascending row)."""
        if k > self.num_docs:
            raise ValueError(f"k of {k} is larger than the number of available scores, which is {self.num_docs}")
        from ..modeling.retrieval import MultiFieldRetriever
        from ..modeling.weighting import LinearWeights
        if k <= nv.MAX_K:
            r = MultiFieldRetriever(None, LinearWeights(1, 1).to(self.device), top_k=k, n_docs=self.num_docs,
                                    device=self.device, sparse_indices=[self])
            s, i = r.search(None, sparse_tokens=[query_tokens], top_k=k)
            self.last_launches = r.last_launches
            return i.cpu().numpy(), s.cpu().numpy()
        # k above the streaming top-k's 128 (the reference's precompute asks for 150, precompute_bm25s_scores.py:60):
        # score once, then peel the ranking off in passes of <= 128 - each pass is the same streaming top-k kernel over
        # the score rows, the docs already taken are sunk to -inf in between.  Passes come out in rank order.
        Q, n = len(query_tokens), self.num_docs
        ld = (n + 64) // 64 * 64                        # >= 1 padding column past the docs (see the scatter below)
        rows = torch.full((Q, 1, ld), float("-inf"), dtype=torch.float32, device=self.device)
        rows[:, 0, :n] = self.get_scores_batch(query_tokens)
        r = MultiFieldRetriever(None, LinearWeights(1, 1).to(self.device), n_sparse=1, top_k=nv.MAX_K, n_docs=n,
                                device=self.device)
        out_s, out_i, left, launches = [], [], int(k), 0
        while left > 0:
            kk = min(left, nv.MAX_K)
            s, i = r.search(None, sparse=rows, top_k=kk, batch=Q)
            launches += r.last_launches
            out_s.append(s)
            out_i.append(i)
            # an empty slot (id -1) must not index the row: it lands in the last padding column, outside the docs
            rows[:, 0, :].scatter_(1, i.remainder(ld), float("-inf"))
            left -= kk
        self.last_launches = launches
        return torch.cat(out_i, dim=1).cpu().numpy(), torch.cat(out_s, dim=1).cpu().numpy()


class BM25FieldSet:
    """The F_s sparse fields of a retriever as pointer tables for the C ABI (HOST arrays of device pointers)."""

    def __init__(self, fields: Sequence[DeviceBM25]):
        if not len(fields):
            raise ValueError("need at least one BM25 field")
        self.fields = list(fields)
        n = {f.num_docs for f in self.fields}
        if len(n) != 1:
            raise ValueError(f"sparse fields disagree on the shard's doc count: {sorted(n)}")
        self.num_docs = n.pop()
        self.device = self.fields[0].device
        F = len(self.fields)
        self.indptr = (ctypes.c_void_p * F)(*[f.scores["indptr"].data_ptr() for f in self.fields])
        self.indices = (ctypes.c_void_p * F)(*[f.scores["indices"].data_ptr() or None for f in self.fields])
        self.data = (ctypes.c_void_p * F)(*[f.scores["data"].data_ptr() or None for f in self.fields])
        self.vocab = (ctypes.c_int32 * F)(*[f.n_vocab for f in self.fields])
        self._plan: Optional[torch.Tensor] = None
        self.last_launches = 0

    def __len__(self) -> int:
        return len(self.fields)

    def entries_host(self, tokens_per_field: Sequence[Sequence[Sequence]]) -> np.ndarray:
        """tokens_per_field[j][q] = token list (str or vocabulary ids) of query q for sparse field j
        -> int32 [n_entries, 3] rows (query row, field, token id), one per token occurrence."""
        return token_entries([f.vocab_dict for f in self.fields], tokens_per_field)

    def entries(self, tokens_per_field) -> torch.Tensor:
        return torch.from_numpy(self.entries_host(tokens_per_field)).to(self.device)

    def plan(self, n_entries: int) -> torch.Tensor:
        need = nv.lib().mfar_bm25_plan_bytes(n_entries)
        if self._plan is None or self._plan.numel() < need:
            self._plan = torch.empty(need, dtype=torch.uint8, device=self.device)
        return self._plan

    def field_scores(self, entries: torch.Tensor, Q: int) -> torch.Tensor:
        """fp32 [Q, F_s, ld]: per-field BM25 score vectors (``get_scores`` of every (query, field)); ld = num_docs
        rounded up to 8.  One scatter launch per field (weight 1)."""
        nv.require_device(entries, "entries")
        ld = (self.num_docs + 7) // 8 * 8
        out = torch.zeros((Q, len(self.fields), ld), dtype=torch.float32, device=self.device)
        ent = entries.to(torch.int32).contiguous()
        launches = 0
        for j in range(len(self.fields)):
            ej = ent[ent[:, 1] == j].clone()
            if ej.numel() == 0:
                continue
            ej[:, 1] = 0
            view = out[:, j, :]                                    # row stride F_s * ld
            plan = self.plan(ej.shape[0])
            nv.check(nv.lib().mfar_bm25_scores(
                ctypes.byref(self.indptr, j * ctypes.sizeof(ctypes.c_void_p)),
                ctypes.byref(self.indices, j * ctypes.sizeof(ctypes.c_void_p)),
                ctypes.byref(self.data, j * ctypes.sizeof(ctypes.c_void_p)),
                ctypes.byref(self.vocab, j * ctypes.sizeof(ctypes.c_int32)), 1, nv.ptr(ej), ej.shape[0], Q, 0, 0, 0,
                self.num_docs, view.data_ptr(), len(self.fields) * ld, 0, nv.ptr(plan), plan.numel(), nv.stream()),
                "bm25_scores")
            launches += nv.lib().mfar_last_launch_count()
        self.last_launches = launches
        return out
