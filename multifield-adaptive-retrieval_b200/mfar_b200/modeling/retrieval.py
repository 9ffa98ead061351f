"""Multi-field retrieval over the packed corpus: the B200 replacement of
``RetrievalTrainingModule.trec_eval_step`` / ``mask_field`` (mfar/modeling/contrastive.py:669-714).

``PackedCorpus``         - device-resident bf16 (or E4M3 + per-row scale) corpus [tiles][F][128][dim] built from
                           the reference's per-field fp32 memmaps (or any [N,d] slabs)
``MultiFieldRetriever``  - exhaustive fused scoring + mixture + top-k (``search``), the
                           reference-faithful union/rescore pipeline (``union_rescore``), field
                           masking, per-field top-k, QRes emission
"""
from __future__ import annotations

import ctypes
from typing import Dict, List, Optional, Sequence, TextIO, Tuple

import numpy as np
import torch

from .. import _native as nv
from ..data.trec import QRes
from .weighting import LinearWeights

TILE_DOCS = nv.TILE_DOCS
KCHUNK = 64   # the tensor-core path consumes K in 64-element (128-byte) chunks
KCHUNK_E4M3 = 128   # ... and an E4M3 corpus in 128-element (128-byte) chunks
DTYPES = ("bf16", "e4m3")


def _round_up(x: int, m: int) -> int:
    return (x + m - 1) // m * m


def _operand(t: Optional[torch.Tensor], scales: Optional[torch.Tensor], e4m3: bool) -> tuple:
    """Pointer arguments of one operand of an entry point: the tensor, then its row scales on the *_e4m3 twin."""
    return (nv.ptr(t), nv.ptr(scales)) if e4m3 else (nv.ptr(t),)


class PackedCorpus:
    """bf16 corpus in the tile layout the scoring kernels stream (include/mfar_b200.h).

    ``dim`` is zero-padded to a multiple of 64 (dot products are unchanged); queries are padded
    the same way by ``prepare_queries``.

    ``dtype="e4m3"`` stores one E4M3 byte per element (``data`` is uint8, ``dim`` padded to a multiple of 128) and one
    power-of-two fp32 scale per (doc, field) row (``scales``, [tiles][F][128]): half the bytes of bf16, scored at the
    tensor cores' FP8 rate.  The dequantized values are bf16 numbers, so a search equals the bf16 search of the
    dequantized corpus up to fp32 summation order (``mfar_corpus_pack_rows_e4m3`` states the rounding rule)."""

    def __init__(self, n_docs: int, n_fields: int, dim: int, device="cuda", normalize: bool = False,
                 dtype: str = "bf16"):
        if n_docs <= 0 or n_fields <= 0 or dim <= 0:
            raise ValueError("n_docs, n_fields, dim must be positive")
        if dtype not in DTYPES:
            raise ValueError(f"dtype must be one of {DTYPES}, got {dtype!r}")
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("PackedCorpus lives in HBM: device must be CUDA (no CPU path)")
        self.n_docs, self.n_fields, self.dim = int(n_docs), int(n_fields), int(dim)
        self.dtype = dtype
        self.dim_pad = _round_up(self.dim, KCHUNK_E4M3 if self.e4m3 else KCHUNK)
        self.normalize = bool(normalize)
        n_el = nv.lib().mfar_corpus_packed_elems(self.n_docs, self.n_fields, self.dim_pad)
        self.data = torch.zeros(n_el, dtype=torch.uint8 if self.e4m3 else torch.bfloat16, device=self.device)
        # tail rows of the last tile: payload 0, scale 1
        self.scales = (torch.ones(n_el // self.dim_pad, dtype=torch.float32, device=self.device) if self.e4m3
                       else None)

    @property
    def e4m3(self) -> bool:
        return self.dtype == "e4m3"

    # ------------------------------------------------------------------ loading
    def load_rows(self, field: int, row_begin: int, rows: torch.Tensor) -> None:
        """rows: [n, dim] fp32/bf16 tensor (host or device) -> docs [row_begin, row_begin+n) of `field`."""
        if rows.dim() != 2 or rows.shape[1] != self.dim:
            raise ValueError(f"expected [n,{self.dim}] rows, got {tuple(rows.shape)}")
        self._pack(rows.to(self.device, non_blocking=True), self.data, self.scales, row_begin, self.n_docs,
                   self.n_fields, field)

    def _pack(self, rows: torch.Tensor, out: torch.Tensor, scales: Optional[torch.Tensor], row_begin: int, n_docs: int,
              n_fields: int, field: int, what: str = "") -> None:
        """Device rows [n, dim] -> rows [row_begin, row_begin + n) of `field` of the packed layout of an n_docs x
        n_fields corpus in `out` (with their `scales` on an E4M3 corpus), padded to dim_pad.  Inputs other than
        fp32 / bf16 are taken to fp32 first."""
        if rows.dtype not in (torch.float32, torch.bfloat16):
            rows = rows.float()
        if self.dim_pad != self.dim:
            rows = torch.nn.functional.pad(rows, (0, self.dim_pad - self.dim))
        rows = rows.contiguous()
        name = "corpus_pack_rows_e4m3" if self.e4m3 else "corpus_pack_rows"
        nv.check(getattr(nv.lib(), "mfar_" + name)(
            nv.ptr(rows), nv.F32 if rows.dtype == torch.float32 else nv.BF16, rows.shape[0], int(row_begin),
            *_operand(out, scales, self.e4m3), n_docs, n_fields, int(field), self.dim_pad, int(self.normalize),
            nv.stream()), name + what)

    def load_field(self, field: int, vectors, chunk_rows: int = 131072) -> None:
        """vectors: np.memmap / ndarray / tensor [N, dim] (the reference's ``MemoryMapDict.file``)."""
        n = vectors.shape[0]
        if n != self.n_docs:
            raise ValueError(f"field has {n} rows, corpus has {self.n_docs}")
        for lb in range(0, n, chunk_rows):
            ub = min(n, lb + chunk_rows)
            chunk = vectors[lb:ub]
            if not torch.is_tensor(chunk):
                chunk = torch.from_numpy(np.ascontiguousarray(chunk))
            self.load_rows(field, lb, chunk)

    @classmethod
    def from_fields(cls, fields: Sequence, device="cuda", normalize: bool = False, dtype: str = "bf16") -> "PackedCorpus":
        """fields: F array-likes [N, dim], in scorer column order (``resolve_fields`` order)."""
        n, d = fields[0].shape
        pc = cls(n, len(fields), d, device, normalize, dtype)
        for f, v in enumerate(fields):
            pc.load_field(f, v)
        return pc

    @classmethod
    def from_vectors_dict(cls, vectors_dict: Dict[str, "object"], dense_keys: Sequence[str], device="cuda",
                          normalize: bool = False, dtype: str = "bf16") -> "PackedCorpus":
        """vectors_dict: field key -> MemoryMapDict, as returned by ``read_and_create_indices``."""
        return cls.from_fields([vectors_dict[k].file for k in dense_keys], device, normalize, dtype)

    def window(self, doc_begin: int, n_docs: int) -> "PackedCorpus":
        """Docs [doc_begin, doc_begin + n_docs) as a corpus of their own WITHOUT a copy (the layout is tile-major, so a
        window that starts on a 128-doc tile boundary is a pointer offset).  A shard that holds a margin of its neighbours'
        docs can move its boundaries this way (``dist.rebalanced_boundaries``)."""
        if doc_begin % TILE_DOCS or doc_begin < 0 or n_docs <= 0 or doc_begin + n_docs > self.n_docs:
            raise ValueError(f"window [{doc_begin}, {doc_begin + n_docs}) must start on a {TILE_DOCS}-doc tile boundary "
                             f"inside the corpus of {self.n_docs} docs")
        view = PackedCorpus.__new__(PackedCorpus)
        view.device, view.n_fields, view.dim, view.dim_pad = self.device, self.n_fields, self.dim, self.dim_pad
        view.normalize, view.n_docs, view.dtype = self.normalize, int(n_docs), self.dtype
        per_tile = self.n_fields * TILE_DOCS * self.dim_pad
        n_el = nv.lib().mfar_corpus_packed_elems(view.n_docs, self.n_fields, self.dim_pad)
        first = (doc_begin // TILE_DOCS) * per_tile
        view.data = self.data[first:first + n_el]
        view.scales = None
        if self.e4m3:
            first_row = (doc_begin // TILE_DOCS) * self.n_fields * TILE_DOCS
            view.scales = self.scales[first_row:first_row + n_el // self.dim_pad]
        return view

    def unpack_field(self, field: int, row_begin: int = 0, n_rows: Optional[int] = None) -> torch.Tensor:
        n_rows = self.n_docs - row_begin if n_rows is None else n_rows
        out = torch.empty((n_rows, self.dim_pad), dtype=torch.float32, device=self.device)
        # exact on an E4M3 corpus too: every dequantized value is a normal fp32 number
        name = "corpus_unpack_rows_e4m3" if self.e4m3 else "corpus_unpack_rows"
        nv.check(getattr(nv.lib(), "mfar_" + name)(*_operand(self.data, self.scales, self.e4m3), self.n_docs,
                                                   self.n_fields, int(field), self.dim_pad, int(row_begin),
                                                   int(n_rows), nv.ptr(out), nv.stream()), name)
        return out[:, : self.dim]

    def prepare_queries(self, q_vecs):
        """[Q, dim] (any float dtype, host or device) -> contiguous bf16 [Q, dim_pad] on the device.

        On a cosine corpus the queries are normalised by the kernel that packs the docs, so both sides are rounded to
        bf16 once, by the same arithmetic: with one field the packed layout [tile][1][128][dim_pad] of Q rows is plain
        row-major [Q, dim_pad].  Inputs other than fp32 / bf16 are taken to fp32 first, as in ``load_rows``.

        On an E4M3 corpus the queries are quantized by the kernel that packs the docs, by the same rule, and the call
        returns (uint8 payload [Q, dim_pad], fp32 scales [Q])."""
        if not torch.is_tensor(q_vecs):
            q_vecs = torch.from_numpy(np.ascontiguousarray(q_vecs))
        if q_vecs.dim() != 2 or q_vecs.shape[1] != self.dim:
            raise ValueError(f"expected [Q,{self.dim}] query vectors, got {tuple(q_vecs.shape)}")
        q = q_vecs.to(self.device)
        if self.e4m3 or self.normalize:
            out = torch.empty((q.shape[0], self.dim_pad), dtype=self.data.dtype, device=self.device)
            qs = torch.empty((q.shape[0],), dtype=torch.float32, device=self.device) if self.e4m3 else None
            if q.shape[0]:
                self._pack(q, out, qs, 0, q.shape[0], 1, 0, " (queries)")
            return (out, qs) if self.e4m3 else out
        q = q.to(torch.bfloat16)
        if self.dim_pad != self.dim:
            q = torch.nn.functional.pad(q, (0, self.dim_pad - self.dim))
        return q.contiguous()


class MultiFieldRetriever:
    """Scores every doc of a shard under all fields, mixes, keeps the top-k - one corpus pass.

    Field order everywhere (W columns, mask rows, weights) is dense fields then sparse fields,
    as ``resolve_fields`` produces (schema.py:130-134)."""

    def __init__(self, corpus: Optional[PackedCorpus], mixture: LinearWeights, n_sparse: int = 0, top_k: int = 100,
                 doc_id_base: int = 0, n_docs: Optional[int] = None, impl: str = "auto",
                 numeric_ids_to_keys: Optional[Sequence[str]] = None, device=None, sparse_indices=None):
        """``sparse_indices``: the shard's ``DeviceBM25`` indices, one per sparse field in field order; with them the
        sparse fields are scored on the device from query tokens (``sparse_tokens=``) and ``n_sparse`` is implied."""
        self.corpus = corpus
        self.n_dense = corpus.n_fields if corpus is not None else 0
        self.bm25 = None
        if sparse_indices is not None and len(sparse_indices):
            from ..data.bm25 import BM25FieldSet
            self.bm25 = BM25FieldSet(sparse_indices)
            n_sparse = len(sparse_indices)
            if n_docs is None and corpus is None:
                n_docs = self.bm25.num_docs
        self.n_sparse = int(n_sparse)
        self.n_docs = corpus.n_docs if corpus is not None else int(n_docs)
        self.device = corpus.device if corpus is not None else torch.device(device or "cuda")
        if self.bm25 is not None and self.bm25.num_docs != self.n_docs:
            raise ValueError(f"BM25 indices hold {self.bm25.num_docs} docs, the shard {self.n_docs}")
        self.mixture = mixture
        if mixture.num_fields != self.n_dense + self.n_sparse:
            raise ValueError(f"mixture has {mixture.num_fields} fields, retriever {self.n_dense}+{self.n_sparse}")
        self.top_k = int(top_k)
        self.doc_id_base = int(doc_id_base)
        self.impl = impl
        self.numeric_ids_to_keys = numeric_ids_to_keys
        self.mask = torch.ones([self.num_fields, 1], device=self.device)      # contrastive.py:270
        self.masked_fields_string = ""
        self._ws: Optional[torch.Tensor] = None
        self._host_scratch: Optional[torch.Tensor] = None
        self.last_launches = 0

    @property
    def num_fields(self) -> int:
        return self.n_dense + self.n_sparse

    # ------------------------------------------------------------------ masking (contrastive.py:706-714)
    def mask_field(self, field_idx_list: Sequence[int], field_names: Optional[Sequence[str]] = None) -> None:
        mask = torch.ones([self.num_fields, 1], device=self.device)
        mask[list(field_idx_list)] = 0
        self.mask = mask
        if field_names is not None:
            self.masked_fields_string = ",".join(field_names[i] for i in field_idx_list)

    def mixture_input(self, q_vecs, q_emb=None) -> Optional[torch.Tensor]:
        """The fp32 [Q,E] device input of a query-conditioned mixture (None for static weights).  ``q_emb`` defaults to
        the query vectors, as in the reference where both come from the same encoder (contrastive.py:688-694); on a
        cosine corpus that encoder ends in ``Normalize()``, so its output ``x_encoded`` - and the default here - is the
        unit-normalised query."""
        if not self.mixture.query_cond:
            return None
        if q_emb is not None:
            return q_emb.to(self.device).float()
        qv = q_vecs if torch.is_tensor(q_vecs) else torch.from_numpy(np.ascontiguousarray(q_vecs))
        qe = qv.to(self.device).float()
        if self.corpus is not None and self.corpus.normalize:
            qe = torch.nn.functional.normalize(qe, p=2, dim=1)
        return qe

    # ------------------------------------------------------------------ internals
    def _workspace(self, Q: int, k: int, n_sparse: int, n_docs: Optional[int] = None,
                   n_entries: int = 0) -> torch.Tensor:
        need = nv.lib().mfar_score_topk_bm25_workspace_bytes(Q, k, self.n_docs if n_docs is None else n_docs,
                                                             n_sparse, n_entries)
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        return self._ws

    def _check_sparse(self, sparse: Optional[torch.Tensor], Q: int) -> Tuple[Optional[torch.Tensor], int]:
        if self.n_sparse == 0:
            return None, nv.F16
        if sparse is None:
            raise ValueError(f"retriever has {self.n_sparse} sparse fields: pass their precomputed scores [Q,Fs,N]")
        nv.require_device(sparse, "sparse")
        if sparse.dim() != 3 or tuple(sparse.shape[:2]) != (Q, self.n_sparse) or sparse.shape[2] < self.n_docs:
            raise ValueError(f"sparse must be [{Q},{self.n_sparse},>={self.n_docs}], got {tuple(sparse.shape)}")
        if sparse.dtype not in (torch.float16, torch.float32):
            sparse = sparse.float()
        return sparse.contiguous(), (nv.F16 if sparse.dtype == torch.float16 else nv.F32)

    def _queries(self, q_vecs) -> Tuple[Optional[torch.Tensor], Optional[torch.Tensor]]:
        """(query operand, query scales) of a call: bf16 rows and None, or E4M3 rows and their fp32 scales."""
        if self.corpus is None:
            return None, None
        q = self.corpus.prepare_queries(q_vecs)
        return q if self.corpus.e4m3 else (q, None)

    def _require_bf16(self, what: str) -> None:
        if self.corpus is not None and self.corpus.e4m3:
            raise ValueError(f"{what} runs on a bf16 corpus only; this corpus is E4M3 (use search / score_candidates)")

    def _check_sparse_coo(self, sparse_coo) -> Tuple[torch.Tensor, torch.Tensor, Sequence[int]]:
        if self.n_sparse == 0:
            raise ValueError("retriever has no sparse fields")
        ck, cv, off = sparse_coo
        nv.require_device(ck, "sparse_coo keys"); nv.require_device(cv, "sparse_coo vals")
        if ck.dtype != torch.int32 or ck.dim() != 2 or ck.shape[1] != 2 or cv.shape[0] != ck.shape[0]:
            raise ValueError("sparse_coo keys must be int32 [nnz,2] with one value per row")
        if len(off) != self.n_sparse + 1 or int(off[-1]) != ck.shape[0]:
            raise ValueError("field_offsets must have n_sparse+1 entries ending at nnz")
        if cv.dtype not in (torch.float16, torch.float32):
            cv = cv.float()
        return ck.contiguous(), cv.contiguous(), off

    def _check_filter(self, doc_filter, Q: int) -> Optional[Tuple[torch.Tensor, int, int]]:
        """(bitmap, rows, words per row) of a ``doc_filter`` argument, or None.  The bitmap is used in place (a
        ``GraphedSearch`` replays with whatever it holds), so it must already be a contiguous device tensor."""
        if doc_filter is None:
            return None
        dev = self.device                                  # "cuda" (no index) accepts the current device's tensors
        if not torch.is_tensor(doc_filter) or doc_filter.device.type != dev.type or (
                dev.index is not None and doc_filter.device.index != dev.index):
            raise ValueError(f"doc_filter must be a tensor on {self.device}")
        if doc_filter.dtype not in (torch.int32, torch.uint32):
            raise ValueError(f"doc_filter must be int32 or uint32 (a bitmap over global doc ids), got {doc_filter.dtype}")
        if doc_filter.dim() == 1:
            rows = 1
        elif doc_filter.dim() == 2 and doc_filter.shape[0] == Q:
            rows = Q
        else:
            raise ValueError(f"doc_filter must be [W] (shared) or [{Q},W] (one row per query), "
                             f"got {tuple(doc_filter.shape)}")
        if not doc_filter.is_contiguous():
            raise ValueError("doc_filter must be contiguous")
        ld = int(doc_filter.shape[-1])
        need = (self.doc_id_base + self.n_docs + 31) // 32
        if ld < need:
            raise ValueError(f"doc_filter rows hold {ld} words; docs [{self.doc_id_base}, "
                             f"{self.doc_id_base + self.n_docs}) need {need}")
        return doc_filter, rows, ld

    def _score_topk(self, q: Tuple[Optional[torch.Tensor], Optional[torch.Tensor]], w: torch.Tensor, sparse: tuple,
                    k: int, field_begin: int, n_dense: int, n_sparse: int, want_keys: bool = False,
                    impl: Optional[str] = None, n_docs: Optional[int] = None, doc_id_base: Optional[int] = None,
                    doc_filter: Optional[Tuple[torch.Tensor, int, int]] = None):
        """``q``: the query operand of ``_queries`` (rows, scales).  ``sparse``: the sparse fields' input in one of
        the layouts of the scoring entry points - ("rows", [Q,Fs,ld] tensor or None, dtype code),
        ("coo", keys, vals, field_offsets) or ("bm25", int32 [n,3] token entries).  ``doc_filter``: the output of
        ``_check_filter`` - the call then runs the ``*_filtered`` twin."""
        Q = w.shape[0]
        n_docs = self.n_docs if n_docs is None else n_docs
        doc_id_base = self.doc_id_base if doc_id_base is None else doc_id_base
        if k > n_docs:
            raise RuntimeError(f"selected index k out of range (k={k}, docs={n_docs})")   # torch.topk's error
        scores = torch.empty((Q, k), dtype=torch.float32, device=self.device)
        ids = torch.empty((Q, k), dtype=torch.int64, device=self.device)
        keys = torch.empty((Q, k), dtype=torch.int64, device=self.device) if want_keys else None
        layout, *sp = sparse
        n_entries = 0
        if layout == "bm25":
            (ent,) = sp
            n_entries = ent.shape[0]
            b = self.bm25
            sparse_args = (b.indptr, b.indices, b.data, b.vocab, n_sparse, nv.ptr(ent), n_entries)
        elif layout == "coo":
            ck, cv, off = sp
            off = (ctypes.c_int64 * (n_sparse + 1))(*[int(x) for x in off])      # host array, alive through the call
            sparse_args = (nv.ptr(ck), nv.ptr(cv), nv.F16 if cv.dtype == torch.float16 else nv.F32,
                           ctypes.addressof(off), n_sparse)
        else:
            t, code = sp
            sparse_args = (nv.ptr(t), n_sparse, code, t.shape[2] if t is not None else n_docs)
        ws = self._workspace(Q, k, n_sparse, n_docs, n_entries)
        c = self.corpus
        e8 = c is not None and c.e4m3
        name = ("score_topk" if layout == "rows" else "score_topk_" + layout) + ("_e4m3" if e8 else "")
        filt_args = ()
        if doc_filter is not None:
            name += "_filtered"
            bits, rows, ld = doc_filter
            filt_args = (nv.ptr(bits), rows, ld)
        fn = getattr(nv.lib(), "mfar_" + name)
        nv.check(fn(*_operand(c.data if c else None, c.scales if c else None, e8), n_docs, c.n_fields if c else 0,
                    field_begin, n_dense, c.dim_pad if c else 0, *_operand(*q, e8), Q, nv.ptr(w), *sparse_args,
                    doc_id_base, *filt_args, k, nv.ptr(keys), nv.ptr(scores), nv.ptr(ids), nv.ptr(ws), ws.numel(),
                    nv.IMPL[impl or self.impl], nv.stream()), name)
        self.last_launches = nv.lib().mfar_last_launch_count()
        return scores, ids, keys

    def _bm25_entries(self, sparse_tokens) -> torch.Tensor:
        if self.bm25 is None:
            raise ValueError("sparse_tokens needs a retriever built with sparse_indices=[DeviceBM25, ...]")
        if torch.is_tensor(sparse_tokens):
            nv.require_device(sparse_tokens, "sparse_tokens")
            if sparse_tokens.dtype != torch.int32 or sparse_tokens.dim() != 2 or sparse_tokens.shape[1] != 3:
                raise ValueError("entry tensor must be int32 [n,3] = (query row, sparse field, token id)")
            return sparse_tokens.contiguous()
        return self.bm25.entries(sparse_tokens)

    @staticmethod
    def _batch_size(q_bf16, sparse, sparse_tokens, batch: Optional[int]) -> int:
        """Number of queries of a call.  A prebuilt int32 [n,3] entry tensor does not carry it (trailing queries may
        have no tokens at all): a sparse-only retriever fed with one needs ``batch=``."""
        if q_bf16 is not None:
            return int(q_bf16.shape[0])
        if sparse is not None:
            return int(sparse.shape[0])
        if batch is not None:
            return int(batch)
        if sparse_tokens is not None and not torch.is_tensor(sparse_tokens):
            return len(sparse_tokens[0])
        raise ValueError("cannot infer the batch size: pass batch= (sparse-only retriever with an entry tensor)")

    def _sparse_from_tokens(self, sparse, sparse_tokens, q_bf16, batch: Optional[int] = None) -> Optional[torch.Tensor]:
        """Per-field score tensor [Q,F_s,ld] from query tokens when the sparse fields are BM25 indices."""
        if sparse_tokens is None:
            return sparse
        return self.bm25_field_scores(sparse_tokens, self._batch_size(q_bf16, None, sparse_tokens, batch))

    def bm25_field_scores(self, sparse_tokens, Q: int) -> torch.Tensor:
        """fp32 [Q, F_s, ld>=N]: what ``get_scores`` returns for every (query, sparse field), on the device."""
        out = self.bm25.field_scores(self._bm25_entries(sparse_tokens), Q)
        self.last_launches = self.bm25.last_launches
        return out

    # ------------------------------------------------------------------ exhaustive fused search
    @torch.no_grad()
    def search(self, q_vecs, q_emb: Optional[torch.Tensor] = None, sparse: Optional[torch.Tensor] = None,
               top_k: Optional[int] = None, return_keys: bool = False, impl: Optional[str] = None, sparse_coo=None,
               sparse_tokens=None, batch: Optional[int] = None, doc_filter: Optional[torch.Tensor] = None):
        """Exhaustive multi-field top-k.

        q_vecs [Q,dim]: query vectors for the dense dots (rounded to bf16);
        q_emb  [Q,E]  : fp32 query embedding for the mixture softmax (defaults to q_vecs - unit-normalised on a
                        cosine corpus - as in the reference where both come from the same encoder,
                        contrastive.py:688-694; ``mixture_input``);
        sparse [Q,Fs,ld>=N]: precomputed per-field BM25 scores of this shard's docs (f16/f32).  With a 32-byte aligned row
                        pitch (``ld`` a multiple of 16 for f16, 8 for f32) the rows are gathered and mixed INSIDE the
                        scoring epilogue; otherwise a pre-mix kernel writes a [Q,N] fp32 block first.
        sparse_coo     : instead of ``sparse``: (keys int32 [nnz,2] = (query row, GLOBAL doc row), vals f16/f32 [nnz],
                        field_offsets [Fs+1]) on the device - the reference's precomputed-BM25 layout
                        (``PrecomputedSparseScores.batch``); pairs that are absent score 0 (index.py:120-125).
        sparse_tokens  : instead of ``sparse`` when the retriever holds BM25 indices (``sparse_indices=``): the query
                        tokens, either ``tokens[j][q]`` = token list (str or vocabulary ids) of query q for sparse
                        field j, or the prebuilt int32 [n,3] entry tensor of ``BM25FieldSet.entries`` - the sparse
                        fields are then scored on the device (bm25s ``get_scores``, index.py:72-76).
        batch          : number of queries, needed only for a sparse-only retriever fed with an entry tensor.
        doc_filter     : restrict the top-k to eligible docs: an int32/uint32 device bitmap over GLOBAL doc ids (bit d
                        of word d >> 5 set <=> doc d is eligible; ``data.bm25.safe_docs_bitmap`` builds one row), either
                        one row [W] for every query or one row per query [Q,W], with 32*W >= doc_id_base + n_docs.
                        Ineligible docs never enter the top-k, inside the scoring pass; a query with fewer than k
                        eligible docs gets (-inf, -1) in the remaining slots.
        Returns (scores [Q,k] fp32, ids [Q,k] int64) sorted by (score desc, id asc), NaN scores first (as
        ``torch.topk`` ranks them), then +inf, finite, -inf; with
        return_keys also the packed uint64 keys (as int64) used for cross-shard merging."""
        k = top_k or self.top_k
        q_bf16, q_sc = self._queries(q_vecs)
        if q_bf16 is None and sparse is None and batch is None and q_emb is not None and (
                sparse_tokens is None or torch.is_tensor(sparse_tokens)):
            batch = int(q_emb.shape[0])
        Q = self._batch_size(q_bf16, sparse, sparse_tokens, batch)
        qe = self.mixture_input(q_vecs, q_emb)
        w = self.mixture.field_weights(qe, self.mask, batch=Q)
        if sparse_tokens is not None:
            sp = ("bm25", self._bm25_entries(sparse_tokens))
        elif sparse_coo is not None:
            sp = ("coo", *self._check_sparse_coo(sparse_coo))
        else:
            sp = ("rows", *self._check_sparse(sparse, Q))
        scores, ids, keys = self._score_topk((q_bf16, q_sc), w, sp, k, 0, self.n_dense, self.n_sparse,
                                             want_keys=return_keys, impl=impl,
                                             doc_filter=self._check_filter(doc_filter, Q))
        return (scores, ids, keys) if return_keys else (scores, ids)

    # ------------------------------------------------------------------ field-masking sweep in one corpus pass
    @staticmethod
    def mask_sweep_plan(field_info) -> List[Tuple[str, List[int]]]:
        """The evaluations ``mask_fields`` runs one after another, each a full pass with the corpus re-encoded
        (mfar/commands/mask_fields.py:142-170): baseline, every single field, all sparse, all dense, every field name.
        Returns (label, masked field indices) in that order (names sorted; the reference iterates a set)."""
        from ..data.typedef import FieldType
        fields = list(field_info.values())
        plan: List[Tuple[str, List[int]]] = [("baseline", [])]
        plan += [(f"field:{k}", [i]) for i, k in enumerate(field_info.keys())]
        sparse_idx = [i for i, f in enumerate(fields) if f.field_type == FieldType.SPARSE]
        dense_idx = [i for i, f in enumerate(fields) if f.field_type == FieldType.DENSE]
        if sparse_idx:
            plan.append(("all_sparse", sparse_idx))
        if dense_idx:
            plan.append(("all_dense", dense_idx))
        for name in sorted({f.name for f in fields}):
            plan.append((f"name:{name}", [i for i, f in enumerate(fields) if f.name == name]))
        return plan

    @torch.no_grad()
    def search_mask_sweep(self, q_vecs, masked_sets: Sequence[Sequence[int]], q_emb: Optional[torch.Tensor] = None,
                          sparse: Optional[torch.Tensor] = None, top_k: Optional[int] = None,
                          max_rows: int = 1024, sparse_tokens=None, batch: Optional[int] = None
                          ) -> Tuple[torch.Tensor, torch.Tensor]:
        """All M maskings of ``mask_field`` evaluated as extra weight rows of ONE fused pass per chunk: the mask only
        multiplies the softmax weights (contrastive.py:686, no renormalisation), so masking m of query q is the
        pseudo-query (q, w[q] * mask_m).  Returns (scores [M,Q,k], ids [M,Q,k]).  Rows are processed in chunks of
        at most ``max_rows`` pseudo-queries; dense sparse-score tensors are repeated per chunk, BM25 token entries
        (``sparse_tokens``, for a retriever with ``sparse_indices``) are replicated with shifted query rows."""
        k = top_k or self.top_k
        q_bf16, q_sc = self._queries(q_vecs)
        ent = self._bm25_entries(sparse_tokens) if sparse_tokens is not None else None
        Q = self._batch_size(q_bf16, sparse, sparse_tokens, batch)
        qe = self.mixture_input(q_vecs, q_emb)
        w = self.mixture.field_weights(qe, None, batch=Q)                      # [Q,F] unmasked softmax weights
        M = len(masked_sets)
        masks = torch.ones((M, self.num_fields), dtype=torch.float32, device=self.device)
        for m, idx in enumerate(masked_sets):
            masks[m, list(idx)] = 0
        sp, code = self._check_sparse(sparse, Q) if ent is None else (None, nv.F16)
        out_s = torch.empty((M, Q, k), dtype=torch.float32, device=self.device)
        out_i = torch.empty((M, Q, k), dtype=torch.int64, device=self.device)
        per_chunk = max(1, max_rows // Q)
        for m0 in range(0, M, per_chunk):
            m1 = min(M, m0 + per_chunk)
            reps = m1 - m0
            w_rows = (w.unsqueeze(0) * masks[m0:m1].unsqueeze(1)).reshape(reps * Q, -1).contiguous()
            q_rows = q_bf16.repeat(reps, 1) if q_bf16 is not None else None
            qs_rows = q_sc.repeat(reps) if q_sc is not None else None
            if ent is not None:                                            # query-major order is kept: rep-major
                ent_rows = ent.unsqueeze(0).repeat(reps, 1, 1)
                ent_rows[:, :, 0] += (torch.arange(reps, device=self.device, dtype=torch.int32) * Q).view(reps, 1)
                sp_rows = ("bm25", ent_rows.view(-1, 3).contiguous())
            else:
                sp_rows = ("rows", sp.repeat(reps, 1, 1) if sp is not None else None, code)
            s, i, _ = self._score_topk((q_rows, qs_rows), w_rows, sp_rows, k, 0, self.n_dense, self.n_sparse)
            out_s[m0:m1] = s.view(reps, Q, k)
            out_i[m0:m1] = i.view(reps, Q, k)
        return out_s, out_i

    # ------------------------------------------------------------------ host-buffer end-to-end call
    def search_host(self, q_vecs_host: torch.Tensor, q_emb_host: Optional[torch.Tensor] = None,
                    sparse_host: Optional[torch.Tensor] = None, top_k: Optional[int] = None,
                    out_scores: Optional[torch.Tensor] = None, out_ids: Optional[torch.Tensor] = None,
                    impl: Optional[str] = None):
        """One C-ABI call with HOST buffers (``mfar_search_host``): H2D of the batch, mixture weights,
        fused scoring + top-k, D2H of the [Q,k] result, stream sync.  q_vecs_host: bf16 [Q,dim_pad] host tensor
        (pinned for full PCIe speed); q_emb_host fp32 [Q,E]; sparse_host f16/f32 [Q,Fs,N].  bf16 corpus only."""
        self._require_bf16("search_host")
        c = self.corpus
        Q = q_vecs_host.shape[0] if q_vecs_host is not None else sparse_host.shape[0]
        if c is not None and (q_vecs_host.dtype != torch.bfloat16 or q_vecs_host.shape[1] != c.dim_pad
                              or q_vecs_host.is_cuda):
            raise ValueError("q_vecs_host must be a host bf16 [Q, dim_pad] tensor")
        if self.mixture.query_cond and (q_emb_host is None or q_emb_host.dtype != torch.float32):
            raise ValueError("q_emb_host must be a host fp32 [Q,E] tensor")
        code = nv.F16
        if self.n_sparse:
            if tuple(sparse_host.shape) != (Q, self.n_sparse, self.n_docs) or not sparse_host.is_contiguous():
                raise ValueError(f"sparse_host must be a contiguous [{Q},{self.n_sparse},{self.n_docs}] host tensor")
            code = nv.F16 if sparse_host.dtype == torch.float16 else nv.F32
        return self._search_host("search_host", Q, q_vecs_host, q_emb_host, (nv.ptr(sparse_host), self.n_sparse, code),
                                 code, top_k, out_scores, out_ids, impl)

    def search_host_bm25(self, q_vecs_host: Optional[torch.Tensor], q_emb_host: Optional[torch.Tensor],
                         entries_host: torch.Tensor, top_k: Optional[int] = None,
                         out_scores: Optional[torch.Tensor] = None, out_ids: Optional[torch.Tensor] = None,
                         impl: Optional[str] = None, batch: Optional[int] = None):
        """``search_host`` for a retriever whose sparse fields are device-resident BM25 indices
        (``mfar_search_host_bm25``): per batch only the query vectors / embedding and the int32 [n,3] token entries
        (``BM25FieldSet.entries_host``, ideally pinned) cross PCIe."""
        if self.bm25 is None:
            raise ValueError("search_host_bm25 needs a retriever built with sparse_indices=[DeviceBM25, ...]")
        self._require_bf16("search_host_bm25")
        c = self.corpus
        if q_vecs_host is not None:
            Q = q_vecs_host.shape[0]
        elif q_emb_host is not None:
            Q = q_emb_host.shape[0]
        else:
            Q = int(batch)
        if c is not None and (q_vecs_host.dtype != torch.bfloat16 or q_vecs_host.shape[1] != c.dim_pad
                              or q_vecs_host.is_cuda):
            raise ValueError("q_vecs_host must be a host bf16 [Q, dim_pad] tensor")
        if self.mixture.query_cond and (q_emb_host is None or q_emb_host.dtype != torch.float32):
            raise ValueError("q_emb_host must be a host fp32 [Q,E] tensor")
        if entries_host.is_cuda or entries_host.dtype != torch.int32 or entries_host.dim() != 2 \
                or entries_host.shape[1] != 3 or not entries_host.is_contiguous():
            raise ValueError("entries_host must be a contiguous host int32 [n,3] tensor")
        n_ent = entries_host.shape[0]
        b = self.bm25
        return self._search_host("search_host_bm25", Q, q_vecs_host, q_emb_host,
                                 (b.indptr, b.indices, b.data, b.vocab, self.n_sparse,
                                  nv.ptr(entries_host) if n_ent else 0, n_ent),
                                 n_ent, top_k, out_scores, out_ids, impl)

    def _search_host(self, entry: str, Q: int, q_vecs_host, q_emb_host, sparse_args: tuple, sizing: int,
                     top_k: Optional[int], out_scores: Optional[torch.Tensor], out_ids: Optional[torch.Tensor],
                     impl: Optional[str]):
        """The call of ``mfar_<entry>`` with the batch's sparse-field arguments ``sparse_args``.  ``sizing`` is the
        sparse argument of ``mfar_<entry>_scratch_bytes``: the score dtype, or the number of token entries."""
        k = top_k or self.top_k
        c = self.corpus
        E = self.mixture.weight.shape[0] if self.mixture.query_cond else 0
        need = getattr(nv.lib(), f"mfar_{entry}_scratch_bytes")(Q, c.dim_pad if c else 0, E, self.n_dense,
                                                                self.n_sparse, self.n_docs, sizing, k)
        if self._host_scratch is None or self._host_scratch.numel() < need:
            self._host_scratch = torch.empty(need, dtype=torch.uint8, device=self.device)
        if out_scores is None:
            out_scores = torch.empty((Q, k), dtype=torch.float32).pin_memory()
        if out_ids is None:
            out_ids = torch.empty((Q, k), dtype=torch.int64).pin_memory()
        W = self.mixture.weight.detach().contiguous().float()
        m = self.mask.reshape(-1).contiguous().float()
        nv.check(getattr(nv.lib(), "mfar_" + entry)(
            nv.ptr(c.data) if c else 0, self.n_docs, c.n_fields if c else 0, 0, self.n_dense, c.dim_pad if c else 0,
            nv.ptr(q_vecs_host), nv.ptr(q_emb_host), Q, E, nv.ptr(W), nv.ptr(m), int(self.mixture.query_cond),
            *sparse_args, self.doc_id_base, k, nv.ptr(out_scores), nv.ptr(out_ids), nv.ptr(self._host_scratch),
            self._host_scratch.numel(), nv.IMPL[impl or self.impl], nv.stream()), entry)
        self.last_launches = nv.lib().mfar_last_launch_count()
        return out_scores, out_ids

    # ------------------------------------------------------------------ per-field top-k (index.py:181-222)
    @torch.no_grad()
    def per_field_topk(self, q_vecs, sparse: Optional[torch.Tensor] = None, top_k: Optional[int] = None,
                       zero_init: bool = True, sparse_tokens=None, batch: Optional[int] = None
                       ) -> Tuple[torch.Tensor, torch.Tensor]:
        """What ``index.retrieve_batch(queries, top_k)`` returns for every field, in field order:
        (scores [F,Q,k], rows [F,Q,k]).  Dense fields reproduce the reference's (0.0, row 0) running-top-k
        initialisation (index.py:192-193) when zero_init is set."""
        k = top_k or self.top_k
        q_bf16, q_sc = self._queries(q_vecs)
        sparse = self._sparse_from_tokens(sparse, sparse_tokens, q_bf16, batch)
        Q = self._batch_size(q_bf16, sparse, None, batch)
        sp, code = self._check_sparse(sparse, Q)
        ones = torch.ones((Q, 1), dtype=torch.float32, device=self.device)
        all_s, all_i, launches = [], [], 0
        for f in range(self.n_dense):
            s, i, _ = self._score_topk((q_bf16, q_sc), ones, ("rows", None, nv.F16), k, f, 1, 0)
            launches += self.last_launches
            i = i - self.doc_id_base
            if zero_init:
                nv.check(nv.lib().mfar_topk_apply_zero_init(nv.ptr(s), nv.ptr(i), Q, k, nv.stream()), "zero_init")
                launches += 1
            all_s.append(s)
            all_i.append(i)
        for j in range(self.n_sparse):
            sj = sp[:, j:j + 1, :].contiguous()
            s, i, _ = self._score_topk((None, None), ones, ("rows", sj, code), k, 0, 0, 1)
            launches += self.last_launches
            all_s.append(s)
            all_i.append(i - self.doc_id_base)
        self.last_launches = launches
        return torch.stack(all_s), torch.stack(all_i)

    # ------------------------------------------------------------------ candidate re-scoring (index.py:227-232)
    @torch.no_grad()
    def score_candidates(self, q_vecs, rows: torch.Tensor, sparse: Optional[torch.Tensor] = None,
                         sparse_tokens=None, batch: Optional[int] = None) -> torch.Tensor:
        """Per-field scores of the given local rows: [F, Q, C] (rows < 0 -> 0, index.py:112-117)."""
        q_bf16, q_sc = self._queries(q_vecs)
        sparse = self._sparse_from_tokens(sparse, sparse_tokens, q_bf16, batch)
        Q = self._batch_size(q_bf16, sparse, None, batch)
        rows = rows.to(self.device, dtype=torch.int64).contiguous()
        C = rows.numel()
        out = torch.zeros((self.num_fields, Q, C), dtype=torch.float32, device=self.device)
        if self.n_dense and C:
            c = self.corpus
            name = "score_candidates_e4m3" if c.e4m3 else "score_candidates"
            nv.check(getattr(nv.lib(), "mfar_" + name)(*_operand(c.data, c.scales, c.e4m3), self.n_docs, c.n_fields, 0,
                                                       self.n_dense, c.dim_pad, *_operand(q_bf16, q_sc, c.e4m3), Q,
                                                       nv.ptr(rows), C, nv.ptr(out), nv.stream()), name)
        if self.n_sparse and C:
            sp, _ = self._check_sparse(sparse, Q)
            g = sp[:, :, rows.clamp(min=0)].float()                       # [Q,Fs,C] gather (index.py:116)
            g = g * (rows >= 0).to(g.dtype)                               # unknown keys -> 0 (index.py:117)
            out[self.n_dense:] = g.permute(1, 0, 2)
        return out

    # ------------------------------------------------------------------ faithful pipeline (contrastive.py:669-704)
    @torch.no_grad()
    def union_rescore_batch(self, q_vecs, q_emb: Optional[torch.Tensor] = None, sparse: Optional[torch.Tensor] = None,
                            top_k: Optional[int] = None, sparse_tokens=None, batch: Optional[int] = None
                            ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """The reference pipeline for a whole batch on the device: per-field top-k (one streaming pass per field,
        ``retrieve_batch``, contrastive.py:672-674) then ONE kernel (``mfar_union_rescore``) for per-query union ->
        rescore under every field -> * mask -> mixture -> top-k (676-696).
        Returns (values [Q,k], local rows [Q,k], union sizes [Q]); rows of a query whose union is smaller than k are
        padded with (-inf, -1) - ``union_rescore`` raises for those, like the reference's ``torch.topk``.
        bf16 corpus only."""
        self._require_bf16("union_rescore")
        k = top_k or self.top_k
        q_bf16 = self.corpus.prepare_queries(q_vecs) if self.corpus is not None else None
        if sparse_tokens is not None:                                      # BM25 get_scores once per (query, field)
            sparse = self._sparse_from_tokens(None, sparse_tokens, q_bf16, batch)
        _, rows = self.per_field_topk(q_vecs, sparse, k, batch=batch)      # [F,Q,k] local rows, (0.0, row 0) quirk applied
        Q = rows.shape[1]
        qe = self.mixture_input(q_vecs, q_emb)
        w = self.mixture.field_weights(qe, self.mask, batch=Q)             # softmax(q@W) * mask, [Q,F]
        sp, code = self._check_sparse(sparse, Q)
        vals = torch.empty((Q, k), dtype=torch.float32, device=self.device)
        out_rows = torch.empty((Q, k), dtype=torch.int64, device=self.device)
        usize = torch.empty((Q,), dtype=torch.int32, device=self.device)
        c = self.corpus
        rows = rows.contiguous()
        nv.check(nv.lib().mfar_union_rescore(
            nv.ptr(c.data) if c is not None else 0, self.n_docs, c.n_fields if c is not None else 0, self.n_dense,
            c.dim_pad if c is not None else 0, nv.ptr(q_bf16), Q, nv.ptr(w), nv.ptr(sp), self.n_sparse, code,
            sp.shape[2] if sp is not None else self.n_docs, nv.ptr(rows), rows.shape[0], rows.shape[2], k, nv.ptr(vals),
            nv.ptr(out_rows), nv.ptr(usize), nv.stream()), "union_rescore")
        self.last_launches += 2                                            # + mixture weights + the union/rescore kernel
        return vals, out_rows, usize

    @torch.no_grad()
    def union_rescore(self, q_vecs, q_emb: Optional[torch.Tensor] = None, sparse: Optional[torch.Tensor] = None,
                      top_k: Optional[int] = None, sparse_tokens=None, batch: Optional[int] = None
                      ) -> Tuple[List[torch.Tensor], List[torch.Tensor]]:
        """per-field top-k -> union -> rescore -> * mask -> mixture -> top-k (``union_rescore_batch``).
        Returns per query (values [k], local rows [k])."""
        k = top_k or self.top_k
        vals, rows, usize = self.union_rescore_batch(q_vecs, q_emb, sparse, k, sparse_tokens, batch)
        if int(usize.min().item()) < k:
            raise RuntimeError("selected index k out of range")           # what torch.topk raises in the reference
        return list(vals.unbind(0)), list(rows.unbind(0))

    # ------------------------------------------------------------------ QRes emission (contrastive.py:696-704)
    def trec_eval_step(self, query_ids: Sequence[str], q_vecs, qres_output: TextIO, q_emb=None, sparse=None,
                       mode: str = "exhaustive", sparse_tokens=None) -> None:
        if self.numeric_ids_to_keys is None:
            raise RuntimeError("trec_eval_step needs numeric_ids_to_keys to name documents")
        if mode == "exhaustive":
            scores, ids = self.search(q_vecs, q_emb, sparse, sparse_tokens=sparse_tokens)
            scores, ids = scores.cpu().tolist(), (ids - self.doc_id_base).cpu().tolist()
        elif mode == "union_rescore":
            v, r = self.union_rescore(q_vecs, q_emb, sparse, sparse_tokens=sparse_tokens)
            scores, ids = [x.cpu().tolist() for x in v], [x.cpu().tolist() for x in r]
        else:
            raise ValueError(mode)
        for qid, svals, rows in zip(query_ids, scores, ids):
            for sim, row in zip(svals, rows):
                print(QRes(query_id=qid, doc_id=self.numeric_ids_to_keys[row], sim=sim), file=qres_output)


class GraphedSearch:
    """``MultiFieldRetriever.search`` for one fixed batch shape captured in a CUDA graph: the mixture-weights kernel,
    the sparse pre-mix / BM25 plan + scatter, the fused scoring kernel and the merge replay as ONE graph launch.
    For small shards (PRIME-2k, Q=64: the kernels take ~60 us, the 4-5 launches with their Python/ctypes calls ~110 us)
    the step is launch-bound and the graph removes that; for corpus-sized shards it changes nothing.

    Inputs are copied into static device buffers (``copy_`` accepts host or device tensors; a ``sparse_buffer`` given at
    construction is adopted as the static sparse input and filled by the caller), outputs are the static ``scores`` /
    ``ids`` tensors (valid until the next call).  BM25 token entries are padded to ``max_entries`` rows
    with (-1, 0, 0), which the plan kernel skips.  The graph holds the retriever's mask / weight tensors as they were at
    capture time: build a new GraphedSearch after ``mask_field``."""

    def __init__(self, retriever: "MultiFieldRetriever", batch: int, sparse: str = "none", max_entries: int = 0,
                 top_k: Optional[int] = None, sparse_dtype=torch.float16, sparse_ld: Optional[int] = None,
                 sharded=None, sparse_buffer: Optional[torch.Tensor] = None,
                 doc_filter: Optional[torch.Tensor] = None):
        """``sharded``: the ``mfar_b200.dist.ShardedRetriever`` wrapping ``retriever`` - the captured step then also holds
        the cross-GPU exchange + merge (its call counter lives in device memory, so the replayed launch is identical on
        every call); every rank must construct and call its GraphedSearch the same number of times.
        ``doc_filter``: a bitmap as ``MultiFieldRetriever.search`` takes it, adopted as a static input (not copied):
        every replay filters with its contents at that time, so the caller may rewrite them between replays."""
        r = self.r = retriever
        self.sharded = sharded
        dev = r.device
        self.k = top_k or r.top_k
        self.Q = int(batch)
        self.sparse_kind = sparse
        dim = r.corpus.dim if r.corpus is not None else 1
        # a cosine corpus normalises the query it is given: the static buffer keeps fp32 queries unrounded, so the graph
        # rounds them to bf16 once, after the normalisation, as the eager search does (without normalisation the one
        # rounding is the copy into a bf16 buffer)
        # (an E4M3 corpus likewise quantizes fp32 queries inside the graph)
        q_dtype = torch.float32 if r.corpus is not None and (r.corpus.normalize or r.corpus.e4m3) else torch.bfloat16
        self.q_vecs = torch.zeros((self.Q, dim), dtype=q_dtype, device=dev) if r.corpus is not None else None
        E = r.mixture.weight.shape[0] if r.mixture.query_cond else 0
        self.q_emb = torch.zeros((self.Q, E), dtype=torch.float32, device=dev) if E else None
        self.sparse = self.entries = None
        self.doc_filter = doc_filter
        if doc_filter is not None:
            r._check_filter(doc_filter, self.Q)            # fail here rather than inside the capture
        if sparse == "dense":
            if sparse_buffer is not None:                 # adopt the caller's [Q,Fs,ld] tensor as the static input: a
                self.sparse = sparse_buffer               # corpus-sized score tensor is not copied per replay
            else:
                ld = sparse_ld or _round_up(r.n_docs, 64)  # 32-byte aligned rows: gathered inside the scoring epilogue
                self.sparse = torch.zeros((self.Q, r.n_sparse, ld), dtype=sparse_dtype, device=dev)
        elif sparse == "bm25":
            if r.bm25 is None or max_entries <= 0:
                raise ValueError("sparse='bm25' needs a retriever with sparse_indices and max_entries > 0")
            self.entries = torch.full((int(max_entries), 3), -1, dtype=torch.int32, device=dev)
        elif sparse != "none":
            raise ValueError("sparse must be 'none', 'dense' or 'bm25'")
        if r.n_sparse and sparse == "none":
            raise ValueError("retriever has sparse fields: pass sparse='dense' or 'bm25'")
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):                       # warm-up: workspaces, attributes, tensor maps
            for _ in range(2):
                self._run()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.scores, self.ids = self._run()
        # + mixture weights (+ epoch bump, exchange; pipelined: bump, push, wait+merge of the previous batch)
        self.launches = r.last_launches + 1 + (0 if sharded is None else (3 if getattr(sharded, "pipelined", False) else 2))

    def _run(self):
        if self.sharded is not None:
            return self.sharded.search(self.q_vecs, self.q_emb, self.sparse, top_k=self.k, sparse_tokens=self.entries,
                                       doc_filter=self.doc_filter)
        return self.r.search(self.q_vecs, self.q_emb, self.sparse, top_k=self.k, sparse_tokens=self.entries,
                             batch=self.Q, doc_filter=self.doc_filter)

    def __call__(self, q_vecs=None, q_emb=None, sparse=None, entries=None):
        if self.q_vecs is not None:
            self.q_vecs.copy_(q_vecs, non_blocking=True)
        if self.q_emb is not None:
            self.q_emb.copy_(q_emb if q_emb is not None else self.r.mixture_input(q_vecs), non_blocking=True)
        if self.sparse is not None and sparse is not None and sparse.data_ptr() != self.sparse.data_ptr():
            self.sparse[:, :, : sparse.shape[2]].copy_(sparse, non_blocking=True)
        if self.entries is not None:
            n = entries.shape[0]
            if n > self.entries.shape[0]:
                raise ValueError(f"{n} token entries exceed the captured capacity {self.entries.shape[0]}")
            self.entries[:n].copy_(entries, non_blocking=True)
            self.entries[n:, 0] = -1
        self.graph.replay()
        return self.scores, self.ids
