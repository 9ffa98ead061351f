"""Filtered search (DESIGN §4.5) without a GPU: the argument checks of the six ``*_filtered`` entry points, the
``doc_filter`` checks of ``MultiFieldRetriever``, and the filtered ranking rule of the float64 helper the GPU tests
compare against (tests/filter_oracle.py)."""
import ctypes
import functools
import os
import re

import numpy as np
import pytest
import torch

import filter_oracle as FO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARG, SHAPE = 1, 2                 # MFAR_ERR_ARG, MFAR_ERR_SHAPE
PTR = 1 << 20                     # 256-byte aligned stand-in for a device buffer; never dereferenced
_offsets = (ctypes.c_int64 * 66)(0, 10, *([20] * 64))
_ptrs = (ctypes.c_void_p * 64)(*([PTR] * 64))
_vocab = (ctypes.c_int32 * 64)(*([100] * 64))
DEFAULTS = {
    "corpus": PTR, "corpus_scales": PTR, "n_docs": 1000, "corpus_fields": 4, "field_begin": 0, "n_dense": 4,
    "dim": 768, "q_vecs": PTR, "q_scales": PTR, "Q": 8, "w": PTR, "sparse": PTR, "n_sparse": 2, "sparse_dtype": 2,
    "sparse_ld": 1024, "coo_keys": PTR, "coo_vals": PTR, "coo_dtype": 2, "field_offsets_host": ctypes.addressof(_offsets),
    "indptr_host": ctypes.addressof(_ptrs), "indices_host": ctypes.addressof(_ptrs),
    "data_host": ctypes.addressof(_ptrs), "vocab_host": ctypes.addressof(_vocab), "entries": PTR, "n_entries": 64,
    "doc_id_base": 0, "filter_bits": PTR, "filter_rows": 1, "filter_ld": 32, "k": 100, "out_keys": PTR,
    "out_scores": PTR, "out_ids": PTR, "workspace": PTR, "workspace_bytes": 1 << 40, "impl": 0, "stream": None,
}
FILTERED = ("mfar_score_topk_filtered", "mfar_score_topk_coo_filtered", "mfar_score_topk_bm25_filtered",
            "mfar_score_topk_e4m3_filtered", "mfar_score_topk_coo_e4m3_filtered", "mfar_score_topk_bm25_e4m3_filtered")


def _lib():
    from mfar_b200 import _native as nv
    return nv.lib()


@functools.lru_cache(maxsize=None)
def _params():
    header = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "mfar_b200.h")).read(), flags=re.S)
    return {name: [re.findall(r"\w+", p)[-1] for p in args.split(",")]
            for name, args in re.findall(r"\b(mfar_\w+)\s*\(([^)]*)\)\s*;", header)}


def _call(entry, overrides):
    return getattr(_lib(), entry)(*[overrides.get(p, DEFAULTS[p]) for p in _params()[entry]])


@pytest.mark.parametrize("entry", FILTERED)
def test_filtered_entry_points_take_the_twin_arguments_plus_the_filter(entry):
    twin = entry[:-len("_filtered")]
    p, t = _params()[entry], _params()[twin]
    i = t.index("doc_id_base") + 1
    assert p == t[:i] + ["filter_bits", "filter_rows", "filter_ld"] + t[i:]
    from mfar_b200 import _native as nv
    assert len(nv.PROTOTYPES[entry][1]) == len(p)


STATUS_CASES = [
    ({"filter_bits": 0}, ARG),
    ({"filter_bits": PTR + 2}, ARG),
    ({"filter_rows": 0}, ARG),
    ({"filter_rows": 2}, ARG),
    ({"filter_rows": 9}, ARG),
    ({"filter_rows": -1}, ARG),
    ({"filter_ld": 31}, SHAPE),                                   # 1000 docs need 32 words
    ({"filter_ld": 0}, SHAPE),
    ({"filter_ld": -5}, SHAPE),
    ({"doc_id_base": 37, "filter_ld": 32}, SHAPE),                # ids up to 1036: 33 words
    ({"doc_id_base": (1 << 32) - 1000, "filter_ld": (1 << 27) - 1}, SHAPE),
    ({"filter_bits": 0, "k": 0}, SHAPE),                          # the twin's own checks come first
    ({"filter_ld": 0, "workspace": 0}, ARG),
]


@pytest.mark.parametrize("entry", FILTERED)
@pytest.mark.parametrize("overrides,status", STATUS_CASES, ids=[",".join(f"{k}={v}" for k, v in o.items())
                                                                 for o, _ in STATUS_CASES])
def test_malformed_filter_returns_its_status(entry, overrides, status):
    assert _call(entry, overrides) == status


def test_per_query_rows_need_rows_equal_q():
    for entry in FILTERED:
        assert _call(entry, {"Q": 3, "filter_rows": 3, "filter_ld": 31}) == SHAPE   # rows = Q accepted, then coverage
        assert _call(entry, {"Q": 3, "filter_rows": 4}) == ARG


# ------------------------------------------------------------------ MultiFieldRetriever.search(doc_filter=...)
def _host_retriever(n_docs=1000, base=0):
    """The checking half of a retriever, on the host: ``_check_filter`` reads device, doc_id_base and n_docs only."""
    from mfar_b200.modeling.retrieval import MultiFieldRetriever
    r = MultiFieldRetriever.__new__(MultiFieldRetriever)
    r.device, r.n_docs, r.doc_id_base = torch.device("cpu"), n_docs, base
    return r


@pytest.mark.parametrize("bad,msg", [
    (lambda: torch.zeros(32, dtype=torch.int64), "int32 or uint32"),
    (lambda: torch.zeros(32, dtype=torch.float32), "int32 or uint32"),
    (lambda: torch.zeros(32, dtype=torch.int32, device="meta"), "tensor on"),
    (lambda: np.zeros(32, dtype=np.uint32), "tensor on"),
    (lambda: torch.zeros(31, dtype=torch.int32), "need 32"),
    (lambda: torch.zeros((5, 32), dtype=torch.int32), r"\[W\]"),
    (lambda: torch.zeros((8, 32, 1), dtype=torch.int32), r"\[W\]"),
    (lambda: torch.zeros((8, 64), dtype=torch.int32)[:, ::2], "contiguous"),
])
def test_search_rejects_a_malformed_doc_filter(bad, msg):
    with pytest.raises(ValueError, match=msg):
        _host_retriever()._check_filter(bad(), 8)


def test_doc_filter_coverage_counts_the_global_ids():
    r = _host_retriever(1000, base=37)                            # ids 37 .. 1036: 33 words
    with pytest.raises(ValueError, match="need 33"):
        r._check_filter(torch.zeros(32, dtype=torch.int32), 8)
    bits, rows, ld = r._check_filter(torch.zeros(33, dtype=torch.uint32), 8)
    assert (rows, ld) == (1, 33)
    bits, rows, ld = r._check_filter(torch.zeros((8, 40), dtype=torch.int32), 8)
    assert (rows, ld) == (8, 40)
    assert _host_retriever()._check_filter(None, 8) is None


# ------------------------------------------------------------------ the float64 helper
def test_bitmap_rows_are_safe_docs_bitmap_at_global_ids():
    rng = np.random.default_rng(0)
    for base in (0, 5, 37, 64):
        el = rng.random((3, 300)) < 0.5
        bits = FO.bitmap_rows(el, base)
        assert bits.shape == (3, (base + 300 + 31) // 32) and bits.dtype == np.uint32
        assert np.array_equal(FO.eligible_from_bits(bits, base, 300), el)
        for r in range(3):                                        # bits below the base stay clear
            assert not FO.eligible_from_bits(bits[r], 0, base).any()


def test_filtered_ranking_rule():
    s = np.array([[3.0, np.nan, 5.0, np.inf, 5.0, -np.inf, 1.0, 5.0]])
    every = np.ones(8, dtype=bool)
    fs, fi = FO.filtered_topk(s, every, 8, doc_id_base=10)        # NaN > +inf > finite desc (id asc) > -inf
    assert fi.tolist() == [[11, 13, 12, 14, 17, 10, 16, 15]]
    el = np.array([True, False, False, True, True, True, False, True])
    fs, fi = FO.filtered_topk(s, el, 4)
    assert fi.tolist() == [[3, 4, 7, 0]] and fs.tolist() == [[np.inf, 5.0, 5.0, 3.0]]
    fs, fi = FO.filtered_topk(s, el, 7)                           # 5 eligible: two padding slots
    assert fi.tolist() == [[3, 4, 7, 0, 5, -1, -1]]
    assert fs[0, 5:].tolist() == [-np.inf, -np.inf] and fs[0, 4] == -np.inf
    fs, fi = FO.filtered_topk(np.vstack([s, s]), np.vstack([el, ~el]), 3)   # per-query rows
    assert fi.tolist() == [[3, 4, 7], [1, 2, 6]]
    fs, fi = FO.filtered_topk(s, np.zeros(8, dtype=bool), 2)
    assert fi.tolist() == [[-1, -1]] and np.isneginf(fs).all()


def test_filtered_helper_equals_the_unfiltered_rank_minus_the_excluded():
    rng = np.random.default_rng(1)
    s = rng.integers(0, 40, size=(5, 500)).astype(np.float64)     # many exact ties
    top = FO.unfiltered_rank(s, 128)
    el = np.ones((5, 500), dtype=bool)
    for q in range(5):
        el[q, top[q][:64]] = False
    _, fi = FO.filtered_topk(s, el, 64)
    assert np.array_equal(fi, np.stack([t[64:128] for t in top]))
