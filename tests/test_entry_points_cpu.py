"""The sizing and argument-checking surface of the scoring entry points, pinned value by value - no GPU needed.

Callers size their workspaces and scratch buffers with ``mfar_score_topk*_workspace_bytes`` and
``mfar_search_host*_scratch_bytes``, so those numbers are part of the ABI.  The status tables hold only calls that a
check rejects before the library looks for a device; they return the same status with or without a GPU (and never
touch the fake pointers they are given).  Every value below is what the library returned when the tables were
written."""
import ctypes
import functools
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

ARG, SHAPE = 1, 2          # MFAR_ERR_ARG, MFAR_ERR_SHAPE
F32, F16 = 0, 2            # MFAR_F32, MFAR_F16

# mfar_score_topk_workspace_bytes(Q, k, n_docs, n_sparse) for n_sparse = 0, 1, 4 (the same for every k)
WORKSPACE = {
    (1, 1): (537088, 537600, 537600),
    (1, 129): (1066496, 1067520, 1067520),
    (1, 4097): (17478144, 17495040, 17495040),
    (1, 330000): (78360064, 79680512, 79680512),
    (1, 10000000): (78360064, 118360064, 118360064),
    (16, 1): (567808, 576000, 576000),
    (16, 129): (1097216, 1113600, 1113600),
    (16, 4097): (17508864, 17779200, 17779200),
    (16, 330000): (78390784, 99517952, 99517952),
    (16, 10000000): (78390784, 718390784, 718390784),
    (17, 1): (569856, 578560, 578560),
    (17, 129): (1099264, 1116672, 1116672),
    (17, 4097): (17510912, 17798144, 17798144),
    (17, 330000): (78392832, 100840448, 100840448),
    (17, 10000000): (78392832, 758392832, 758392832),
    (64, 1): (666368, 699136, 699136),
    (64, 129): (1195776, 1261312, 1261312),
    (64, 4097): (17607424, 18688768, 18688768),
    (64, 330000): (78489344, 162998016, 162998016),
    (64, 10000000): (78489344, 2638489344, 2638489344),
    (65, 1): (668672, 701952, 701952),
    (65, 129): (1198080, 1264640, 1264640),
    (65, 4097): (17609728, 18707968, 18707968),
    (65, 330000): (78491648, 164320768, 164320768),
    (65, 10000000): (78491648, 2678491648, 2678491648),
    (129, 1): (1330688, 1396736, 1396736),
    (129, 129): (2389504, 2521600, 2521600),
    (129, 4097): (35212800, 37392384, 37392384),
    (129, 330000): (78624256, 248962048, 248962048),
    (129, 10000000): (78624256, 5238624256, 5238624256),
    (512, 1): (3178752, 3440896, 3440896),
    (512, 129): (5296384, 5820672, 5820672),
    (512, 4097): (70942976, 79593728, 79593728),
    (512, 330000): (157765888, 833835264, 833835264),
    (512, 10000000): (157765888, 20637765888, 20637765888),
}
# the BM25 workspace adds the token plan: mfar_bm25_plan_bytes(n_entries) for n_entries = 0, 64
BM25_PLAN = {0: 256, 64: 1280}

# batch shapes of the host-buffer calls: (dim, n_dense, E, n_sparse, k)
HOST_CONFIGS = [(0, 0, 0, 1, 100), (0, 0, 768, 4, 1), (64, 1, 0, 0, 128), (768, 4, 768, 0, 100), (768, 4, 768, 4, 128)]
# mfar_search_host_scratch_bytes per (Q, n_docs): for each of HOST_CONFIGS, sparse_dtype = F16 then F32
SCRATCH = {
    (1, 1): (539904, 539904, 541952, 542464, 539392, 539392, 543488, 543488, 544512, 545024),
    (1, 4097): (17505536, 17513728, 17532160, 17565440, 17480448, 17480448, 17484544, 17484544, 17534720, 17568000),
    (1, 10000000): (138362112, 158362112, 198363904, 278363904, 78362368, 78362368, 78366464, 78366464, 198366464,
                    278366464),
    (17, 1): (602112, 604160, 640512, 649216, 598784, 598784, 669440, 669440, 692480, 701184),
    (17, 4097): (17960960, 18102272, 18417152, 18982912, 17539840, 17539840, 17610496, 17610496, 18469120, 19034880),
    (17, 10000000): (1098414080, 1438414080, 2118446080, 3478446080, 78421760, 78421760, 78492416, 78492416,
                     2118498048, 3478498048),
    (65, 1): (789760, 797952, 937472, 970752, 777984, 777984, 1047808, 1047808, 1136896, 1170176),
    (65, 4097): (19328256, 19868928, 21073408, 23236608, 17719040, 17719040, 17988864, 17988864, 21272832, 23436032),
    (65, 10000000): (3978571008, 5278571008, 7878693888, 13078693888, 78600960, 78600960, 78870784, 78870784,
                     7878893312, 13078893312),
    (512, 1): (4124928, 4190464, 5290240, 5552384, 4034816, 4034816, 6160640, 6160640, 6865152, 7127296),
    (512, 4097): (84472064, 88731904, 98220288, 115259648, 71799040, 71799040, 73924864, 73924864, 99795200,
                  116834560),
    (512, 10000000): (30878384384, 41118384384, 61599353088, 102559353088, 158621952, 158621952, 160747776,
                      160747776, 61600928000, 102560928000),
}
# mfar_search_host_bm25_scratch_bytes per (Q, n_docs): for each of HOST_CONFIGS, n_entries = 0 then 64.  With no
# dense field it is one 256-byte block larger than the score-row layout: it reserves a query row of at least 1 element.
SCRATCH_BM25 = {
    (1, 1): (540416, 541952, 542208, 543744, 539904, 541440, 544000, 545536, 544512, 546048),
    (1, 4097): (17497856, 17499392, 17499648, 17501184, 17480960, 17482496, 17485056, 17486592, 17501952, 17503488),
    (1, 10000000): (118362880, 118364416, 118364672, 118366208, 78362880, 78364416, 78366976, 78368512, 118366976,
                    118368512),
    (17, 1): (600576, 602112, 632576, 634112, 599296, 600832, 669952, 671488, 684288, 685824),
    (17, 4097): (17820160, 17821696, 17852160, 17853696, 17540352, 17541888, 17611008, 17612544, 17903872, 17905408),
    (17, 10000000): (758414848, 758416384, 758446848, 758448384, 78422272, 78423808, 78492928, 78494464, 758498560,
                     758500096),
    (65, 1): (782080, 783616, 904960, 906496, 778496, 780032, 1048320, 1049856, 1104128, 1105664),
    (65, 4097): (18788096, 18789632, 18910976, 18912512, 17719552, 17721088, 17989376, 17990912, 19110144, 19111680),
    (65, 10000000): (2678571776, 2678573312, 2678694656, 2678696192, 78601472, 78603008, 78871296, 78872832,
                     2678893824, 2678895360),
    (512, 1): (4060928, 4062464, 5029632, 5031168, 4035328, 4036864, 6161152, 6162688, 6603520, 6605056),
    (512, 4097): (80213760, 80215296, 81182464, 81184000, 71799552, 71801088, 73925376, 73926912, 82756352,
                  82757888),
    (512, 10000000): (20638385920, 20638387456, 20639354624, 20639356160, 158622464, 158624000, 160748288, 160749824,
                      20640928512, 20640930048),
}


def _lib():
    from mfar_b200 import _native as nv
    return nv.lib()


def test_score_topk_workspace_bytes():
    lib = _lib()
    for k in (1, 100, 128):
        got = {(Q, n): tuple(lib.mfar_score_topk_workspace_bytes(Q, k, n, ns) for ns in (0, 1, 4)) for Q, n in WORKSPACE}
        assert got == WORKSPACE, k
        for ne, plan in BM25_PLAN.items():
            got = {(Q, n): tuple(lib.mfar_score_topk_bm25_workspace_bytes(Q, k, n, ns, ne) - plan for ns in (0, 1, 4))
                   for Q, n in WORKSPACE}
            assert got == WORKSPACE, (k, ne)


@pytest.mark.parametrize("entry,table,variants", [
    ("mfar_search_host_scratch_bytes", SCRATCH, (F16, F32)),
    ("mfar_search_host_bm25_scratch_bytes", SCRATCH_BM25, (0, 64))])
def test_search_host_scratch_bytes(entry, table, variants):
    fn = getattr(_lib(), entry)
    got = {(Q, n): tuple(fn(Q, dim, E, nd, ns, n, v, k) for (dim, nd, E, ns, k) in HOST_CONFIGS for v in variants)
           for (Q, n) in table}
    assert got == table


# ------------------------------------------------------------------ argument checks ahead of the device check
PTR = 1 << 20                     # a 256-byte aligned stand-in for a device / host buffer; never dereferenced
N_SPARSE = 2
_offsets = (ctypes.c_int64 * 66)(0, 10, *([20] * 64))          # host field offsets: n_sparse + 1 of them are read
_ptrs = (ctypes.c_void_p * 64)(*([PTR] * 64))                  # host arrays of per-field device pointers
_vocab = (ctypes.c_int32 * 64)(*([100] * 64))
DEFAULTS = {
    "corpus": PTR, "corpus_scales": PTR, "n_docs": 1000, "corpus_fields": 4, "field_begin": 0, "n_dense": 4,
    "dim": 768, "q_vecs": PTR, "q_scales": PTR, "Q": 8, "w": PTR, "sparse": PTR, "n_sparse": N_SPARSE,
    "sparse_dtype": F16, "sparse_ld": 1024, "coo_keys": PTR, "coo_vals": PTR, "coo_dtype": F16,
    "field_offsets_host": ctypes.addressof(_offsets), "indptr_host": ctypes.addressof(_ptrs),
    "indices_host": ctypes.addressof(_ptrs), "data_host": ctypes.addressof(_ptrs), "vocab_host": ctypes.addressof(_vocab),
    "entries": PTR, "n_entries": 64, "doc_id_base": 0, "k": 100, "out_keys": PTR, "out_scores": PTR, "out_ids": PTR,
    "workspace": PTR, "workspace_bytes": 1 << 40, "impl": 0, "stream": None,
    "q_vecs_host": PTR, "q_emb_host": PTR, "E": 768, "W": PTR, "mask": PTR, "query_cond": 1, "sparse_host": PTR,
    "entries_host": PTR, "out_scores_host": PTR, "out_ids_host": PTR, "scratch": PTR, "scratch_bytes": 1 << 40,
    "n_fields": 4, "rows": PTR, "C": 10, "out": PTR,
}


@functools.lru_cache(maxsize=None)
def _params():
    """Parameter names of every entry point, read from the header."""
    header = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "mfar_b200.h")).read(), flags=re.S)
    return {name: [re.findall(r"\w+", p)[-1] for p in args.split(",")]
            for name, args in re.findall(r"\b(mfar_\w+)\s*\(([^)]*)\)\s*;", header)}


def _call(entry: str, overrides: dict) -> int:
    return getattr(_lib(), entry)(*[overrides.get(p, DEFAULTS[p]) for p in _params()[entry]])


TOPK = ("mfar_score_topk", "mfar_score_topk_e4m3")
TOPK_COO = ("mfar_score_topk_coo", "mfar_score_topk_coo_e4m3")
TOPK_BM25 = ("mfar_score_topk_bm25", "mfar_score_topk_bm25_e4m3")
E4M3 = ("mfar_score_topk_e4m3", "mfar_score_topk_coo_e4m3", "mfar_score_topk_bm25_e4m3")
HOST = ("mfar_search_host", "mfar_search_host_bm25")
CANDIDATES = ("mfar_score_candidates", "mfar_score_candidates_e4m3")
ALL_TOPK = TOPK + TOPK_COO + TOPK_BM25

# (entry points, overrides of DEFAULTS, status)
STATUS_CASES = [
    (ALL_TOPK, {"workspace": 0}, ARG),
    (ALL_TOPK, {"w": 0}, ARG),
    (ALL_TOPK, {"out_keys": 0, "out_scores": 0, "out_ids": 0}, ARG),
    (ALL_TOPK, {"corpus": 0}, ARG),
    (ALL_TOPK, {"q_vecs": 0}, ARG),
    (ALL_TOPK, {"n_docs": 0}, ARG),
    (ALL_TOPK, {"Q": 0}, ARG),
    (ALL_TOPK, {"k": 0}, SHAPE),
    (ALL_TOPK, {"k": 129}, SHAPE),
    (ALL_TOPK, {"doc_id_base": (1 << 32) - 999}, SHAPE),
    (ALL_TOPK, {"doc_id_base": -1}, SHAPE),
    (ALL_TOPK, {"impl": 4}, ARG),
    (ALL_TOPK, {"impl": -1}, ARG),
    (ALL_TOPK, {"n_dense": 63}, SHAPE),
    (ALL_TOPK, {"field_begin": 1}, ARG),
    (E4M3, {"corpus_scales": 0}, ARG),
    (E4M3, {"q_scales": 0}, ARG),
    (TOPK, {"sparse": 0}, ARG),
    (TOPK, {"sparse_ld": 999}, ARG),
    (TOPK, {"n_dense": 0, "n_sparse": 0}, SHAPE),
    (TOPK_COO, {"n_dense": 0, "n_sparse": 0}, ARG),          # the COO checks run first
    (TOPK_COO, {"n_sparse": -1}, ARG),
    (TOPK_COO, {"n_sparse": 0, "k": 0}, ARG),
    (TOPK_COO, {"field_offsets_host": 0}, ARG),
    (TOPK_COO, {"coo_keys": 0}, ARG),
    (TOPK_COO, {"coo_vals": 0}, ARG),
    (TOPK_COO, {"coo_keys": 0, "workspace": 0}, ARG),
    (TOPK_BM25, {"n_dense": 0, "n_sparse": 0}, SHAPE),         # so do the BM25 ones
    (TOPK_BM25, {"n_sparse": 65}, SHAPE),
    (TOPK_BM25, {"indptr_host": 0}, ARG),
    (TOPK_BM25, {"vocab_host": 0, "k": 0}, ARG),
    (TOPK_BM25, {"n_sparse": 0, "workspace": 0}, SHAPE),
    (TOPK_BM25, {"n_entries": -1}, ARG),
    (TOPK_BM25, {"entries": 0}, ARG),
    (HOST, {"scratch": 0}, ARG),
    (HOST, {"scratch": PTR + 64}, ARG),
    (HOST, {"W": 0}, ARG),
    (HOST, {"out_scores_host": 0}, ARG),
    (HOST, {"out_ids_host": 0}, ARG),
    (HOST, {"Q": 0}, ARG),
    (HOST, {"n_docs": 0}, ARG),
    (HOST, {"q_vecs_host": 0}, ARG),
    (HOST, {"q_emb_host": 0}, ARG),
    (("mfar_search_host",), {"sparse_host": 0}, ARG),
    (("mfar_search_host_bm25",), {"n_entries": -1}, ARG),
    (("mfar_search_host_bm25",), {"entries_host": 0}, ARG),
    (CANDIDATES, {"corpus": 0}, ARG),
    (CANDIDATES, {"q_vecs": 0}, ARG),
    (CANDIDATES, {"rows": 0}, ARG),
    (CANDIDATES, {"out": 0}, ARG),
    (CANDIDATES, {"Q": 0}, ARG),
    (CANDIDATES, {"C": -1}, ARG),
    (CANDIDATES, {"n_docs": 0}, ARG),
    (CANDIDATES, {"n_fields": 0}, SHAPE),
    (CANDIDATES, {"field_begin": 1}, SHAPE),
    (CANDIDATES, {"dim": 0}, SHAPE),
    (("mfar_score_candidates_e4m3",), {"corpus_scales": 0}, ARG),
    (("mfar_score_candidates_e4m3",), {"q_scales": 0}, ARG),
]


@pytest.mark.parametrize("entry,overrides,status",
                         [(e, o, s) for entries, o, s in STATUS_CASES for e in entries],
                         ids=lambda v: v if isinstance(v, str) else ",".join(f"{k}={x}" for k, x in v.items())
                         if isinstance(v, dict) else str(v))
def test_malformed_calls_return_their_status(entry, overrides, status):
    assert _call(entry, overrides) == status
