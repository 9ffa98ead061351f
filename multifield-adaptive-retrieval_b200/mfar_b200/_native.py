"""ctypes binding of libmfar_b200.so (C ABI: include/mfar_b200.h).

The library is built in-tree by ``multifield-adaptive-retrieval_b200/build.py``.  Loading
fails loudly when it is missing - there is no Python / PyTorch fallback for any compute call.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MFAR_LIB") or os.path.join(_HERE, "libmfar_b200.so")   # MFAR_LIB: instrumented builds

F32, BF16, F16, E4M3 = 0, 1, 2, 3
IMPL = {"auto": 0, "simt": 1, "tcgen05": 2, "tcgen05_qs": 3}
TILE_DOCS = 128
MAX_K = 128
MAX_FIELDS = 64

_lib = None

_vp, _i, _i64, _sz, _f64, _f32 = C.c_void_p, C.c_int, C.c_int64, C.c_size_t, C.c_double, C.c_float

# name -> (restype, argtypes); kept in one table so tests can check every symbol of the header
PROTOTYPES = {
    "mfar_abi_version": (_i, []),
    "mfar_status_string": (C.c_char_p, [_i]),
    "mfar_device_check": (_i, [_i]),
    "mfar_corpus_packed_elems": (_i64, [_i64, _i, _i]),
    "mfar_corpus_pack_rows": (_i, [_vp, _i, _i64, _i64, _vp, _i64, _i, _i, _i, _i, _vp]),
    "mfar_corpus_unpack_rows": (_i, [_vp, _i64, _i, _i, _i, _i64, _i64, _vp, _vp]),
    "mfar_corpus_pack_rows_e4m3": (_i, [_vp, _i, _i64, _i64, _vp, _vp, _i64, _i, _i, _i, _i, _vp]),
    "mfar_corpus_unpack_rows_e4m3": (_i, [_vp, _vp, _i64, _i, _i, _i, _i64, _i64, _vp, _vp]),
    "mfar_mixture_weights": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    "mfar_mixture_apply": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    "mfar_score_topk_workspace_bytes": (_sz, [_i, _i, _i64, _i]),
    "mfar_score_topk": (_i, [_vp, _i64, _i, _i, _i, _i, _vp, _i, _vp, _vp, _i, _i, _i64, _i64, _i, _vp, _vp, _vp,
                             _vp, _sz, _i, _vp]),
    "mfar_score_topk_coo": (_i, [_vp, _i64, _i, _i, _i, _i, _vp, _i, _vp, _vp, _vp, _i, _vp, _i, _i64, _i, _vp, _vp, _vp,
                                 _vp, _sz, _i, _vp]),
    "mfar_score_topk_e4m3": (_i, [_vp, _vp, _i64, _i, _i, _i, _i, _vp, _vp, _i, _vp, _vp, _i, _i, _i64, _i64, _i, _vp,
                                  _vp, _vp, _vp, _sz, _i, _vp]),
    "mfar_score_topk_coo_e4m3": (_i, [_vp, _vp, _i64, _i, _i, _i, _i, _vp, _vp, _i, _vp, _vp, _vp, _i, _vp, _i, _i64, _i,
                                      _vp, _vp, _vp, _vp, _sz, _i, _vp]),
    "mfar_score_topk_bm25_e4m3": (_i, [_vp, _vp, _i64, _i, _i, _i, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _i, _vp,
                                       _i64, _i64, _i, _vp, _vp, _vp, _vp, _sz, _i, _vp]),
    # *_filtered: the twin's arguments with (filter_bits, filter_rows, filter_ld) after doc_id_base
    "mfar_score_topk_filtered": (_i, [_vp, _i64, _i, _i, _i, _i, _vp, _i, _vp, _vp, _i, _i, _i64, _i64, _vp, _i, _i64, _i,
                                      _vp, _vp, _vp, _vp, _sz, _i, _vp]),
    "mfar_score_topk_coo_filtered": (_i, [_vp, _i64, _i, _i, _i, _i, _vp, _i, _vp, _vp, _vp, _i, _vp, _i, _i64, _vp, _i,
                                          _i64, _i, _vp, _vp, _vp, _vp, _sz, _i, _vp]),
    "mfar_score_topk_bm25_filtered": (_i, [_vp, _i64, _i, _i, _i, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i64,
                                           _i64, _vp, _i, _i64, _i, _vp, _vp, _vp, _vp, _sz, _i, _vp]),
    "mfar_score_topk_e4m3_filtered": (_i, [_vp, _vp, _i64, _i, _i, _i, _i, _vp, _vp, _i, _vp, _vp, _i, _i, _i64, _i64,
                                           _vp, _i, _i64, _i, _vp, _vp, _vp, _vp, _sz, _i, _vp]),
    "mfar_score_topk_coo_e4m3_filtered": (_i, [_vp, _vp, _i64, _i, _i, _i, _i, _vp, _vp, _i, _vp, _vp, _vp, _i, _vp, _i,
                                               _i64, _vp, _i, _i64, _i, _vp, _vp, _vp, _vp, _sz, _i, _vp]),
    "mfar_score_topk_bm25_e4m3_filtered": (_i, [_vp, _vp, _i64, _i, _i, _i, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _i,
                                                _vp, _i64, _i64, _vp, _i, _i64, _i, _vp, _vp, _vp, _vp, _sz, _i, _vp]),
    "mfar_score_candidates_e4m3": (_i, [_vp, _vp, _i64, _i, _i, _i, _i, _vp, _vp, _i, _vp, _i, _vp, _vp]),
    "mfar_topk_merge": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "mfar_exchange_buffer_bytes": (_sz, [_i, _i, _i]),
    "mfar_topk_exchange_merge": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "mfar_topk_exchange_merge_dev_epoch": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "mfar_topk_exchange_push": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _i, _vp, _vp]),
    "mfar_topk_exchange_wait_merge": (_i, [_i, _i, _i, _i, _i, _vp, _i, _i, _vp, _i, _vp, _vp, _vp, _vp]),
    "mfar_union_rescore": (_i, [_vp, _i64, _i, _i, _i, _vp, _i, _vp, _vp, _i, _i, _i64, _vp, _i, _i, _i, _vp, _vp, _vp,
                                _vp]),
    "mfar_topk_apply_zero_init": (_i, [_vp, _vp, _i, _i, _vp]),
    "mfar_score_candidates": (_i, [_vp, _i64, _i, _i, _i, _i, _vp, _i, _vp, _i, _vp, _vp]),
    "mfar_search_host_scratch_bytes": (_sz, [_i, _i, _i, _i, _i, _i64, _i, _i]),
    "mfar_search_host": (_i, [_vp, _i64, _i, _i, _i, _i, _vp, _vp, _i, _i, _vp, _vp, _i, _vp, _i, _i, _i64, _i,
                              _vp, _vp, _vp, _sz, _i, _vp]),
    "mfar_bm25_build_scores": (_i, [_vp, _vp, _vp, _i64, _vp, _vp, _i64, _f64, _f64, _f64, _vp, _vp]),
    "mfar_bm25_plan_bytes": (_sz, [_i64]),
    "mfar_bm25_scores": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _i64, _i, _vp, _i, _i, _i64, _vp, _i64, _i, _vp, _sz, _vp]),
    "mfar_sparse_coo_offsets_len": (_i64, [_i, _i64]),
    "mfar_sparse_coo_count": (_i, [_vp, _i64, _i, _i64, _vp, _i64, _vp, _vp]),
    "mfar_sparse_coo_write": (_i, [_vp, _i64, _i, _i64, _vp, _vp, _i64, _vp, _vp, _vp, _i, _vp]),
    "mfar_score_topk_bm25_workspace_bytes": (_sz, [_i, _i, _i64, _i, _i64]),
    "mfar_score_topk_bm25": (_i, [_vp, _i64, _i, _i, _i, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i64, _i64, _i,
                                  _vp, _vp, _vp, _vp, _sz, _i, _vp]),
    "mfar_search_host_bm25_scratch_bytes": (_sz, [_i, _i, _i, _i, _i, _i64, _i64, _i]),
    "mfar_search_host_bm25": (_i, [_vp, _i64, _i, _i, _i, _i, _vp, _vp, _i, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp, _i,
                                   _vp, _i64, _i64, _i, _vp, _vp, _vp, _sz, _i, _vp]),
    "mfar_field_components_fwd": (_i, [_vp, _i, _i, _vp, _i64, _i, _i64, _i64, _i64, _i64, _f32, _vp, _vp]),
    "mfar_field_components_bwd": (_i, [_vp, _i, _i, _vp, _i64, _i, _i64, _i64, _i64, _i64, _f32, _vp, _vp, _vp, _vp]),
    "mfar_mixture_bwd": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "mfar_last_launch_count": (_i, []),
    "mfar_profile_enable": (_i, [_i]),
    "mfar_profile_collect": (_i, [_vp, _i]),
    "mfar_profile_cluster4_ctas": (C.c_longlong, []),
}


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found - build it with `python multifield-adaptive-retrieval_b200/build.py` "
                "(mfar_b200 has no CPU / PyTorch fallback)")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().mfar_status_string(rc).decode()
        raise RuntimeError(f"mfar_b200 {what} failed: {msg} (status {rc})")


def ptr(t) -> int:
    """Device (or pinned host) address of a torch tensor / None."""
    return 0 if t is None else t.data_ptr()


def stream() -> int:
    import torch
    return torch.cuda.current_stream().cuda_stream


def require_device(t, name: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(f"mfar_b200: `{name}` must live on a CUDA (sm_100) device; there is no CPU path")
