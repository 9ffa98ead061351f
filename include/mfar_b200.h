/*
 * mfar_b200.h - C ABI of the B200-native multi-field scoring + top-k retrieval path.
 *
 * The reference (microsoft/multifield-adaptive-retrieval) is pure Python and has no FFI of
 * its own; the boundary this library replaces is the set of Python call sites listed next to
 * each entry point (paths relative to the reference root).  INTEGRATION.md shows the ctypes
 * binding a maintainer adds on the reference side.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - the caller allocates every buffer; the library borrows, never frees;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it and no entry
 *     point synchronises (except the *_host convenience calls, which say so);
 *   - return value: 0 = MFAR_OK, otherwise an mfar_status (mfar_status_string() names it);
 *   - re-entrant, no global mutable state apart from a per-process cache of TMA descriptors'
 *     driver entry point and the per-device diagnostic counter of mfar_profile_cluster4_ctas(); one process per GPU;
 *   - sm_100 only.  There is no CPU fallback: on any other device every compute entry point
 *     returns MFAR_ERR_ARCH.
 */
#ifndef MFAR_B200_H_
#define MFAR_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define MFAR_API __attribute__((visibility("default")))
#else
#define MFAR_API
#endif

#define MFAR_ABI_VERSION 1
#define MFAR_TILE_DOCS 128   /* docs per corpus tile (UMMA M)                       */
#define MFAR_EXCHANGE_SLOTS 4   /* key / flag slots per (rank, query) in an exchange buffer (epoch % slots) */
#define MFAR_MAX_K 128       /* top-k depth limit (reference hard-codes k = 100)    */
#define MFAR_MAX_FIELDS 64   /* dense + sparse fields (reference max: 44, PRIME)    */

typedef enum mfar_status {
  MFAR_OK = 0,
  MFAR_ERR_ARG = 1,        /* null pointer / non-positive size / misaligned pointer  */
  MFAR_ERR_SHAPE = 2,      /* dim, k, field count outside the supported envelope     */
  MFAR_ERR_ARCH = 3,       /* current device is not compute capability 10.x          */
  MFAR_ERR_WORKSPACE = 4,  /* workspace smaller than mfar_score_topk_workspace_bytes */
  MFAR_ERR_CUDA = 5,       /* a CUDA runtime/driver call failed (see stderr)         */
  MFAR_ERR_K_RANGE = 6     /* k > number of docs (reference: torch.topk raises)      */
} mfar_status;

typedef enum mfar_dtype { MFAR_F32 = 0, MFAR_BF16 = 1, MFAR_F16 = 2, MFAR_E4M3 = 3 } mfar_dtype;

/* which scoring kernel mfar_score_topk runs */
typedef enum mfar_impl {
  MFAR_IMPL_AUTO = 0,   /* tensor-core paths whenever their shape constraints hold; QS for Q > 64 */
  MFAR_IMPL_SIMT = 1,   /* CUDA-core streaming path (small query batches, cross-check) */
  MFAR_IMPL_TCGEN05 = 2, /* TMA + tcgen05.mma + TMEM, docs on the MMA M axis (small/medium batches)  */
  MFAR_IMPL_TCGEN05_QS = 3 /* query-stationary: queries resident in TMEM, CTA pairs (large batches) */
} mfar_impl;

MFAR_API int mfar_abi_version(void);
MFAR_API const char* mfar_status_string(int status);
/* 0 when `device` (or the current device if < 0) can run this library (sm_100). */
MFAR_API int mfar_device_check(int device);

/* ------------------------------------------------------------------------------------------
 * Corpus store.  Replaces: the per-field headerless fp32 memmaps {temp_dir}/{field.name}.npy
 * written at mfar/modeling/contrastive.py:482-490 and read at mfar/data/index.py:196,230
 * (MemoryMapDict, mfar/data/util.py:28-59).
 *
 * Packed layout in HBM (bf16):  [n_tiles][n_fields][MFAR_TILE_DOCS][dim]
 *   n_tiles = ceil(n_docs / 128); rows of the last tile beyond n_docs are zero.
 * One (tile, field) block is 128*dim*2 contiguous bytes = one TMA box column.
 * ------------------------------------------------------------------------------------------ */
MFAR_API int64_t mfar_corpus_packed_elems(int64_t n_docs, int n_fields, int dim);

/* Convert rows [row_begin, row_begin + n_rows) of ONE field from a row-major [n_rows, dim]
 * slab (fp32 or bf16) into the packed corpus; optional per-row L2 normalisation (the
 * reference's Normalize() module, mfar/modeling/util.py:50-51) before rounding to bf16.
 * Call once per (field, slab); slabs may arrive in any order.  Zero the packed buffer first
 * if n_docs is not a multiple of 128. */
MFAR_API int mfar_corpus_pack_rows(const void* src, int src_dtype, int64_t n_rows, int64_t row_begin,
                          void* packed, int64_t n_docs, int n_fields, int field, int dim,
                          int normalize, void* stream);

/* Inverse view for tests / candidate export: copy rows of one field out as fp32 [n_rows, dim]. */
MFAR_API int mfar_corpus_unpack_rows(const void* packed, int64_t n_docs, int n_fields, int field, int dim,
                            int64_t row_begin, int64_t n_rows, float* dst, void* stream);

/* ------------------------------------------------------------------------------------------
 * FP8 (E4M3) corpus: half the bytes of the bf16 store, scored at the tensor cores' FP8 rate.
 *   payload  uint8 [n_tiles][n_fields][MFAR_TILE_DOCS][dim]   one E4M3 byte per element
 *   scales   fp32  [n_tiles][n_fields][MFAR_TILE_DOCS]        one power of two per (doc, field) row
 * The scoring kernels need dim % 128 == 0 (one 128-byte swizzle span per K-chunk).  Tail rows of the last tile hold
 * payload 0 and scale 1: zero the payload and fill the scales with 1.0f before the first pack.
 *
 * A row x (fp32 or bf16; with normalize, first x / max(||x||_2, float32(1e-12)) in float64, as mfar_corpus_pack_rows)
 * is stored as s = 2^e with e = clamp(ceil(log2(amax / 448)), -117, 119), amax = max|x_i|, and p_i = the E4M3 value
 * nearest to x_i / s (ties to even, ONE rounding from float64, saturating to +-448).  p_i * s is then exactly a normal
 * fp32 / bf16 number: scoring the E4M3 corpus equals scoring its dequantized bf16 copy up to fp32 summation order.
 * A row of zeros stores s = 1 and payload 0; a row holding a NaN or an infinity stores s = NaN and payload 0 (its
 * dequantized row, and every score of its doc, is NaN).  Queries are quantized by the same call as a one-field corpus
 * of Q docs: [Q][dim] payload rows and [Q] scales.
 * ------------------------------------------------------------------------------------------ */
MFAR_API int mfar_corpus_pack_rows_e4m3(const void* src, int src_dtype, int64_t n_rows, int64_t row_begin,
                                        uint8_t* payload, float* scales, int64_t n_docs, int n_fields, int field,
                                        int dim, int normalize, void* stream);
/* Exact dequantization of rows of one field: dst fp32 [n_rows, dim] = float(p) * s. */
MFAR_API int mfar_corpus_unpack_rows_e4m3(const uint8_t* payload, const float* scales, int64_t n_docs, int n_fields,
                                          int field, int dim, int64_t row_begin, int64_t n_rows, float* dst,
                                          void* stream);

/* ------------------------------------------------------------------------------------------
 * Field mixture.  Replaces LinearWeights.forward, mfar/modeling/weighting.py:17-29, and the
 * field mask of mfar/modeling/contrastive.py:686,706-714.
 * ------------------------------------------------------------------------------------------ */
/* out_w[q,f] = softmax_f(q_emb[q,:] @ W[:,f]) * mask[f]       (query_cond != 0, W is [E,F])
 * out_w[q,f] = softmax_f(W[f,0]) * mask[f]                    (query_cond == 0, W is [F,1])
 * mask may be NULL (all ones).  The mask multiplies AFTER the softmax: masked fields keep
 * their softmax mass, weights are not renormalised - exactly contrastive.py:686 followed by
 * weighting.py:28-29.  fp32 throughout. */
MFAR_API int mfar_mixture_weights(const float* q_emb, const float* W, const float* mask, int Q, int E, int F,
                         int query_cond, float* out_w, void* stream);

/* out[b,s] = sum_f w[b or 0, f] * x[b,s,f]   (weighting.py:29).  w_rows is Q or 1. */
MFAR_API int mfar_mixture_apply(const float* x, const float* w, int B, int S, int F, int w_rows, float* out,
                       void* stream);

/* ------------------------------------------------------------------------------------------
 * Fused scoring + streaming top-k.  Replaces, in one pass over the corpus:
 *   DenseFlatIndex.retrieve_batch   mfar/data/index.py:181-222   (q.V^T + running top-k)
 *   DenseFlatIndex.score_batch      mfar/data/index.py:227-232   (subsumed: every doc is scored)
 *   BM25sSparseIndex.score_batch    mfar/data/index.py:111-118   (gather of precomputed scores)
 *   mask + LinearWeights + topk     mfar/modeling/contrastive.py:686,694,696
 *
 *   score[q,n] = sum_{f<n_dense} w[q,f] * <q_vec[q,:], corpus[n, field_begin+f, :]>
 *              + sum_{j<n_sparse} w[q,n_dense+j] * sparse[q, j, n]
 *   out = top-k over n of score[q,:], sorted by (score desc, doc id asc).
 *
 * corpus        packed bf16 corpus holding corpus_fields fields per tile; fields
 *               [field_begin, field_begin+n_dense) are scored
 * q_vecs        bf16 [Q, dim] row-major
 * w             fp32 [Q, n_dense+n_sparse] (mask already folded in by mfar_mixture_weights)
 * sparse        [Q, n_sparse, sparse_ld] fp32/f16 precomputed per-field scores of THIS shard's
 *               docs (column n = local doc n); NULL when n_sparse == 0
 * doc_id_base   added to the local doc index to form the emitted (global) doc id; ids must
 *               stay below 2^32
 * out_keys      optional uint64 [Q,k]: order-preserving (score,id) keys for mfar_topk_merge
 * out_scores    fp32 [Q,k];  out_ids  int64 [Q,k];  slots beyond n_docs: (-inf, -1)
 * ------------------------------------------------------------------------------------------ */
MFAR_API size_t mfar_score_topk_workspace_bytes(int Q, int k, int64_t n_docs, int n_sparse);

MFAR_API int mfar_score_topk(const void* corpus, int64_t n_docs, int corpus_fields, int field_begin, int n_dense,
                    int dim, const void* q_vecs, int Q, const float* w, const void* sparse, int n_sparse,
                    int sparse_dtype, int64_t sparse_ld, int64_t doc_id_base, int k, uint64_t* out_keys,
                    float* out_scores, int64_t* out_ids, void* workspace, size_t workspace_bytes, int impl,
                    void* stream);

/* Same pass with the sparse scores in the reference's precomputed-BM25 file layout instead of a dense tensor
 * (mfar/commands/precompute_bm25s_scores.py:21-30, read back by read_sparse_scores, mfar/modeling/util.py:151-173,
 * looked up by BM25sSparseIndex.score_batch_with_cache, mfar/data/index.py:120-125 - missing pairs score 0):
 *   coo_keys   int32 [nnz,2]: (query row in this batch, GLOBAL doc row); rows of other shards / batches are skipped
 *   coo_vals   [nnz] f16 (the file dtype) or f32
 *   field_offsets_host  HOST int64 [n_sparse+1]: entries [off[j], off[j+1]) belong to sparse field j; off[0] = 0
 * Duplicate (query, field, doc) entries add up. */
MFAR_API int mfar_score_topk_coo(const void* corpus, int64_t n_docs, int corpus_fields, int field_begin, int n_dense,
                        int dim, const void* q_vecs, int Q, const float* w, const int32_t* coo_keys,
                        const void* coo_vals, int coo_dtype, const int64_t* field_offsets_host, int n_sparse,
                        int64_t doc_id_base, int k, uint64_t* out_keys, float* out_scores, int64_t* out_ids,
                        void* workspace, size_t workspace_bytes, int impl, void* stream);

/* ------------------------------------------------------------------------------------------
 * BM25 sparse fields scored on the device.  Replaces bm25s.BM25.get_scores as the reference calls it
 * (BM25sSparseIndex.get_scores / score_batch / retrieve_batch, mfar/data/index.py:72-76, 95-118) and the
 * score-matrix arithmetic of bm25s.BM25.index (BM25sSparseIndex.create, index.py:134-145; method "lucene",
 * k1 = 1.2, b = 0.75).  bm25s (0.1.10) is a third-party dependency of the reference: BM25 parity is unpinned
 * (oracle/bm25_oracle.py restates its published algorithm).
 *
 * Per sparse field the index is the token-major (CSC) postings matrix bm25s builds and saves:
 *   indptr int64 [V+1], indices int32 [nnz] (LOCAL doc rows of this shard, ascending per token), data fp32 [nnz].
 * The *_host arguments below are HOST arrays of n_sparse DEVICE pointers (one per field).
 * A query batch is `entries`: DEVICE int32 [n_entries, 3] = (query row, sparse field j, token id), one entry per
 * query-token occurrence (repeats add up, as in bm25s); entries with an out-of-range member are skipped (a token
 * that is not in the vocabulary contributes nothing, index.py:112-117 / bm25s get_tokens_ids).
 * ------------------------------------------------------------------------------------------ */
/* data[p] = float32( float64(float32(ln(1 + (N - df + 0.5)/(df + 0.5)))) * tf / (k1*(1 - b + b*len/l_avg) + tf) )
 * for posting p = (post_token[p], post_doc[p], post_tf[p]); df int32 [V], doc_len int32 [n_docs_total]. */
MFAR_API int mfar_bm25_build_scores(const int32_t* post_token, const int32_t* post_doc, const int32_t* post_tf,
                                    int64_t nnz, const int32_t* df, const int32_t* doc_len, int64_t n_docs_total,
                                    double l_avg, double k1, double b, float* data, void* stream);

/* Device scratch the BM25 entry points need for a batch of n_entries query tokens. */
MFAR_API size_t mfar_bm25_plan_bytes(int64_t n_entries);

/* out[q, doc] (+)= w[q, w_off + j] * score_j(q, doc) over every entry; w == NULL means weight 1.
 * zero_first != 0 clears out[Q, ld] first: with n_sparse = 1 and w = NULL this is get_scores for a batch
 * (index.py:72-76) written as fp32 [Q, ld]. */
MFAR_API int mfar_bm25_scores(const void* const* indptr_host, const void* const* indices_host,
                              const void* const* data_host, const int32_t* vocab_host, int n_sparse,
                              const int32_t* entries, int64_t n_entries, int Q, const float* w, int w_ld, int w_off,
                              int64_t n_docs, float* out, int64_t ld, int zero_first, void* plan, size_t plan_bytes,
                              void* stream);

/* ------------------------------------------------------------------------------------------
 * Producer of the precomputed-BM25 score files the COO input above consumes.  Replaces
 * precompute_score_for_field (mfar/commands/precompute_bm25s_scores.py:12-30) over
 * BM25sSparseIndex.get_scores_sparse (mfar/data/index.py:78-84): of a batch of full-corpus score rows
 * `scores` fp32 [Q, ld] (mfar_bm25_scores output) keep the entries that are != 0 and whose doc is in the
 * safe set, as pairs (qids[q], doc_id_base + row) int32 [nnz, 2] + one value per pair (np.float16(score):
 * MFAR_F16, round-to-nearest; or MFAR_F32), ordered by (query row, doc) - the order the reference appends.
 *   safe_bits: bit (doc_id_base + row) of a uint32 bitmap over GLOBAL doc ids, or NULL = every doc is safe;
 *   qids: int32 [Q] query ids written into the pairs, or NULL = the row number;
 *   seg_offsets: int64 [mfar_sparse_coo_offsets_len(Q, n_docs)] scratch.  mfar_sparse_coo_count fills it with
 *     exclusive offsets per (query, 4096-doc segment); its LAST element is nnz: read it back (the one host
 *     round trip), allocate out_keys [nnz,2] / out_vals [nnz], then call mfar_sparse_coo_write with the same
 *     arguments.  No atomics: the output is deterministic.
 * ------------------------------------------------------------------------------------------ */
MFAR_API int64_t mfar_sparse_coo_offsets_len(int Q, int64_t n_docs);
MFAR_API int mfar_sparse_coo_count(const float* scores, int64_t ld, int Q, int64_t n_docs, const uint32_t* safe_bits,
                                   int64_t doc_id_base, int64_t* seg_offsets, void* stream);
MFAR_API int mfar_sparse_coo_write(const float* scores, int64_t ld, int Q, int64_t n_docs, const uint32_t* safe_bits,
                                   const int32_t* qids, int64_t doc_id_base, const int64_t* seg_offsets,
                                   int32_t* out_keys, void* out_vals, int vals_dtype, void* stream);

/* mfar_score_topk with the sparse fields given as BM25 postings + query tokens instead of score tensors:
 * workspace must hold mfar_score_topk_bm25_workspace_bytes(...). */
MFAR_API size_t mfar_score_topk_bm25_workspace_bytes(int Q, int k, int64_t n_docs, int n_sparse, int64_t n_entries);

MFAR_API int mfar_score_topk_bm25(const void* corpus, int64_t n_docs, int corpus_fields, int field_begin, int n_dense,
                                  int dim, const void* q_vecs, int Q, const float* w,
                                  const void* const* indptr_host, const void* const* indices_host,
                                  const void* const* data_host, const int32_t* vocab_host, int n_sparse,
                                  const int32_t* entries, int64_t n_entries, int64_t doc_id_base, int k,
                                  uint64_t* out_keys, float* out_scores, int64_t* out_ids, void* workspace,
                                  size_t workspace_bytes, int impl, void* stream);

/* The three entry points above on an E4M3 corpus (mfar_corpus_pack_rows_e4m3) and E4M3 queries: same arguments, plus
 * corpus_scales fp32 [n_tiles][corpus_fields][128] and q_scales fp32 [Q]; q_vecs is uint8 [Q, dim].
 *   score[q,n] = sum_f fmaf-accumulated  w[q,f] * ((D_f[q,n] * q_scales[q]) * corpus_scales[n,f])  (+ sparse terms)
 * with D_f the fp32 dot product of the two payload rows (every E4M3 x E4M3 product is exact in fp32).  The two scale
 * products are rounded one after the other: folded into one factor they could underflow (2^-117 * 2^-117).
 * impl: AUTO runs the tcgen05 kernel (kind::f8f6f4) at every batch size, SIMT the CUDA-core cross-check;
 * MFAR_IMPL_TCGEN05_QS returns MFAR_ERR_SHAPE.  Ordering, ties, NaN ranking, doc_id_base and k as mfar_score_topk. */
MFAR_API int mfar_score_topk_e4m3(const void* corpus, const float* corpus_scales, int64_t n_docs, int corpus_fields,
                                  int field_begin, int n_dense, int dim, const void* q_vecs, const float* q_scales,
                                  int Q, const float* w, const void* sparse, int n_sparse, int sparse_dtype,
                                  int64_t sparse_ld, int64_t doc_id_base, int k, uint64_t* out_keys, float* out_scores,
                                  int64_t* out_ids, void* workspace, size_t workspace_bytes, int impl, void* stream);
MFAR_API int mfar_score_topk_coo_e4m3(const void* corpus, const float* corpus_scales, int64_t n_docs,
                                      int corpus_fields, int field_begin, int n_dense, int dim, const void* q_vecs,
                                      const float* q_scales, int Q, const float* w, const int32_t* coo_keys,
                                      const void* coo_vals, int coo_dtype, const int64_t* field_offsets_host,
                                      int n_sparse, int64_t doc_id_base, int k, uint64_t* out_keys, float* out_scores,
                                      int64_t* out_ids, void* workspace, size_t workspace_bytes, int impl,
                                      void* stream);
MFAR_API int mfar_score_topk_bm25_e4m3(const void* corpus, const float* corpus_scales, int64_t n_docs,
                                       int corpus_fields, int field_begin, int n_dense, int dim, const void* q_vecs,
                                       const float* q_scales, int Q, const float* w, const void* const* indptr_host,
                                       const void* const* indices_host, const void* const* data_host,
                                       const int32_t* vocab_host, int n_sparse, const int32_t* entries,
                                       int64_t n_entries, int64_t doc_id_base, int k, uint64_t* out_keys,
                                       float* out_scores, int64_t* out_ids, void* workspace, size_t workspace_bytes,
                                       int impl, void* stream);

/* ------------------------------------------------------------------------------------------
 * Filtered search: the six scoring entry points above with a doc filter.  No reference counterpart - a widening
 * (DESIGN §0, §4.5): deleted docs, a metadata subset or docs a query has already seen are left out of the top-k
 * inside the scoring pass, so a query still gets k eligible docs however many of its best docs are ineligible.
 *   filter_bits  DEVICE uint32 bitmap over GLOBAL doc ids: bit d of word d >> 5 set <=> doc d is eligible (the
 *                layout of mfar_sparse_coo_count's safe_bits); 4-byte aligned
 *   filter_rows  1: one row [filter_ld] shared by every query;  Q: one row per query, [Q, filter_ld]
 *   filter_ld    words per row, 32 * filter_ld >= doc_id_base + n_docs
 * Each takes its unfiltered twin's arguments with these three after doc_id_base.  Result: the (score desc, id asc)
 * top-k of the eligible docs (NaN > +inf > finite > -inf); a query with fewer than k eligible docs gets (-inf, -1) in
 * the remaining slots.  Workspace sizes are the twin's.  MFAR_ERR_ARG: filter_bits NULL or misaligned, filter_rows
 * not 1 or Q;  MFAR_ERR_SHAPE: a row shorter than doc_id_base + n_docs bits.
 * ------------------------------------------------------------------------------------------ */
MFAR_API int mfar_score_topk_filtered(const void* corpus, int64_t n_docs, int corpus_fields, int field_begin,
                                      int n_dense, int dim, const void* q_vecs, int Q, const float* w,
                                      const void* sparse, int n_sparse, int sparse_dtype, int64_t sparse_ld,
                                      int64_t doc_id_base, const uint32_t* filter_bits, int filter_rows,
                                      int64_t filter_ld, int k, uint64_t* out_keys, float* out_scores,
                                      int64_t* out_ids, void* workspace, size_t workspace_bytes, int impl,
                                      void* stream);
/* mfar_score_topk_coo with a doc filter (no reference counterpart, DESIGN §4.5) */
MFAR_API int mfar_score_topk_coo_filtered(const void* corpus, int64_t n_docs, int corpus_fields, int field_begin,
                                          int n_dense, int dim, const void* q_vecs, int Q, const float* w,
                                          const int32_t* coo_keys, const void* coo_vals, int coo_dtype,
                                          const int64_t* field_offsets_host, int n_sparse, int64_t doc_id_base,
                                          const uint32_t* filter_bits, int filter_rows, int64_t filter_ld, int k,
                                          uint64_t* out_keys, float* out_scores, int64_t* out_ids, void* workspace,
                                          size_t workspace_bytes, int impl, void* stream);
/* mfar_score_topk_bm25 with a doc filter (no reference counterpart, DESIGN §4.5) */
MFAR_API int mfar_score_topk_bm25_filtered(const void* corpus, int64_t n_docs, int corpus_fields, int field_begin,
                                           int n_dense, int dim, const void* q_vecs, int Q, const float* w,
                                           const void* const* indptr_host, const void* const* indices_host,
                                           const void* const* data_host, const int32_t* vocab_host, int n_sparse,
                                           const int32_t* entries, int64_t n_entries, int64_t doc_id_base,
                                           const uint32_t* filter_bits, int filter_rows, int64_t filter_ld, int k,
                                           uint64_t* out_keys, float* out_scores, int64_t* out_ids, void* workspace,
                                           size_t workspace_bytes, int impl, void* stream);
/* mfar_score_topk_e4m3 with a doc filter (no reference counterpart, DESIGN §4.5) */
MFAR_API int mfar_score_topk_e4m3_filtered(const void* corpus, const float* corpus_scales, int64_t n_docs,
                                           int corpus_fields, int field_begin, int n_dense, int dim,
                                           const void* q_vecs, const float* q_scales, int Q, const float* w,
                                           const void* sparse, int n_sparse, int sparse_dtype, int64_t sparse_ld,
                                           int64_t doc_id_base, const uint32_t* filter_bits, int filter_rows,
                                           int64_t filter_ld, int k, uint64_t* out_keys, float* out_scores,
                                           int64_t* out_ids, void* workspace, size_t workspace_bytes, int impl,
                                           void* stream);
/* mfar_score_topk_coo_e4m3 with a doc filter (no reference counterpart, DESIGN §4.5) */
MFAR_API int mfar_score_topk_coo_e4m3_filtered(const void* corpus, const float* corpus_scales, int64_t n_docs,
                                               int corpus_fields, int field_begin, int n_dense, int dim,
                                               const void* q_vecs, const float* q_scales, int Q, const float* w,
                                               const int32_t* coo_keys, const void* coo_vals, int coo_dtype,
                                               const int64_t* field_offsets_host, int n_sparse, int64_t doc_id_base,
                                               const uint32_t* filter_bits, int filter_rows, int64_t filter_ld, int k,
                                               uint64_t* out_keys, float* out_scores, int64_t* out_ids,
                                               void* workspace, size_t workspace_bytes, int impl, void* stream);
/* mfar_score_topk_bm25_e4m3 with a doc filter (no reference counterpart, DESIGN §4.5) */
MFAR_API int mfar_score_topk_bm25_e4m3_filtered(const void* corpus, const float* corpus_scales, int64_t n_docs,
                                                int corpus_fields, int field_begin, int n_dense, int dim,
                                                const void* q_vecs, const float* q_scales, int Q, const float* w,
                                                const void* const* indptr_host, const void* const* indices_host,
                                                const void* const* data_host, const int32_t* vocab_host,
                                                int n_sparse, const int32_t* entries, int64_t n_entries,
                                                int64_t doc_id_base, const uint32_t* filter_bits, int filter_rows,
                                                int64_t filter_ld, int k, uint64_t* out_keys, float* out_scores,
                                                int64_t* out_ids, void* workspace, size_t workspace_bytes, int impl,
                                                void* stream);

/* Merge L sorted-or-unsorted key lists per query into the global top-k.  Used for (a) the
 * per-CTA partial lists inside mfar_score_topk and (b) the per-shard lists after the NCCL
 * all-gather (replaces the {rank}.qres file merge of mfar/modeling/contrastive.py:616-631).
 * keys: uint64 [L, Q, k_in]; key 0 = empty slot. */
MFAR_API int mfar_topk_merge(const uint64_t* keys, int L, int Q, int k_in, int k, uint64_t* out_keys,
                    float* out_scores, int64_t* out_ids, void* stream);

/* Cross-GPU exchange + merge in one kernel over NVLink peer memory (no NCCL call on the data path): every rank pushes
 * its [Q,k_in] keys into all peers' exchange buffers, waits for theirs, merges.  Replaces, together with
 * mfar_score_topk, the {rank}.qres file exchange of mfar/modeling/contrastive.py:566-581,616-631.
 *   peer_buffers_host: HOST array of `world` device addresses; entry r = rank r's exchange buffer as mapped into
 *     THIS process (CUDA VMM / IPC; torch.distributed._symmetric_memory provides them), each of
 *     mfar_exchange_buffer_bytes(world, q_cap, k_cap) bytes, zero-filled once before the first call;
 *   epoch: 1, 2, 3, ... - must increase by one per call, identically on every rank (slot = epoch % MFAR_EXCHANGE_SLOTS);
 *   every rank must call with the same Q, k_in, k.  world <= 8, world * k_in <= 1024. */
MFAR_API size_t mfar_exchange_buffer_bytes(int world, int q_cap, int k_cap);
MFAR_API int mfar_topk_exchange_merge(const uint64_t* local_keys, int Q, int k_in, int k, int rank, int world,
                             const uint64_t* peer_buffers_host, int q_cap, int k_cap, int epoch, uint64_t* out_keys,
                             float* out_scores, int64_t* out_ids, void* stream);
/* Same exchange with the call counter kept in DEVICE memory (epoch_dev: int32 [1 + MFAR_EXCHANGE_SLOTS], zero before the
 * first call, owned by the caller: word 0 = the counter, words 1.. = the batch size each slot's epoch was pushed with):
 * the call enqueues a one-thread kernel that increments it, then the exchange kernel that reads it - no host-side value
 * is baked into the launch, so the whole sharded step (mixture weights, scoring, local merge, exchange) can be captured
 * once in a CUDA graph and replayed.  Every rank must issue the same number of calls. */
MFAR_API int mfar_topk_exchange_merge_dev_epoch(const uint64_t* local_keys, int Q, int k_in, int k, int rank, int world,
                                       const uint64_t* peer_buffers_host, int q_cap, int k_cap, int32_t* epoch_dev,
                                       uint64_t* out_keys, float* out_scores, int64_t* out_ids, void* stream);
/* The exchange in two halves, for a PIPELINED sharded step: `push` opens a new epoch (increments *epoch_dev) and stores
 * this rank's keys into every rank's buffer without waiting for anybody; `wait_merge(lag)` merges epoch
 * (*epoch_dev - lag) - lag 0: the epoch just pushed (push + wait_merge(0) == mfar_topk_exchange_merge_dev_epoch),
 * lag 1: the previous one.  A step that pushes its own keys and merges the PREVIOUS step's never waits for the slowest
 * rank of the current step: the peers' pushes it needs landed a whole step ago.  Results then trail the inputs by one
 * call; the first wait_merge(1) (epoch 0) returns empty lists; finish a stream of batches with wait_merge(0).
 * k_in must not change between a push and the wait_merge that reads it; after a change of Q a lag-1 merge returns empty
 * lists for the queries the previous epoch did not push. */
MFAR_API int mfar_topk_exchange_push(const uint64_t* local_keys, int Q, int k_in, int rank, int world,
                            const uint64_t* peer_buffers_host, int q_cap, int k_cap, int32_t* epoch_dev, void* stream);
MFAR_API int mfar_topk_exchange_wait_merge(int Q, int k_in, int k, int rank, int world, const uint64_t* peer_buffers_host,
                                  int q_cap, int k_cap, const int32_t* epoch_dev, int lag, uint64_t* out_keys,
                                  float* out_scores, int64_t* out_ids, void* stream);

/* The candidate stage of trec_eval_step (mfar/modeling/contrastive.py:676-696) for a whole batch in one launch: per
 * query the union of the per-field hit lists (678-679), the re-scoring of that union under every field (681-683,
 * DenseFlatIndex.score_batch / BM25sSparseIndex.score_batch), mask + mixture (685-694, folded into w) and the final
 * top-k (696).
 *   cand_rows : int64 [n_lists, Q, k_in] LOCAL doc rows, one list per field index as retrieve_batch returned them
 *               (rows < 0 or >= n_docs are ignored); n_lists * k_in <= 8192;
 *   w         : fp32 [Q, n_dense + n_sparse] = softmax(q@W) * mask (mfar_mixture_weights);
 *   sparse    : [Q, n_sparse, sparse_ld] f16/f32 stored per-field scores of this shard's docs (or NULL);
 *   out_scores fp32 [Q,k], out_rows int64 [Q,k] (local rows; score desc, row asc), out_union_size int32 [Q] = size of
 *   each query's union - where it is below k the reference's torch.topk raises, and the tail is (-inf, -1) here. */
MFAR_API int mfar_union_rescore(const void* corpus, int64_t n_docs, int corpus_fields, int n_dense, int dim,
                       const void* q_vecs, int Q, const float* w, const void* sparse, int n_sparse, int sparse_dtype,
                       int64_t sparse_ld, const int64_t* cand_rows, int n_lists, int k_in, int k, float* out_scores,
                       int64_t* out_rows, int32_t* out_union_size, void* stream);

/* Reference quirk, mfar/data/index.py:192-193: the running top-k starts as k entries of
 * (score 0.0, row 0).  Applies that to a finished [Q,k] result in place: entries scoring
 * below 0.0 are replaced by (0.0, 0) and the list re-sorted. */
MFAR_API int mfar_topk_apply_zero_init(float* scores, int64_t* ids, int Q, int k, void* stream);

/* ------------------------------------------------------------------------------------------
 * Candidate re-scoring.  Replaces DenseFlatIndex.score_batch (mfar/data/index.py:227-232) and
 * BM25sSparseIndex.score_batch's gather (index.py:116-117) for the union_rescore mode of
 * trec_eval_step (contrastive.py:681-683).
 *   out[f, q, c] = <q_vec[q], corpus[rows[c], field_begin+f]>      rows[c] < 0 -> 0
 * ------------------------------------------------------------------------------------------ */
MFAR_API int mfar_score_candidates(const void* corpus, int64_t n_docs, int corpus_fields, int field_begin,
                          int n_fields, int dim, const void* q_vecs, int Q, const int64_t* rows, int C,
                          float* out, void* stream);
/* The same on an E4M3 corpus and E4M3 queries:  out[f, q, c] = (D * q_scales[q]) * corpus_scales[rows[c], f]. */
MFAR_API int mfar_score_candidates_e4m3(const void* corpus, const float* corpus_scales, int64_t n_docs,
                                        int corpus_fields, int field_begin, int n_fields, int dim, const void* q_vecs,
                                        const float* q_scales, int Q, const int64_t* rows, int C, float* out,
                                        void* stream);

/* ------------------------------------------------------------------------------------------
 * Host-buffer convenience call (the end-to-end path a reference-side caller uses): copies the
 * per-batch inputs host->device, runs mixture weights + mfar_score_topk on `stream`, copies the
 * [Q,k] result back and synchronises the stream.  The corpus stays resident on the device.
 * q_vecs_host: bf16 [Q,dim]; q_emb_host: fp32 [Q,E] (NULL if !query_cond); W/mask: DEVICE
 * pointers (model state); sparse_host may be NULL.  scratch: device buffer of at least
 * mfar_search_host_scratch_bytes(...) bytes.
 * ------------------------------------------------------------------------------------------ */
MFAR_API size_t mfar_search_host_scratch_bytes(int Q, int dim, int E, int n_dense, int n_sparse, int64_t n_docs,
                                      int sparse_dtype, int k);

MFAR_API int mfar_search_host(const void* corpus, int64_t n_docs, int corpus_fields, int field_begin, int n_dense,
                     int dim, const void* q_vecs_host, const float* q_emb_host, int Q, int E, const float* W,
                     const float* mask, int query_cond, const void* sparse_host, int n_sparse,
                     int sparse_dtype, int64_t doc_id_base, int k, float* out_scores_host,
                     int64_t* out_ids_host, void* scratch, size_t scratch_bytes, int impl, void* stream);

/* Host-buffer call for hybrid retrieval with device-resident BM25 indices: per batch only the query vectors,
 * the query embedding and the token entries (HOST int32 [n_entries,3]) cross PCIe - not a [Q,F_s,N] score tensor. */
MFAR_API size_t mfar_search_host_bm25_scratch_bytes(int Q, int dim, int E, int n_dense, int n_sparse, int64_t n_docs,
                                                    int64_t n_entries, int k);

MFAR_API int mfar_search_host_bm25(const void* corpus, int64_t n_docs, int corpus_fields, int field_begin,
                                   int n_dense, int dim, const void* q_vecs_host, const float* q_emb_host, int Q,
                                   int E, const float* W, const float* mask, int query_cond,
                                   const void* const* indptr_host, const void* const* indices_host,
                                   const void* const* data_host, const int32_t* vocab_host, int n_sparse,
                                   const int32_t* entries_host, int64_t n_entries, int64_t doc_id_base, int k,
                                   float* out_scores_host, int64_t* out_ids_host, void* scratch,
                                   size_t scratch_bytes, int impl, void* stream);

/* ------------------------------------------------------------------------------------------
 * Training-time scorer (fp32, forward + backward).  Replaces
 *   DecomposedContrastiveLoss.compute_query_doc_field_components   mfar/modeling/losses.py:176-188
 *   DecomposedContrastiveLoss.compute_doc_query_scores             mfar/modeling/losses.py:199-202
 *   the autograd of LinearWeights.forward                          mfar/modeling/weighting.py:17-29
 * Doc n = (p, s) with p = n / inner, s = n % inner; the E-vector of (doc n, field f) starts at
 * docs + p*stride_p + f*stride_f + s*stride_s (in elements): d_pos [P,F,E] is inner = 1, stride_p = F*E,
 * stride_f = E; d_neg [P,F,Neg,E] is inner = Neg, stride_p = F*Neg*E, stride_f = Neg*E, stride_s = E, which yields
 * the doc order of d_neg.permute(0,2,1,3).view(1, P*Neg, F, E) (losses.py:186) without a copy.
 * E % 4 == 0, E <= 1024, rows 16-byte aligned.
 * ------------------------------------------------------------------------------------------ */
/* comp[b, n, f] = <q[b,:], doc[n,f,:]> / temperature            comp: fp32 [B, N, F] */
MFAR_API int mfar_field_components_fwd(const float* q, int B, int E, const float* docs, int64_t N, int F,
                                       int64_t inner, int64_t stride_p, int64_t stride_f, int64_t stride_s,
                                       float temperature, float* comp, void* stream);
/* dq[b,:]     = sum_{n,f} dcomp[b,n,f] * doc[n,f,:] / temperature      (dq: fp32 [B,E], overwritten; may be NULL)
 * ddocs[n,f,:] = sum_b    dcomp[b,n,f] * q[b,:]     / temperature      (ddocs: same layout as docs; may be NULL) */
MFAR_API int mfar_field_components_bwd(const float* q, int B, int E, const float* docs, int64_t N, int F,
                                       int64_t inner, int64_t stride_p, int64_t stride_f, int64_t stride_s,
                                       float temperature, const float* dcomp, float* dq, float* ddocs, void* stream);
/* Backward of out[b,s] = sum_f w[b,f] x[b,s,f], w = softmax(q_emb @ W) (query_cond) or softmax(W^T) (W is [F,1]):
 *   dx[b,s,f] = g[b,s] w[b,f]            (dx may be NULL)
 *   dW        = q_emb^T dlogit  ([E,F])  or  sum_b dlogit[b,:] ([F,1]),   dlogit = softmax backward of sum_s g x
 *   dq[b,:]   = dlogit[b,:] W^T          (query_cond only; may be NULL)
 * w: the forward's weights, fp32 [w_rows, F] with w_rows = B or 1 (mfar_mixture_weights without a mask);
 * dlogit_scratch: fp32 [B, F]. */
MFAR_API int mfar_mixture_bwd(const float* x, const float* q_emb, const float* W, const float* w, int w_rows,
                              const float* g, int B, int S, int E, int F, int query_cond, float* dx, float* dW,
                              float* dq, float* dlogit_scratch, void* stream);

/* Number of kernels the last mfar_score_topk call on this thread launched (bench bookkeeping). */
MFAR_API int mfar_last_launch_count(void);

/* Per-launch device timing of the scoring kernel (the dominant kernel of a step), for the roofline
 * bench.py reports.  mfar_profile_enable(1) arms a ring of 256 CUDA event pairs recorded on the launch
 * stream around the scoring launches of each subsequent mfar_score_topk call (the main pass and, where threshold
 * seeding applies, its one or two prefix passes with their small merge / seed kernels in between - together they read
 * the corpus exactly once); mfar_profile_collect()
 * synchronises those events, writes their durations (ms) to a HOST array, returns how many, and
 * resets the ring.  Diagnostics only.  The ring is per host thread (thread-local state, events on the thread's current
 * device): arm and collect it from the thread that issues the calls; other threads / devices are unaffected.  It is off
 * by default and the compute entry points never depend on it. */
MFAR_API int mfar_profile_enable(int on);
MFAR_API int mfar_profile_collect(float* out_ms_host, int max_n);
/* CTAs of the large-batch scoring kernel that ran in 4-CTA clusters (two CTA pairs sharing every doc tile by TMA
 * multicast) on the current device since the previous call, which resets the count; -1 on a CUDA error.  Synchronous.
 * Diagnostics only: the count is kept whether profiling is armed or not. */
MFAR_API long long mfar_profile_cluster4_ctas(void);

#ifdef __cplusplus
}
#endif
#endif /* MFAR_B200_H_ */
