// Internal launcher declarations (host side).  Each returns an mfar_status.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/mfar_b200.h"

namespace mfar {

// BM25 postings of every sparse field (device pointers), passed to kernels by value.
struct Bm25Fields {
  const long long* indptr[MFAR_MAX_FIELDS];   // int64 [V_j + 1]
  const int* indices[MFAR_MAX_FIELDS];        // int32 [nnz_j] local doc rows
  const float* data[MFAR_MAX_FIELDS];         // fp32  [nnz_j]
  int vocab[MFAR_MAX_FIELDS];                 // V_j
};
int launch_bm25_plan(const int* entries, long long n_entries, const Bm25Fields& f, int n_sparse, int Q,
                     long long* ent_first, long long* flat_start, cudaStream_t st);
int launch_bm25_scatter(const int* entries, long long n_entries, const long long* ent_first,
                        const long long* flat_start, const Bm25Fields& f, const float* w, int w_ld, int w_off,
                        long long n_docs, float* base, long long base_ld, cudaStream_t st);
int launch_bm25_build_scores(const int* post_token, const int* post_doc, const int* post_tf, long long nnz,
                             const int* df, const int* doc_len, long long n_docs_total, double l_avg, double k1,
                             double b, float* data, cudaStream_t st);

// Dense score rows -> COO pairs in the reference's precomputed-BM25 file layout (sparse_coo.cu).
long long sparse_coo_segments(long long n_docs);
int launch_sparse_coo_count(const float* scores, long long ld, int Q, long long n_docs, const uint32_t* safe_bits,
                            long long doc_id_base, long long* seg_offsets, cudaStream_t st);
int launch_sparse_coo_write(const float* scores, long long ld, int Q, long long n_docs, const uint32_t* safe_bits,
                            const int* qids, long long doc_id_base, const long long* seg_offsets, int* out_keys,
                            void* out_vals, int vals_dtype, cudaStream_t st);

int launch_pack_rows(const void* src, int src_dtype, int64_t n_rows, int64_t row_begin, void* packed,
                     int n_fields, int field, int dim, int normalize, cudaStream_t st);
int launch_unpack_rows(const void* packed, int n_fields, int field, int dim, int64_t row_begin, int64_t n_rows,
                       float* dst, cudaStream_t st);
int launch_pack_rows_e4m3(const void* src, int src_dtype, int64_t n_rows, int64_t row_begin, uint8_t* payload,
                          float* scales, int n_fields, int field, int dim, int normalize, cudaStream_t st);
int launch_unpack_rows_e4m3(const uint8_t* payload, const float* scales, int n_fields, int field, int dim,
                            int64_t row_begin, int64_t n_rows, float* dst, cudaStream_t st);
int launch_mixture_weights(const float* q_emb, const float* W, const float* mask, int Q, int E, int F,
                           int query_cond, float* out_w, cudaStream_t st);
int launch_mixture_apply(const float* x, const float* w, int B, int S, int F, int w_rows, float* out,
                         cudaStream_t st);
// corpus_scales / q_scales: nullptr for a bf16 corpus, the row scales of an E4M3 corpus and its queries otherwise
int launch_score_candidates(const void* corpus, const float* corpus_scales, int64_t n_docs, int corpus_fields,
                            int field_begin, int n_fields, int dim, const void* q_vecs, const float* q_scales, int Q,
                            const int64_t* rows, int C, float* out, cudaStream_t st);
int launch_sparse_premix(const void* sparse, int sparse_dtype, int64_t sparse_ld, int n_sparse, const float* w,
                         int w_ld, int w_off, int Q, int64_t n_docs, float* base, int64_t base_ld,
                         cudaStream_t st);
int launch_sparse_premix_coo(const int32_t* keys, const void* vals, int val_dtype, const int64_t* field_offsets_host,
                             int n_sparse, const float* w, int w_ld, int w_off, int Q, int64_t doc_id_base,
                             int64_t n_docs, float* base, int64_t base_ld, cudaStream_t st);
// extra / extra_n: one more list per query, [Q, extra_n] keys (0 = empty slot), or nullptr
int launch_merge(const uint64_t* keys, const int* counts, const uint64_t* thr, int L, int q_stride, int slots, int Q,
                 int k, uint64_t* out_keys, float* out_scores, int64_t* out_ids, cudaStream_t st,
                 const uint64_t* extra = nullptr, int extra_n = 0);
int launch_zero_init(float* scores, int64_t* ids, int n, cudaStream_t st);
// union of per-field candidate lists + gather-rescore + mixture + top-k for a whole batch (union_rescore.cu)
int launch_union_rescore(const void* corpus, int64_t n_docs, int corpus_fields, int n_dense, int dim, const void* q_vecs,
                         int Q, const float* w, int w_ld, const void* sparse, int sparse_dtype, int64_t sparse_ld,
                         int n_sparse, const int64_t* cand, int L, int k_in, int k_out, float* out_scores,
                         int64_t* out_rows, int* out_union, cudaStream_t st);
int launch_exchange_merge(const uint64_t* local_keys, int Q, int k_in, int k, int rank, int world,
                          const unsigned long long* peer_bases, int q_cap, int k_cap, int epoch, int* epoch_dev, int mode,
                          int lag, uint64_t* out_keys, float* out_scores, int64_t* out_ids, cudaStream_t st);

// Training-time scorer (train.cu).  Doc n = (p, s), p = n / inner, s = n % inner, row of field f at
// docs + p*stride_p + f*stride_f + s*stride_s (elements).
struct DocLayout { long long inner, stride_p, stride_f, stride_s; };
int launch_field_components_fwd(const float* q, int B, int E, const float* docs, long long N, int F,
                                const DocLayout& L, float temperature, float* comp, cudaStream_t st);
int launch_field_components_bwd(const float* q, int B, int E, const float* docs, long long N, int F,
                                const DocLayout& L, float temperature, const float* dcomp, float* dq, float* ddocs,
                                cudaStream_t st);
int launch_mixture_bwd(const float* x, const float* q, const float* W, const float* w, int w_rows, const float* g,
                       int B, int S, int E, int F, int query_cond, float* dx, float* dW, float* dq, float* dlogit,
                       cudaStream_t st);

// Arguments common to both scoring kernels (all device pointers).
struct ScoreArgs {
  const void* corpus;       // packed bf16 [tiles][corpus_fields][128][dim], or E4M3 bytes (corpus_dtype == MFAR_E4M3)
  int corpus_dtype;         // MFAR_BF16 or MFAR_E4M3 (queries have the corpus's type)
  const float* corpus_scales;   // E4M3: fp32 [tiles][corpus_fields][128] row scales (powers of two), else nullptr
  const float* q_scales;        // E4M3: fp32 [Q] query scales, else nullptr
  int64_t n_docs;
  int n_tiles;
  int corpus_fields;
  int field_begin;
  int n_dense;
  int dim;
  const void* q_vecs;       // bf16 / E4M3 [Q, dim]
  int Q;
  const float* w;           // fp32 [Q, w_ld]
  int w_ld;
  const float* base;        // fp32 [Q, base_ld] pre-mixed sparse contribution or nullptr
  int64_t base_ld;
  // per-field sparse scores gathered INSIDE the scoring epilogue (tensor-core kernels; dense [Q, n_sparse, sparse_ld]
  // input with 32-byte aligned rows): acc starts as sum_j w[q, n_dense + j] * sparse[q, j, n].  Exclusive with base.
  const void* sparse;
  int sparse_dtype;         // MFAR_F16 / MFAR_F32
  int64_t sparse_ld;
  int64_t sparse_cols;      // valid columns of a row counted from `sparse` (0 = sparse_ld; smaller when the pointer has been
                            // advanced past a scored prefix, capi.cu)
  int n_sparse;
  int64_t doc_id_base;
  int k;
  // optional per-query admission thresholds known before the pass starts (packed keys, [Q], 0 = none): copied into the
  // workspace's shared threshold words right after they are zeroed (score_topk_core's prefix pass)
  const unsigned long long* gthr_seed;
  // optional doc filter (bitmap over GLOBAL doc ids, common.cuh): indexed by doc_id_base + local doc, so moving
  // doc_id_base past a scored prefix (skip_tiles) moves the filter with it
  const uint32_t* filter_bits;   // nullptr: every doc is eligible
  int64_t filter_stride;         // words between the rows of consecutive queries: 0 (one shared row) or the row length
  int filter_words;              // ceil((doc_id_base + n_docs) / 32): the words of a row that hold docs of the shard
};

// gthr[q] = seed[q] (after the workspace tail was zeroed)
int launch_seed_gthr(unsigned long long* gthr, const unsigned long long* seed, int Q, cudaStream_t st);
// seed[q] = keys[q, k-1] - 1 (the k-th best key of a prefix, made exclusive), 0 when the prefix holds fewer than k docs
int launch_seed_from_keys(const uint64_t* keys, int Q, int k, unsigned long long* seed, cudaStream_t st);

constexpr int kImplRows = 100;    // pass kind of sparse-only scorers (no dense field): streaming top-k of the base rows

// One scoring pass's launch geometry and candidate-list layout, filled completely by its kind's plan_* function.  The
// workspace is carved for (lists, q_pad_total) once per pass: the kernel writes its lists there and the merge reads them.
struct PassPlan {
  int impl;           // MFAR_IMPL_SIMT, MFAR_IMPL_TCGEN05, MFAR_IMPL_TCGEN05_QS or kImplRows
  int workers;        // doc-side grid size (rows: segments per query)
  int q_tiles;
  int q_pad;          // queries per tile (tc, qs), or all queries padded (simt, rows)
  int q_pad_total;    // q_pad * q_tiles
  int cg;             // qs: CTAs per MMA group (1 or 2)
  int lists;          // candidate lists per query: workers, or 2 x workers (qs: two epilogue sets)
  long long seg_docs; // rows: docs per segment
};
PassPlan plan_score_simt(int Q, int n_tiles);
PassPlan plan_score_tc(int Q, int n_tiles);
PassPlan plan_score_qs(int Q, int n_tiles, int n_dense);
PassPlan plan_topk_rows(int Q, long long n_docs);

// The scoring passes.  Each fills the candidate lists of `ws` (carved from `plan`, its tail zeroed and seeded by the
// caller where the kind reads it) and adds the kernels it enqueued to *launches.
struct TopkWorkspace;
// SIMT (CUDA-core) scoring pass.
int launch_score_simt(const ScoreArgs& a, const PassPlan& plan, const TopkWorkspace& ws, cudaStream_t st,
                      int* launches);
// TMA + tcgen05 scoring pass.
int launch_score_tc(const ScoreArgs& a, const PassPlan& plan, const TopkWorkspace& ws, cudaStream_t st,
                    int* launches);
// Query-stationary tcgen05 pass for large batches (queries resident in TMEM, CTA pairs when cg == 2).
int launch_score_qs(const ScoreArgs& a, const PassPlan& plan, const TopkWorkspace& ws, cudaStream_t st,
                    int* launches);
// Streaming top-k of the pre-mixed fp32 score rows (sparse-only scorers: no dense field).
int launch_topk_rows(const ScoreArgs& a, const PassPlan& plan, const TopkWorkspace& ws, cudaStream_t st,
                     int* launches);
long long qs_cluster4_ctas_collect();   // CTAs that ran in 4-CTA clusters since the last call (resets); -1: CUDA error
bool score_qs_supported(const ScoreArgs& a);
// rows of a dense sparse-score tensor can be gathered by the scoring epilogues (32-byte vector loads)
inline bool sparse_rows_fusable(const void* sparse, int dtype, int64_t ld) {
  const int es = dtype == MFAR_F32 ? 4 : 2;
  return sparse != nullptr && (dtype == MFAR_F16 || dtype == MFAR_F32) && (ld * es) % 32 == 0 &&
         reinterpret_cast<uintptr_t>(sparse) % 32 == 0;
}
// Shape envelope of the tcgen05 path.
bool score_tc_supported(const ScoreArgs& a);

}  // namespace mfar
