// extern "C" entry points declared in include/mfar_b200.h.
#include <algorithm>

#include "common.cuh"
#include "kernels.h"

using namespace mfar;

static thread_local int t_last_launches = 0;

// Optional per-launch timing of the scoring kernel (bench.py's roofline): a ring of CUDA event pairs recorded
// on the launch stream around the scoring kernel only.  Off by default; costs two event records per call.
// The ring belongs to the calling host thread (thread_local): two threads driving two streams - or two devices - each
// see only their own launches; events are created on the thread's current device when profiling is switched on.
constexpr int kProfRing = 256;
static thread_local bool g_prof_on = false;
static thread_local cudaEvent_t g_prof_ev[kProfRing][2];
static thread_local int g_prof_dev = -1;     // device the events were created on (-1: none yet)
static thread_local int g_prof_n = 0;

// compute-capability check, cached per device (a process may drive several)
static int check_arch() {
  constexpr int kMaxDev = 64;
  static int cached[kMaxDev];                 // 0 = unknown, 1 = sm_100, 2 = other (benign race: idempotent writes)
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return MFAR_ERR_CUDA;
  if (dev >= 0 && dev < kMaxDev && cached[dev]) return cached[dev] == 1 ? MFAR_OK : MFAR_ERR_ARCH;
  int major = 0;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return MFAR_ERR_CUDA;
  if (dev >= 0 && dev < kMaxDev) cached[dev] = (major == 10) ? 1 : 2;
  return major == 10 ? MFAR_OK : MFAR_ERR_ARCH;
}

static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
static size_t seed_scratch_bytes(int Q, int k) {      // two [Q,k] key buffers (prefix levels alternate) + [Q] seeds
  return 2 * align_up(size_t(Q) * k * 8, 256) + align_up(size_t(Q) * 8, 256);
}

constexpr int kQsMinBatch = 65;   // AUTO: batches above 64 queries take the query-stationary kernel

#ifdef MFAR_DEBUG_SEED
static const unsigned long long* g_debug_seed = nullptr;
#endif

// The pass `impl` asks for (AUTO resolved), planned for `a`.
static PassPlan plan_pass(const ScoreArgs& a, int impl) {
  if (a.n_dense == 0) return plan_topk_rows(a.Q, a.n_docs);   // every impl request: there is nothing to contract
  if (impl == MFAR_IMPL_AUTO) {
    if (a.Q >= kQsMinBatch && score_qs_supported(a)) impl = MFAR_IMPL_TCGEN05_QS;
    else impl = score_tc_supported(a) ? MFAR_IMPL_TCGEN05 : MFAR_IMPL_SIMT;
  }
  if (impl == MFAR_IMPL_TCGEN05_QS) return plan_score_qs(a.Q, a.n_tiles, a.n_dense);
  if (impl == MFAR_IMPL_TCGEN05) return plan_score_tc(a.Q, a.n_tiles);
  return plan_score_simt(a.Q, a.n_tiles);
}

static size_t plan_workspace_bytes(const PassPlan& p) { return topk_workspace_bytes(p.lists, p.q_pad_total); }

// One scoring pass: carves the candidate lists of `plan` from `workspace` into *ws (the merge reads the same carve),
// zeroes the workspace tail and copies a.gthr_seed into the shared thresholds for the kinds that read them, and
// launches the pass.  Counts every kernel it enqueued in t_last_launches.
static int launch_pass(const ScoreArgs& a, const PassPlan& plan, void* workspace, cudaStream_t st,
                       TopkWorkspace* ws) {
  *ws = carve_workspace(workspace, plan.lists, plan.q_pad_total);
  int launches = 0;
  if (plan.impl != MFAR_IMPL_SIMT) {      // progress counters (score_qs lockstep), shared thresholds, pooled bounds
    MFAR_CUDA_OK(cudaMemsetAsync(ws->progress, 0, workspace_zero_bytes(ws->workers, ws->q_pad), st));
    if (a.gthr_seed) {
      if (int rc = launch_seed_gthr(ws->gthr, a.gthr_seed, a.Q, st)) return rc;
      ++launches;
    }
  }
  int rc;
  if (plan.impl == kImplRows) rc = launch_topk_rows(a, plan, *ws, st, &launches);
  else if (plan.impl == MFAR_IMPL_TCGEN05_QS) rc = launch_score_qs(a, plan, *ws, st, &launches);
  else if (plan.impl == MFAR_IMPL_TCGEN05) rc = launch_score_tc(a, plan, *ws, st, &launches);
  else rc = launch_score_simt(a, plan, *ws, st, &launches);
  if (rc) return rc;
  t_last_launches += launches;
  return MFAR_OK;
}

extern "C" {

int mfar_abi_version(void) { return MFAR_ABI_VERSION; }

const char* mfar_status_string(int status) {
  switch (status) {
    case MFAR_OK: return "ok";
    case MFAR_ERR_ARG: return "invalid argument (null / non-positive / misaligned)";
    case MFAR_ERR_SHAPE:
      return "shape outside the supported envelope (fields <= 64, k <= 128, doc_id_base + n_docs <= 2^32, dims the "
             "selected kernel supports)";
    case MFAR_ERR_ARCH: return "device is not sm_100 (no fallback path exists)";
    case MFAR_ERR_WORKSPACE: return "workspace too small";
    case MFAR_ERR_CUDA: return "CUDA call failed";
    case MFAR_ERR_K_RANGE: return "k out of range";
    default: return "unknown status";
  }
}

int mfar_device_check(int device) {
  int dev = device;
  if (dev < 0 && cudaGetDevice(&dev) != cudaSuccess) return MFAR_ERR_CUDA;
  int major = 0;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return MFAR_ERR_CUDA;
  return major == 10 ? MFAR_OK : MFAR_ERR_ARCH;
}

int64_t mfar_corpus_packed_elems(int64_t n_docs, int n_fields, int dim) {
  if (n_docs < 0 || n_fields <= 0 || dim <= 0) return -1;
  const int64_t tiles = (n_docs + kTileDocs - 1) / kTileDocs;
  return tiles * n_fields * kTileDocs * dim;
}

int mfar_corpus_pack_rows(const void* src, int src_dtype, int64_t n_rows, int64_t row_begin, void* packed,
                          int64_t n_docs, int n_fields, int field, int dim, int normalize, void* stream) {
  if (!src || !packed || n_rows < 0 || row_begin < 0 || row_begin + n_rows > n_docs) return MFAR_ERR_ARG;
  if (field < 0 || field >= n_fields || dim <= 0) return MFAR_ERR_SHAPE;
  if (int rc = check_arch()) return rc;
  return launch_pack_rows(src, src_dtype, n_rows, row_begin, packed, n_fields, field, dim, normalize,
                          static_cast<cudaStream_t>(stream));
}

int mfar_corpus_unpack_rows(const void* packed, int64_t n_docs, int n_fields, int field, int dim, int64_t row_begin,
                            int64_t n_rows, float* dst, void* stream) {
  if (!packed || !dst || n_rows < 0 || row_begin < 0 || row_begin + n_rows > n_docs) return MFAR_ERR_ARG;
  if (field < 0 || field >= n_fields || dim <= 0) return MFAR_ERR_SHAPE;
  if (int rc = check_arch()) return rc;
  return launch_unpack_rows(packed, n_fields, field, dim, row_begin, n_rows, dst, static_cast<cudaStream_t>(stream));
}

// Replaces, as mfar_corpus_pack_rows does, the per-field fp32 memmaps of mfar/modeling/contrastive.py:482-490 (read at
// mfar/data/index.py:196,230), stored at one byte per element.
int mfar_corpus_pack_rows_e4m3(const void* src, int src_dtype, int64_t n_rows, int64_t row_begin, uint8_t* payload,
                               float* scales, int64_t n_docs, int n_fields, int field, int dim, int normalize,
                               void* stream) {
  if (!src || !payload || !scales || n_rows < 0 || row_begin < 0 || row_begin + n_rows > n_docs) return MFAR_ERR_ARG;
  if (field < 0 || field >= n_fields || dim <= 0) return MFAR_ERR_SHAPE;
  if (int rc = check_arch()) return rc;
  return launch_pack_rows_e4m3(src, src_dtype, n_rows, row_begin, payload, scales, n_fields, field, dim, normalize,
                               static_cast<cudaStream_t>(stream));
}

int mfar_corpus_unpack_rows_e4m3(const uint8_t* payload, const float* scales, int64_t n_docs, int n_fields, int field,
                                 int dim, int64_t row_begin, int64_t n_rows, float* dst, void* stream) {
  if (!payload || !scales || !dst || n_rows < 0 || row_begin < 0 || row_begin + n_rows > n_docs) return MFAR_ERR_ARG;
  if (field < 0 || field >= n_fields || dim <= 0) return MFAR_ERR_SHAPE;
  if (int rc = check_arch()) return rc;
  return launch_unpack_rows_e4m3(payload, scales, n_fields, field, dim, row_begin, n_rows, dst,
                                 static_cast<cudaStream_t>(stream));
}

int mfar_mixture_weights(const float* q_emb, const float* W, const float* mask, int Q, int E, int F, int query_cond,
                         float* out_w, void* stream) {
  if (!W || !out_w || Q <= 0 || (query_cond && (!q_emb || E <= 0))) return MFAR_ERR_ARG;
  if (F <= 0 || F > MFAR_MAX_FIELDS) return MFAR_ERR_SHAPE;
  if (int rc = check_arch()) return rc;
  return launch_mixture_weights(q_emb, W, mask, Q, E, F, query_cond, out_w, static_cast<cudaStream_t>(stream));
}

int mfar_mixture_apply(const float* x, const float* w, int B, int S, int F, int w_rows, float* out, void* stream) {
  if (!x || !w || !out || B <= 0 || S < 0) return MFAR_ERR_ARG;
  if (F <= 0 || F > MFAR_MAX_FIELDS || (w_rows != 1 && w_rows != B)) return MFAR_ERR_SHAPE;
  if (int rc = check_arch()) return rc;
  return launch_mixture_apply(x, w, B, S, F, w_rows, out, static_cast<cudaStream_t>(stream));
}

size_t mfar_score_topk_workspace_bytes(int Q, int k, int64_t n_docs, int n_sparse) {
  if (Q <= 0 || n_docs < 0) return 0;
  (void)k;
  const int n_tiles = std::max(int((n_docs + kTileDocs - 1) / kTileDocs), 1);
  // the largest pass any call of this shape may plan; n_dense is not known here (plan_score_qs)
  size_t best = std::max({plan_workspace_bytes(plan_score_tc(Q, n_tiles)),
                          plan_workspace_bytes(plan_score_simt(Q, n_tiles)),
                          plan_workspace_bytes(plan_score_qs(Q, n_tiles, 0))});
  if (n_sparse > 0) best = std::max(best, plan_workspace_bytes(plan_topk_rows(Q, std::max<int64_t>(n_docs, 1))));
  size_t total = align_up(best, 256);
  if (n_sparse > 0) total += align_up(size_t(Q) * size_t(align_up(size_t(n_docs), kTileDocs)) * 4, 256);
  total += seed_scratch_bytes(Q, MFAR_MAX_K);         // threshold-seeding prefix pass
  return total;
}

// The n_sparse fields' scores: dense [Q,Fs,ld] rows, COO (query row, global doc row, value) grouped by field, or BM25
// postings + query tokens.  `status`: the layout's own argument checks, which run before every other check of a call.
enum SparseKind { kSparseNone, kSparseRows, kSparseCoo, kSparseBm25 };
struct SparseInput {
  int status = MFAR_OK; SparseKind kind = kSparseNone; int n_sparse = 0;
  const void* dense = nullptr; int dense_dtype = MFAR_F16; int64_t dense_ld = 0;
  const int32_t* coo_keys = nullptr; const void* coo_vals = nullptr; int coo_dtype = MFAR_F16;
  const int64_t* field_offsets_host = nullptr;
  Bm25Fields bm25{}; const int32_t* entries = nullptr; int64_t n_entries = 0;
};

static size_t bm25_plan_bytes(int64_t n_entries) {
  // ent_first [n] + flat_start [n+1], int64
  return align_up(size_t(2 * std::max<int64_t>(n_entries, 0) + 1) * 8, 256);
}

static int fill_bm25_fields(const void* const* indptr_host, const void* const* indices_host,
                            const void* const* data_host, const int32_t* vocab_host, int n_sparse, Bm25Fields* f) {
  if (!indptr_host || !indices_host || !data_host || !vocab_host) return MFAR_ERR_ARG;
  if (n_sparse <= 0 || n_sparse > MFAR_MAX_FIELDS) return MFAR_ERR_SHAPE;
  for (int j = 0; j < n_sparse; ++j) {
    if (!indptr_host[j] || vocab_host[j] < 0) return MFAR_ERR_ARG;
    f->indptr[j] = static_cast<const long long*>(indptr_host[j]);
    f->indices[j] = static_cast<const int*>(indices_host[j]);     // may be null for an empty field (nnz == 0)
    f->data[j] = static_cast<const float*>(data_host[j]);
    f->vocab[j] = vocab_host[j];
  }
  return MFAR_OK;
}

static SparseInput rows_input(const void* rows, int n_sparse, int dtype, int64_t ld) {
  SparseInput sp;
  sp.n_sparse = n_sparse;
  if (n_sparse > 0) { sp.kind = kSparseRows; sp.dense = rows; sp.dense_dtype = dtype; sp.dense_ld = ld; }
  return sp;
}

static SparseInput coo_input(const int32_t* coo_keys, const void* coo_vals, int coo_dtype,
                             const int64_t* field_offsets_host, int n_sparse) {
  SparseInput sp;
  sp.kind = kSparseCoo; sp.n_sparse = n_sparse; sp.field_offsets_host = field_offsets_host;
  sp.coo_keys = coo_keys; sp.coo_vals = coo_vals; sp.coo_dtype = coo_dtype;
  if (n_sparse <= 0 || !field_offsets_host) sp.status = MFAR_ERR_ARG;
  else if (field_offsets_host[n_sparse] > 0 && (!coo_keys || !coo_vals)) sp.status = MFAR_ERR_ARG;
  return sp;
}

static SparseInput bm25_input(const void* const* indptr_host, const void* const* indices_host,
                              const void* const* data_host, const int32_t* vocab_host, int n_sparse,
                              const int32_t* entries, int64_t n_entries) {
  SparseInput sp;
  sp.kind = kSparseBm25; sp.n_sparse = n_sparse; sp.entries = entries; sp.n_entries = n_entries;
  sp.status = fill_bm25_fields(indptr_host, indices_host, data_host, vocab_host, n_sparse, &sp.bm25);
  return sp;
}

// score_topk_core's dense operands, in the ScoreArgs fields the kernels read: bf16, or E4M3 with the row scales.
static ScoreArgs dense_operands(int dtype, const void* corpus, const float* corpus_scales, const void* q_vecs,
                                const float* q_scales) {
  ScoreArgs a{};
  a.corpus_dtype = dtype; a.corpus = corpus; a.corpus_scales = corpus_scales; a.q_vecs = q_vecs; a.q_scales = q_scales;
  return a;
}

// Moves every per-doc pointer and count of `a` past its first `tiles` tiles (the pass behind a seeding prefix).  A new
// per-doc field of ScoreArgs must be moved here too, or that pass scores the prefix twice and reads past the shard.
// (The doc filter is indexed by global doc id, doc_id_base + local doc: moving doc_id_base moves it.)
static void skip_tiles(ScoreArgs& a, int tiles) {
  const int64_t docs = int64_t(tiles) * kTileDocs;
  const size_t rows = size_t(tiles) * a.corpus_fields * kTileDocs;
  a.corpus = static_cast<const char*>(a.corpus) + rows * a.dim * (a.corpus_dtype == MFAR_E4M3 ? 1 : 2);
  if (a.corpus_scales) a.corpus_scales += rows;
  a.n_tiles -= tiles;
  a.n_docs -= docs;
  a.doc_id_base += docs;
  if (a.base) a.base += docs;
  if (a.sparse) {
    a.sparse = static_cast<const char*>(a.sparse) + size_t(docs) * (a.sparse_dtype == MFAR_F16 ? 2 : 4);
    a.sparse_cols = (a.sparse_cols ? a.sparse_cols : a.sparse_ld) - docs;
  }
}

// The doc filter of a *_filtered call: bitmap rows over global doc ids, `rows` = 1 (shared) or Q, `ld` words each.
struct FilterInput {
  bool on = false; const uint32_t* bits = nullptr; int rows = 0; int64_t ld = 0;
};

static FilterInput filter_input(const uint32_t* bits, int rows, int64_t ld) {
  FilterInput f;
  f.on = true; f.bits = bits; f.rows = rows; f.ld = ld;
  return f;
}

static int score_topk_core(ScoreArgs a, int64_t n_docs, int corpus_fields, int field_begin, int n_dense, int dim,
                           int Q, const float* w, const SparseInput& sp, int64_t doc_id_base, int k, uint64_t* out_keys,
                           float* out_scores, int64_t* out_ids, void* workspace, size_t workspace_bytes, int impl,
                           void* stream, const FilterInput& filt = FilterInput{}) {
  if (sp.status) return sp.status;
  const int n_sparse = sp.n_sparse;
  t_last_launches = 0;
  if (n_docs <= 0 || Q <= 0 || !w || !workspace || (!out_scores && !out_ids && !out_keys)) return MFAR_ERR_ARG;
  if (n_dense < 0 || n_sparse < 0 || n_dense + n_sparse <= 0 || n_dense + n_sparse > MFAR_MAX_FIELDS)
    return MFAR_ERR_SHAPE;
  if (n_dense > 0 && (!a.corpus || !a.q_vecs || dim <= 0 || field_begin < 0 || field_begin + n_dense > corpus_fields))
    return MFAR_ERR_ARG;
  if (n_dense > 0 && a.corpus_dtype == MFAR_E4M3 && (!a.corpus_scales || !a.q_scales)) return MFAR_ERR_ARG;
  if (n_sparse > 0 && sp.kind == kSparseRows && (!sp.dense || sp.dense_ld < n_docs)) return MFAR_ERR_ARG;
  if (n_sparse > 0 && sp.kind == kSparseCoo && (!sp.field_offsets_host || sp.field_offsets_host[0] != 0))
    return MFAR_ERR_ARG;
  if (n_sparse > 0 && sp.kind == kSparseBm25 && (sp.n_entries < 0 || (sp.n_entries > 0 && !sp.entries)))
    return MFAR_ERR_ARG;
  if (k <= 0 || k > MFAR_MAX_K) return MFAR_ERR_SHAPE;
  if (doc_id_base < 0 || doc_id_base + n_docs > (int64_t(1) << 32)) return MFAR_ERR_SHAPE;
  if (filt.on) {
    if (!filt.bits || reinterpret_cast<uintptr_t>(filt.bits) % 4 != 0 || (filt.rows != 1 && filt.rows != Q))
      return MFAR_ERR_ARG;
    if (filt.ld < (doc_id_base + n_docs + 31) / 32) return MFAR_ERR_SHAPE;   // a row covers every doc of the shard
  }
  if (impl < MFAR_IMPL_AUTO || impl > MFAR_IMPL_TCGEN05_QS) return MFAR_ERR_ARG;
  if (int rc = check_arch()) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);

  a.n_docs = n_docs; a.n_tiles = int((n_docs + kTileDocs - 1) / kTileDocs);
  a.corpus_fields = corpus_fields; a.field_begin = field_begin; a.n_dense = n_dense; a.dim = dim;
  a.Q = Q; a.w = w; a.w_ld = n_dense + n_sparse; a.doc_id_base = doc_id_base; a.k = k;
  if (filt.on) {
    a.filter_bits = filt.bits;
    a.filter_stride = filt.rows == 1 ? 0 : filt.ld;
    a.filter_words = int((doc_id_base + n_docs + 31) / 32);    // unchanged by skip_tiles
  }
  if (n_dense > 0 && impl == MFAR_IMPL_TCGEN05 && !score_tc_supported(a)) return MFAR_ERR_SHAPE;
  if (n_dense > 0 && impl == MFAR_IMPL_TCGEN05_QS && !score_qs_supported(a)) return MFAR_ERR_SHAPE;
  const PassPlan g = plan_pass(a, impl);

  const size_t ws_topk = align_up(plan_workspace_bytes(g), 256);
  const int64_t base_ld = int64_t(align_up(size_t(n_docs), kTileDocs));   // tile-wide vector reads stay in bounds
  // Dense [Q,Fs,ld] score rows are gathered and mixed INSIDE the tensor-core scoring epilogues (no [Q,N] intermediate
  // in HBM) when their rows are 32-byte aligned; COO pairs / BM25 postings scatter into the fp32 base block, and the
  // SIMT cross-check kernel and the sparse-only row scan read that block too.
  const bool fuse_sparse = n_sparse > 0 && sp.kind == kSparseRows && n_dense > 0 &&
                           (g.impl == MFAR_IMPL_TCGEN05 || g.impl == MFAR_IMPL_TCGEN05_QS) &&
                           sparse_rows_fusable(sp.dense, sp.dense_dtype, sp.dense_ld);
  const size_t ws_base = (n_sparse > 0 && !fuse_sparse) ? align_up(size_t(Q) * base_ld * 4, 256) : 0;
  const size_t ws_plan = (n_sparse > 0 && sp.kind == kSparseBm25) ? bm25_plan_bytes(sp.n_entries) : 0;
  // prefix keys 2 x [Q,k] + seed thresholds [Q] of the threshold-seeding passes (used when the caller's workspace has room)
  size_t ws_seed = seed_scratch_bytes(Q, k);
  if (workspace_bytes < ws_topk + ws_base + ws_plan) return MFAR_ERR_WORKSPACE;
  if (workspace_bytes < ws_topk + ws_base + ws_plan + ws_seed) ws_seed = 0;
  if (reinterpret_cast<uintptr_t>(workspace) % 256 != 0) return MFAR_ERR_ARG;

  if (fuse_sparse) {
    a.sparse = sp.dense; a.sparse_dtype = sp.dense_dtype; a.sparse_ld = sp.dense_ld; a.n_sparse = n_sparse;
  } else if (n_sparse > 0) {
    float* base = reinterpret_cast<float*>(static_cast<char*>(workspace) + ws_topk);
    if (sp.kind == kSparseRows) {
      if (int rc = launch_sparse_premix(sp.dense, sp.dense_dtype, sp.dense_ld, n_sparse, w, a.w_ld, n_dense, Q, n_docs,
                                        base, base_ld, st))
        return rc;
      ++t_last_launches;
    } else if (sp.kind == kSparseBm25) {
      MFAR_CUDA_OK(cudaMemsetAsync(base, 0, size_t(Q) * base_ld * 4, st));
      ++t_last_launches;
      if (sp.n_entries > 0) {
        long long* ent_first = reinterpret_cast<long long*>(static_cast<char*>(workspace) + ws_topk + ws_base);
        long long* flat_start = ent_first + sp.n_entries;
        if (int rc = launch_bm25_plan(sp.entries, sp.n_entries, sp.bm25, n_sparse, Q, ent_first, flat_start, st))
          return rc;
        if (int rc = launch_bm25_scatter(sp.entries, sp.n_entries, ent_first, flat_start, sp.bm25, w, a.w_ld, n_dense,
                                         n_docs, base, base_ld, st))
          return rc;
        t_last_launches += 2;
      }
    } else {
      MFAR_CUDA_OK(cudaMemsetAsync(base, 0, size_t(Q) * base_ld * 4, st));
      if (int rc = launch_sparse_premix_coo(sp.coo_keys, sp.coo_vals, sp.coo_dtype, sp.field_offsets_host, n_sparse, w,
                                            a.w_ld, n_dense, Q, doc_id_base, n_docs, base, base_ld, st))
        return rc;
      t_last_launches += 2;
    }
    a.base = base;
    a.base_ld = base_ld;
  }
  int rc;
  TopkWorkspace ws;
  // Threshold seeding (tensor-core kernels, shards of >= 16 tiles per CTA): the same kernel first scores a PREFIX of one
  // tile per CTA, the merge ranks it, and the k-th best key of the prefix (a valid lower bound of the shard's k-th key)
  // becomes every query's initial admission threshold.  Without it every candidate list fills unfiltered and is
  // compacted twice before the shared thresholds bite - 64 of the ~70 compactions per epilogue warp on a 700k-doc
  // shard, ~10 % of that kernel plus the tensor-pipe stalls behind them; the prefix costs ~0.1 ms.
  // Not for small batches: below ~32 queries there are few lists to compact and the prefix's fixed ~0.1 ms shows
  // (measured: MAG-shaped Q=64 step 1.04 -> 0.93 ms, Q=512 2.82 -> 2.74 ms, 1.25M-doc shard Q=512 6.92 -> 6.60 ms,
  // single_ Q=128 3.21 -> 2.73 ms; Q=1 0.81 -> 0.87 ms without this rule).
  const uint64_t* prefix_keys = nullptr;              // set when a scored prefix is left out of the main pass
  const bool seed = n_dense > 0 && (g.impl == MFAR_IMPL_TCGEN05 || g.impl == MFAR_IMPL_TCGEN05_QS) && Q >= 32 &&
                    a.n_tiles >= 16 * g.workers && ws_seed > 0;
  // the profiled interval covers every scoring launch of the call: the seeding passes are part of the corpus pass
  const bool prof = g_prof_on && g_prof_n < kProfRing;
  if (prof) MFAR_CUDA_OK(cudaEventRecord(g_prof_ev[g_prof_n][0], st));
  if (seed) {
    char* sb = static_cast<char*>(workspace) + ws_topk + ws_base + ws_plan;
    const size_t keys_bytes = align_up(size_t(Q) * k * 8, 256);
    uint64_t* pref_buf[2] = {reinterpret_cast<uint64_t*>(sb), reinterpret_cast<uint64_t*>(sb + keys_bytes)};
    unsigned long long* seed_thr = reinterpret_cast<unsigned long long*>(sb + 2 * keys_bytes);
    // Two prefix levels.  A: one tile per CTA, unseeded (a list takes its 128 docs without a compaction).  B: up to 31
    // more tiles per CTA admitted against A's threshold (k-th best of workers*128 docs: ~2 % pass at Q=512 where a
    // query has 37 lists, 0.5 % at Q<=64) - still no list fills - after which the seed is the k-th best of up to
    // 32*workers*128 docs (0.07 % / 0.02 %).  Measured with the TRUE k-th keys as the seed (tools/seed_potential.py): a
    // 1.25M-doc x 8-field shard at Q=512 runs 6.26 ms with A alone and 5.47 ms with a perfect seed, 5.49 ms with the
    // k-th keys of a 150k-doc prefix - the lists of a mid-size shard never fill, so their thresholds never tighten
    // by themselves and every weakly filtered doc costs the epilogue its slow path.
    // B only where A's threshold would still let a list fill during the main pass (expected admissions per list
    // n_docs * k / (docs of A) / lists above ~96): a 700k-doc shard at Q=64 has 148 lists per query and ~25 admissions
    // per list after A alone - there B's extra launch and merge cost 2 %.
    const int per_worker = a.n_tiles / g.workers;
    const double after_a = double(a.n_docs) * k / (double(g.workers) * kTileDocs) / double(g.lists);
    int level_tiles[2] = {1, std::min(31, per_worker / 4 - 1)};
    const int n_levels = (level_tiles[1] >= 3 && after_a > 96.0) ? 2 : 1;
    for (int lv = 0; lv < n_levels; ++lv) {
      ScoreArgs ap = a;                                 // `a` already starts behind the previous level
      ap.n_tiles = g.workers * level_tiles[lv];
      ap.n_docs = int64_t(ap.n_tiles) * kTileDocs;
      const PassPlan gp = plan_pass(ap, g.impl);
      if ((rc = launch_pass(ap, gp, workspace, st, &ws))) return rc;
      uint64_t* pref_keys = pref_buf[lv & 1];           // ranked top k of everything scored so far
      rc = launch_merge(ws.cand_keys, ws.cand_cnt, ws.cand_thr, ws.workers, ws.q_pad, kCandCap, Q, k, pref_keys,
                        nullptr, nullptr, st, prefix_keys, prefix_keys ? k : 0);
      if (rc) return rc;
      if ((rc = launch_seed_from_keys(pref_keys, Q, k, seed_thr, st))) return rc;
#ifdef MFAR_DEBUG_SEED   // experiment builds only: replace the prefix seed by thresholds the caller supplies
      if (g_debug_seed) MFAR_CUDA_OK(cudaMemcpyAsync(seed_thr, g_debug_seed, size_t(Q) * 8, cudaMemcpyDeviceToDevice, st));
#endif
      t_last_launches += 2;                             // merge + seed
      // A prefix is not scored twice: the next pass starts behind it and the next merge takes the prefix's ranked top
      // k as one more list.
      skip_tiles(a, ap.n_tiles);
      a.gthr_seed = seed_thr;
      prefix_keys = pref_keys;
    }
  }
  if ((rc = launch_pass(a, g, workspace, st, &ws))) return rc;
  if (prof) { MFAR_CUDA_OK(cudaEventRecord(g_prof_ev[g_prof_n][1], st)); ++g_prof_n; }
  rc = launch_merge(ws.cand_keys, ws.cand_cnt, ws.cand_thr, ws.workers, ws.q_pad, kCandCap, Q, k, out_keys,
                    out_scores, out_ids, st, prefix_keys, prefix_keys ? k : 0);
  if (rc) return rc;
  ++t_last_launches;
  return MFAR_OK;
}


int mfar_score_topk(const void* corpus, int64_t n_docs, int corpus_fields, int field_begin, int n_dense, int dim,
                    const void* q_vecs, int Q, const float* w, const void* sparse, int n_sparse, int sparse_dtype,
                    int64_t sparse_ld, int64_t doc_id_base, int k, uint64_t* out_keys, float* out_scores,
                    int64_t* out_ids, void* workspace, size_t workspace_bytes, int impl, void* stream) {
  return score_topk_core(dense_operands(MFAR_BF16, corpus, nullptr, q_vecs, nullptr), n_docs, corpus_fields,
                         field_begin, n_dense, dim, Q, w, rows_input(sparse, n_sparse, sparse_dtype, sparse_ld),
                         doc_id_base, k, out_keys, out_scores, out_ids, workspace, workspace_bytes, impl, stream);
}

// mfar_score_topk on an E4M3 corpus: the same reference lines (index.py:181-232, 111-118; contrastive.py:686,694,696)
int mfar_score_topk_e4m3(const void* corpus, const float* corpus_scales, int64_t n_docs, int corpus_fields,
                         int field_begin, int n_dense, int dim, const void* q_vecs, const float* q_scales, int Q,
                         const float* w, const void* sparse, int n_sparse, int sparse_dtype, int64_t sparse_ld,
                         int64_t doc_id_base, int k, uint64_t* out_keys, float* out_scores, int64_t* out_ids,
                         void* workspace, size_t workspace_bytes, int impl, void* stream) {
  return score_topk_core(dense_operands(MFAR_E4M3, corpus, corpus_scales, q_vecs, q_scales), n_docs, corpus_fields,
                         field_begin, n_dense, dim, Q, w, rows_input(sparse, n_sparse, sparse_dtype, sparse_ld),
                         doc_id_base, k, out_keys, out_scores, out_ids, workspace, workspace_bytes, impl, stream);
}

int mfar_score_topk_coo(const void* corpus, int64_t n_docs, int corpus_fields, int field_begin, int n_dense, int dim,
                        const void* q_vecs, int Q, const float* w, const int32_t* coo_keys, const void* coo_vals,
                        int coo_dtype, const int64_t* field_offsets_host, int n_sparse, int64_t doc_id_base, int k,
                        uint64_t* out_keys, float* out_scores, int64_t* out_ids, void* workspace,
                        size_t workspace_bytes, int impl, void* stream) {
  return score_topk_core(dense_operands(MFAR_BF16, corpus, nullptr, q_vecs, nullptr), n_docs, corpus_fields,
                         field_begin, n_dense, dim, Q, w,
                         coo_input(coo_keys, coo_vals, coo_dtype, field_offsets_host, n_sparse), doc_id_base, k,
                         out_keys, out_scores, out_ids, workspace, workspace_bytes, impl, stream);
}

// mfar_score_topk_coo on an E4M3 corpus (precompute_bm25s_scores.py:21-30, util.py:151-173, index.py:120-125)
int mfar_score_topk_coo_e4m3(const void* corpus, const float* corpus_scales, int64_t n_docs, int corpus_fields,
                             int field_begin, int n_dense, int dim, const void* q_vecs, const float* q_scales, int Q,
                             const float* w, const int32_t* coo_keys, const void* coo_vals, int coo_dtype,
                             const int64_t* field_offsets_host, int n_sparse, int64_t doc_id_base, int k,
                             uint64_t* out_keys, float* out_scores, int64_t* out_ids, void* workspace,
                             size_t workspace_bytes, int impl, void* stream) {
  return score_topk_core(dense_operands(MFAR_E4M3, corpus, corpus_scales, q_vecs, q_scales), n_docs, corpus_fields,
                         field_begin, n_dense, dim, Q, w,
                         coo_input(coo_keys, coo_vals, coo_dtype, field_offsets_host, n_sparse), doc_id_base, k,
                         out_keys, out_scores, out_ids, workspace, workspace_bytes, impl, stream);
}

int mfar_bm25_build_scores(const int32_t* post_token, const int32_t* post_doc, const int32_t* post_tf, int64_t nnz,
                           const int32_t* df, const int32_t* doc_len, int64_t n_docs_total, double l_avg, double k1,
                           double b, float* data, void* stream) {
  if (nnz < 0 || n_docs_total <= 0 || !(l_avg > 0.0)) return MFAR_ERR_ARG;
  if (nnz > 0 && (!post_token || !post_doc || !post_tf || !df || !doc_len || !data)) return MFAR_ERR_ARG;
  if (int rc = check_arch()) return rc;
  return launch_bm25_build_scores(post_token, post_doc, post_tf, nnz, df, doc_len, n_docs_total, l_avg, k1, b, data,
                                  static_cast<cudaStream_t>(stream));
}

size_t mfar_bm25_plan_bytes(int64_t n_entries) { return bm25_plan_bytes(n_entries); }

int mfar_bm25_scores(const void* const* indptr_host, const void* const* indices_host, const void* const* data_host,
                     const int32_t* vocab_host, int n_sparse, const int32_t* entries, int64_t n_entries, int Q,
                     const float* w, int w_ld, int w_off, int64_t n_docs, float* out, int64_t ld, int zero_first,
                     void* plan, size_t plan_bytes, void* stream) {
  t_last_launches = 0;
  if (!out || Q <= 0 || n_docs <= 0 || ld < n_docs || n_entries < 0 || (n_entries > 0 && (!entries || !plan)))
    return MFAR_ERR_ARG;
  if (w && (w_ld <= 0 || w_off < 0 || w_off + n_sparse > w_ld)) return MFAR_ERR_ARG;
  if (plan_bytes < bm25_plan_bytes(n_entries)) return MFAR_ERR_WORKSPACE;
  Bm25Fields f{};
  if (int rc = fill_bm25_fields(indptr_host, indices_host, data_host, vocab_host, n_sparse, &f)) return rc;
  if (int rc = check_arch()) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (zero_first) { MFAR_CUDA_OK(cudaMemsetAsync(out, 0, size_t(Q) * ld * 4, st)); ++t_last_launches; }
  if (n_entries == 0) return MFAR_OK;
  long long* ent_first = static_cast<long long*>(plan);
  long long* flat_start = ent_first + n_entries;
  if (int rc = launch_bm25_plan(entries, n_entries, f, n_sparse, Q, ent_first, flat_start, st)) return rc;
  if (int rc = launch_bm25_scatter(entries, n_entries, ent_first, flat_start, f, w, w_ld, w_off, n_docs, out, ld, st))
    return rc;
  t_last_launches += 2;
  return MFAR_OK;
}

static int check_sparse_coo(const float* scores, int64_t ld, int Q, int64_t n_docs, int64_t doc_id_base,
                            const void* seg_offsets) {
  if (!scores || !seg_offsets || Q <= 0 || n_docs <= 0 || ld < n_docs || doc_id_base < 0) return MFAR_ERR_ARG;
  if (doc_id_base + n_docs > int64_t(0x7fffffff) || Q > 65535) return MFAR_ERR_SHAPE;   // int32 doc ids in the files
  return MFAR_OK;
}

int64_t mfar_sparse_coo_offsets_len(int Q, int64_t n_docs) {
  if (Q <= 0 || n_docs <= 0) return 0;
  return int64_t(Q) * sparse_coo_segments(n_docs) + 1;
}

int mfar_sparse_coo_count(const float* scores, int64_t ld, int Q, int64_t n_docs, const uint32_t* safe_bits,
                          int64_t doc_id_base, int64_t* seg_offsets, void* stream) {
  t_last_launches = 0;
  if (int rc = check_sparse_coo(scores, ld, Q, n_docs, doc_id_base, seg_offsets)) return rc;
  if (int rc = check_arch()) return rc;
  if (int rc = launch_sparse_coo_count(scores, ld, Q, n_docs, safe_bits, doc_id_base,
                                       reinterpret_cast<long long*>(seg_offsets), static_cast<cudaStream_t>(stream)))
    return rc;
  t_last_launches = 2;
  return MFAR_OK;
}

int mfar_sparse_coo_write(const float* scores, int64_t ld, int Q, int64_t n_docs, const uint32_t* safe_bits,
                          const int32_t* qids, int64_t doc_id_base, const int64_t* seg_offsets, int32_t* out_keys,
                          void* out_vals, int vals_dtype, void* stream) {
  t_last_launches = 0;
  if (int rc = check_sparse_coo(scores, ld, Q, n_docs, doc_id_base, seg_offsets)) return rc;
  if (!out_keys || !out_vals || reinterpret_cast<uintptr_t>(out_keys) % 8 != 0) return MFAR_ERR_ARG;
  if (vals_dtype != MFAR_F16 && vals_dtype != MFAR_F32) return MFAR_ERR_ARG;
  if (int rc = check_arch()) return rc;
  if (int rc = launch_sparse_coo_write(scores, ld, Q, n_docs, safe_bits, qids, doc_id_base,
                                       reinterpret_cast<const long long*>(seg_offsets), out_keys, out_vals, vals_dtype,
                                       static_cast<cudaStream_t>(stream)))
    return rc;
  t_last_launches = 1;
  return MFAR_OK;
}

size_t mfar_score_topk_bm25_workspace_bytes(int Q, int k, int64_t n_docs, int n_sparse, int64_t n_entries) {
  const size_t b = mfar_score_topk_workspace_bytes(Q, k, n_docs, n_sparse);
  return b ? b + bm25_plan_bytes(n_entries) : 0;
}

int mfar_score_topk_bm25(const void* corpus, int64_t n_docs, int corpus_fields, int field_begin, int n_dense, int dim,
                         const void* q_vecs, int Q, const float* w, const void* const* indptr_host,
                         const void* const* indices_host, const void* const* data_host, const int32_t* vocab_host,
                         int n_sparse, const int32_t* entries, int64_t n_entries, int64_t doc_id_base, int k,
                         uint64_t* out_keys, float* out_scores, int64_t* out_ids, void* workspace,
                         size_t workspace_bytes, int impl, void* stream) {
  return score_topk_core(dense_operands(MFAR_BF16, corpus, nullptr, q_vecs, nullptr), n_docs, corpus_fields,
                         field_begin, n_dense, dim, Q, w,
                         bm25_input(indptr_host, indices_host, data_host, vocab_host, n_sparse, entries, n_entries),
                         doc_id_base, k, out_keys, out_scores, out_ids, workspace, workspace_bytes, impl, stream);
}

// mfar_score_topk_bm25 on an E4M3 corpus (index.py:72-76, 95-118 for the sparse fields)
int mfar_score_topk_bm25_e4m3(const void* corpus, const float* corpus_scales, int64_t n_docs, int corpus_fields,
                              int field_begin, int n_dense, int dim, const void* q_vecs, const float* q_scales, int Q,
                              const float* w, const void* const* indptr_host, const void* const* indices_host,
                              const void* const* data_host, const int32_t* vocab_host, int n_sparse,
                              const int32_t* entries, int64_t n_entries, int64_t doc_id_base, int k,
                              uint64_t* out_keys, float* out_scores, int64_t* out_ids, void* workspace,
                              size_t workspace_bytes, int impl, void* stream) {
  return score_topk_core(dense_operands(MFAR_E4M3, corpus, corpus_scales, q_vecs, q_scales), n_docs, corpus_fields,
                         field_begin, n_dense, dim, Q, w,
                         bm25_input(indptr_host, indices_host, data_host, vocab_host, n_sparse, entries, n_entries),
                         doc_id_base, k, out_keys, out_scores, out_ids, workspace, workspace_bytes, impl, stream);
}

// The six scoring entry points with a doc filter (filter_bits / filter_rows / filter_ld after doc_id_base): the same
// pass, in which a doc whose bit is clear never enters a candidate list.  No reference counterpart (DESIGN §4.5).
int mfar_score_topk_filtered(const void* corpus, int64_t n_docs, int corpus_fields, int field_begin, int n_dense,
                             int dim, const void* q_vecs, int Q, const float* w, const void* sparse, int n_sparse,
                             int sparse_dtype, int64_t sparse_ld, int64_t doc_id_base, const uint32_t* filter_bits,
                             int filter_rows, int64_t filter_ld, int k, uint64_t* out_keys, float* out_scores,
                             int64_t* out_ids, void* workspace, size_t workspace_bytes, int impl, void* stream) {
  return score_topk_core(dense_operands(MFAR_BF16, corpus, nullptr, q_vecs, nullptr), n_docs, corpus_fields,
                         field_begin, n_dense, dim, Q, w, rows_input(sparse, n_sparse, sparse_dtype, sparse_ld),
                         doc_id_base, k, out_keys, out_scores, out_ids, workspace, workspace_bytes, impl, stream,
                         filter_input(filter_bits, filter_rows, filter_ld));
}

int mfar_score_topk_e4m3_filtered(const void* corpus, const float* corpus_scales, int64_t n_docs, int corpus_fields,
                                  int field_begin, int n_dense, int dim, const void* q_vecs, const float* q_scales,
                                  int Q, const float* w, const void* sparse, int n_sparse, int sparse_dtype,
                                  int64_t sparse_ld, int64_t doc_id_base, const uint32_t* filter_bits,
                                  int filter_rows, int64_t filter_ld, int k, uint64_t* out_keys, float* out_scores,
                                  int64_t* out_ids, void* workspace, size_t workspace_bytes, int impl, void* stream) {
  return score_topk_core(dense_operands(MFAR_E4M3, corpus, corpus_scales, q_vecs, q_scales), n_docs, corpus_fields,
                         field_begin, n_dense, dim, Q, w, rows_input(sparse, n_sparse, sparse_dtype, sparse_ld),
                         doc_id_base, k, out_keys, out_scores, out_ids, workspace, workspace_bytes, impl, stream,
                         filter_input(filter_bits, filter_rows, filter_ld));
}

int mfar_score_topk_coo_filtered(const void* corpus, int64_t n_docs, int corpus_fields, int field_begin, int n_dense,
                                 int dim, const void* q_vecs, int Q, const float* w, const int32_t* coo_keys,
                                 const void* coo_vals, int coo_dtype, const int64_t* field_offsets_host, int n_sparse,
                                 int64_t doc_id_base, const uint32_t* filter_bits, int filter_rows, int64_t filter_ld,
                                 int k, uint64_t* out_keys, float* out_scores, int64_t* out_ids, void* workspace,
                                 size_t workspace_bytes, int impl, void* stream) {
  return score_topk_core(dense_operands(MFAR_BF16, corpus, nullptr, q_vecs, nullptr), n_docs, corpus_fields,
                         field_begin, n_dense, dim, Q, w,
                         coo_input(coo_keys, coo_vals, coo_dtype, field_offsets_host, n_sparse), doc_id_base, k,
                         out_keys, out_scores, out_ids, workspace, workspace_bytes, impl, stream,
                         filter_input(filter_bits, filter_rows, filter_ld));
}

int mfar_score_topk_coo_e4m3_filtered(const void* corpus, const float* corpus_scales, int64_t n_docs,
                                      int corpus_fields, int field_begin, int n_dense, int dim, const void* q_vecs,
                                      const float* q_scales, int Q, const float* w, const int32_t* coo_keys,
                                      const void* coo_vals, int coo_dtype, const int64_t* field_offsets_host,
                                      int n_sparse, int64_t doc_id_base, const uint32_t* filter_bits, int filter_rows,
                                      int64_t filter_ld, int k, uint64_t* out_keys, float* out_scores,
                                      int64_t* out_ids, void* workspace, size_t workspace_bytes, int impl,
                                      void* stream) {
  return score_topk_core(dense_operands(MFAR_E4M3, corpus, corpus_scales, q_vecs, q_scales), n_docs, corpus_fields,
                         field_begin, n_dense, dim, Q, w,
                         coo_input(coo_keys, coo_vals, coo_dtype, field_offsets_host, n_sparse), doc_id_base, k,
                         out_keys, out_scores, out_ids, workspace, workspace_bytes, impl, stream,
                         filter_input(filter_bits, filter_rows, filter_ld));
}

int mfar_score_topk_bm25_filtered(const void* corpus, int64_t n_docs, int corpus_fields, int field_begin,
                                  int n_dense, int dim, const void* q_vecs, int Q, const float* w,
                                  const void* const* indptr_host, const void* const* indices_host,
                                  const void* const* data_host, const int32_t* vocab_host, int n_sparse,
                                  const int32_t* entries, int64_t n_entries, int64_t doc_id_base,
                                  const uint32_t* filter_bits, int filter_rows, int64_t filter_ld, int k,
                                  uint64_t* out_keys, float* out_scores, int64_t* out_ids, void* workspace,
                                  size_t workspace_bytes, int impl, void* stream) {
  return score_topk_core(dense_operands(MFAR_BF16, corpus, nullptr, q_vecs, nullptr), n_docs, corpus_fields,
                         field_begin, n_dense, dim, Q, w,
                         bm25_input(indptr_host, indices_host, data_host, vocab_host, n_sparse, entries, n_entries),
                         doc_id_base, k, out_keys, out_scores, out_ids, workspace, workspace_bytes, impl, stream,
                         filter_input(filter_bits, filter_rows, filter_ld));
}

int mfar_score_topk_bm25_e4m3_filtered(const void* corpus, const float* corpus_scales, int64_t n_docs,
                                       int corpus_fields, int field_begin, int n_dense, int dim, const void* q_vecs,
                                       const float* q_scales, int Q, const float* w, const void* const* indptr_host,
                                       const void* const* indices_host, const void* const* data_host,
                                       const int32_t* vocab_host, int n_sparse, const int32_t* entries,
                                       int64_t n_entries, int64_t doc_id_base, const uint32_t* filter_bits,
                                       int filter_rows, int64_t filter_ld, int k, uint64_t* out_keys,
                                       float* out_scores, int64_t* out_ids, void* workspace, size_t workspace_bytes,
                                       int impl, void* stream) {
  return score_topk_core(dense_operands(MFAR_E4M3, corpus, corpus_scales, q_vecs, q_scales), n_docs, corpus_fields,
                         field_begin, n_dense, dim, Q, w,
                         bm25_input(indptr_host, indices_host, data_host, vocab_host, n_sparse, entries, n_entries),
                         doc_id_base, k, out_keys, out_scores, out_ids, workspace, workspace_bytes, impl, stream,
                         filter_input(filter_bits, filter_rows, filter_ld));
}

int mfar_topk_merge(const uint64_t* keys, int L, int Q, int k_in, int k, uint64_t* out_keys, float* out_scores,
                    int64_t* out_ids, void* stream) {
  if (!keys || L <= 0 || Q <= 0 || k_in <= 0) return MFAR_ERR_ARG;
  if (k <= 0 || k > MFAR_MAX_K) return MFAR_ERR_SHAPE;
  if (int rc = check_arch()) return rc;
  return launch_merge(keys, nullptr, nullptr, L, Q, k_in, Q, k, out_keys, out_scores, out_ids,
                      static_cast<cudaStream_t>(stream));
}

size_t mfar_exchange_buffer_bytes(int world, int q_cap, int k_cap) {
  if (world < 1 || world > 8 || q_cap <= 0 || k_cap <= 0) return 0;
  return align_up(size_t(MFAR_EXCHANGE_SLOTS) * world * q_cap * sizeof(int) +
                  size_t(MFAR_EXCHANGE_SLOTS) * world * q_cap * k_cap * sizeof(uint64_t) + 16, 256);
}

static int exchange_args_ok(int Q, int k_in, int k, int rank, int world, const uint64_t* peer_buffers_host) {
  if (!peer_buffers_host || Q <= 0 || k_in <= 0 || rank < 0 || rank >= world) return MFAR_ERR_ARG;
  if (k <= 0 || k > MFAR_MAX_K) return MFAR_ERR_SHAPE;
  for (int r = 0; r < world; ++r)
    if (!peer_buffers_host[r] || peer_buffers_host[r] % 16 != 0) return MFAR_ERR_ARG;
  return check_arch();
}

int mfar_topk_exchange_merge(const uint64_t* local_keys, int Q, int k_in, int k, int rank, int world,
                             const uint64_t* peer_buffers_host, int q_cap, int k_cap, int epoch, uint64_t* out_keys,
                             float* out_scores, int64_t* out_ids, void* stream) {
  if (!local_keys || epoch <= 0) return MFAR_ERR_ARG;
  if (int rc = exchange_args_ok(Q, k_in, k, rank, world, peer_buffers_host)) return rc;
  return launch_exchange_merge(local_keys, Q, k_in, k, rank, world,
                               reinterpret_cast<const unsigned long long*>(peer_buffers_host), q_cap, k_cap, epoch,
                               nullptr, 0, 0, out_keys, out_scores, out_ids, static_cast<cudaStream_t>(stream));
}

int mfar_topk_exchange_merge_dev_epoch(const uint64_t* local_keys, int Q, int k_in, int k, int rank, int world,
                                       const uint64_t* peer_buffers_host, int q_cap, int k_cap, int32_t* epoch_dev,
                                       uint64_t* out_keys, float* out_scores, int64_t* out_ids, void* stream) {
  if (!local_keys || !epoch_dev) return MFAR_ERR_ARG;
  if (int rc = exchange_args_ok(Q, k_in, k, rank, world, peer_buffers_host)) return rc;
  return launch_exchange_merge(local_keys, Q, k_in, k, rank, world,
                               reinterpret_cast<const unsigned long long*>(peer_buffers_host), q_cap, k_cap, 0,
                               epoch_dev, 0, 0, out_keys, out_scores, out_ids, static_cast<cudaStream_t>(stream));
}

int mfar_topk_exchange_push(const uint64_t* local_keys, int Q, int k_in, int rank, int world,
                            const uint64_t* peer_buffers_host, int q_cap, int k_cap, int32_t* epoch_dev, void* stream) {
  if (!local_keys || !epoch_dev) return MFAR_ERR_ARG;
  if (int rc = exchange_args_ok(Q, k_in, 1, rank, world, peer_buffers_host)) return rc;
  return launch_exchange_merge(local_keys, Q, k_in, 1, rank, world,
                               reinterpret_cast<const unsigned long long*>(peer_buffers_host), q_cap, k_cap, 0,
                               epoch_dev, 1, 0, nullptr, nullptr, nullptr, static_cast<cudaStream_t>(stream));
}

int mfar_topk_exchange_wait_merge(int Q, int k_in, int k, int rank, int world, const uint64_t* peer_buffers_host,
                                  int q_cap, int k_cap, const int32_t* epoch_dev, int lag, uint64_t* out_keys,
                                  float* out_scores, int64_t* out_ids, void* stream) {
  if (!epoch_dev || lag < 0 || lag > MFAR_EXCHANGE_SLOTS - 3) return MFAR_ERR_ARG;
  if (int rc = exchange_args_ok(Q, k_in, k, rank, world, peer_buffers_host)) return rc;
  return launch_exchange_merge(nullptr, Q, k_in, k, rank, world,
                               reinterpret_cast<const unsigned long long*>(peer_buffers_host), q_cap, k_cap, 0,
                               const_cast<int32_t*>(epoch_dev), 2, lag, out_keys, out_scores, out_ids,
                               static_cast<cudaStream_t>(stream));
}

int mfar_topk_apply_zero_init(float* scores, int64_t* ids, int Q, int k, void* stream) {
  if (!scores || !ids || Q <= 0 || k <= 0) return MFAR_ERR_ARG;
  if (int rc = check_arch()) return rc;
  return launch_zero_init(scores, ids, Q * k, static_cast<cudaStream_t>(stream));
}

int mfar_score_candidates(const void* corpus, int64_t n_docs, int corpus_fields, int field_begin, int n_fields,
                          int dim, const void* q_vecs, int Q, const int64_t* rows, int C, float* out, void* stream) {
  if (!corpus || !q_vecs || !rows || !out || Q <= 0 || C < 0 || n_docs <= 0) return MFAR_ERR_ARG;
  if (n_fields <= 0 || field_begin < 0 || field_begin + n_fields > corpus_fields || dim <= 0) return MFAR_ERR_SHAPE;
  if (int rc = check_arch()) return rc;
  return launch_score_candidates(corpus, nullptr, n_docs, corpus_fields, field_begin, n_fields, dim, q_vecs, nullptr, Q,
                                 rows, C, out, static_cast<cudaStream_t>(stream));
}

// mfar_score_candidates on an E4M3 corpus (index.py:227-232)
int mfar_score_candidates_e4m3(const void* corpus, const float* corpus_scales, int64_t n_docs, int corpus_fields,
                               int field_begin, int n_fields, int dim, const void* q_vecs, const float* q_scales, int Q,
                               const int64_t* rows, int C, float* out, void* stream) {
  if (!corpus || !corpus_scales || !q_vecs || !q_scales || !rows || !out || Q <= 0 || C < 0 || n_docs <= 0)
    return MFAR_ERR_ARG;
  if (n_fields <= 0 || field_begin < 0 || field_begin + n_fields > corpus_fields || dim <= 0) return MFAR_ERR_SHAPE;
  if (int rc = check_arch()) return rc;
  return launch_score_candidates(corpus, corpus_scales, n_docs, corpus_fields, field_begin, n_fields, dim, q_vecs,
                                 q_scales, Q, rows, C, out, static_cast<cudaStream_t>(stream));
}

int mfar_union_rescore(const void* corpus, int64_t n_docs, int corpus_fields, int n_dense, int dim, const void* q_vecs,
                       int Q, const float* w, const void* sparse, int n_sparse, int sparse_dtype, int64_t sparse_ld,
                       const int64_t* cand_rows, int n_lists, int k_in, int k, float* out_scores, int64_t* out_rows,
                       int32_t* out_union_size, void* stream) {
  t_last_launches = 0;
  if (!w || !cand_rows || !out_scores || !out_rows || !out_union_size || Q <= 0 || n_docs <= 0 || n_lists <= 0 ||
      k_in <= 0)
    return MFAR_ERR_ARG;
  if (n_dense < 0 || n_sparse < 0 || n_dense + n_sparse <= 0 || n_dense + n_sparse > MFAR_MAX_FIELDS) return MFAR_ERR_SHAPE;
  if (n_dense > 0 && (!corpus || !q_vecs || dim <= 0 || dim % 8 != 0 || n_dense > corpus_fields)) return MFAR_ERR_ARG;
  if (n_sparse > 0 && (!sparse || sparse_ld < n_docs || (sparse_dtype != MFAR_F16 && sparse_dtype != MFAR_F32)))
    return MFAR_ERR_ARG;
  if (k <= 0 || k > MFAR_MAX_K || int64_t(n_lists) * k_in > 8192 || n_docs > (int64_t(1) << 32) - 2) return MFAR_ERR_SHAPE;
  if (int rc = check_arch()) return rc;
  if (int rc = launch_union_rescore(corpus, n_docs, corpus_fields, n_dense, dim, q_vecs, Q, w, n_dense + n_sparse, sparse,
                                    sparse_dtype, sparse_ld, n_sparse, cand_rows, n_lists, k_in, k, out_scores, out_rows,
                                    out_union_size, static_cast<cudaStream_t>(stream)))
    return rc;
  t_last_launches = 1;
  return MFAR_OK;
}

// Scratch layout of the host-buffer calls: queries, query embedding, mixture weights, the sparse input (score rows
// re-pitched to sparse_ld, or BM25 token entries), result, workspace.  The BM25 layout keeps a query block without a
// dense field (its sizes are ABI).
struct HostScratch {
  size_t off_q, off_qe, off_w, off_sparse, off_scores, off_ids, off_ws, total, ws_bytes;
  int64_t sparse_ld;
};
static HostScratch host_scratch_layout(int Q, int dim, int E, int n_dense, int n_sparse, int64_t n_docs, int k,
                                       bool bm25, int sparse_dtype, int64_t n_entries) {
  HostScratch h{};
  size_t o = 0;
  h.off_q = o;      o += align_up(size_t(Q) * (bm25 ? std::max(dim, 1) : dim) * 2, 256);
  h.off_qe = o;     o += align_up(size_t(Q) * std::max(E, 1) * 4, 256);
  h.off_w = o;      o += align_up(size_t(Q) * (n_dense + n_sparse) * 4, 256);
  h.sparse_ld = int64_t(align_up(size_t(n_docs), 64));   // 128-/256-byte row pitch: the epilogue gather's vector loads
  h.off_sparse = o;
  if (bm25) o += align_up(size_t(std::max<int64_t>(n_entries, 1)) * 12, 256);
  else      o += align_up(size_t(Q) * n_sparse * size_t(h.sparse_ld) * (sparse_dtype == MFAR_F32 ? 4 : 2), 256);
  h.off_scores = o; o += align_up(size_t(Q) * k * 4, 256);
  h.off_ids = o;    o += align_up(size_t(Q) * k * 8, 256);
  h.off_ws = o;
  h.ws_bytes = bm25 ? mfar_score_topk_bm25_workspace_bytes(Q, k, n_docs, n_sparse, n_entries)
                    : mfar_score_topk_workspace_bytes(Q, k, n_docs, n_sparse);
  h.total = o + h.ws_bytes;
  return h;
}

size_t mfar_search_host_scratch_bytes(int Q, int dim, int E, int n_dense, int n_sparse, int64_t n_docs,
                                      int sparse_dtype, int k) {
  if (Q <= 0 || n_docs <= 0) return 0;
  return host_scratch_layout(Q, dim, E, n_dense, n_sparse, n_docs, k, false, sparse_dtype, 0).total;
}

size_t mfar_search_host_bm25_scratch_bytes(int Q, int dim, int E, int n_dense, int n_sparse, int64_t n_docs,
                                           int64_t n_entries, int k) {
  if (Q <= 0 || n_docs <= 0 || n_entries < 0) return 0;
  return host_scratch_layout(Q, dim, E, n_dense, n_sparse, n_docs, k, true, MFAR_F16, n_entries).total;
}

// The host-buffer calls: `sp` (HOST score rows of pitch n_docs, or token entries) is copied into the scratch buffer.
static int search_host_core(const void* corpus, int64_t n_docs, int corpus_fields, int field_begin, int n_dense,
                            int dim, const void* q_vecs_host, const float* q_emb_host, int Q, int E, const float* W,
                            const float* mask, int query_cond, SparseInput sp, int64_t doc_id_base, int k,
                            float* out_scores_host, int64_t* out_ids_host, void* scratch, size_t scratch_bytes,
                            int impl, void* stream) {
  const int n_sparse = sp.n_sparse;
  const bool bm25 = sp.kind == kSparseBm25;
  if (!scratch || !W || !out_scores_host || !out_ids_host || Q <= 0 || n_docs <= 0) return MFAR_ERR_ARG;
  if (n_dense > 0 && !q_vecs_host) return MFAR_ERR_ARG;
  if (query_cond && !q_emb_host) return MFAR_ERR_ARG;
  if (sp.kind == kSparseRows && !sp.dense) return MFAR_ERR_ARG;
  if (bm25 && (sp.n_entries < 0 || (sp.n_entries > 0 && !sp.entries))) return MFAR_ERR_ARG;
  if (reinterpret_cast<uintptr_t>(scratch) % 256 != 0) return MFAR_ERR_ARG;
  if (int rc = check_arch()) return rc;
  const auto h = host_scratch_layout(Q, dim, E, n_dense, n_sparse, n_docs, k, bm25, sp.dense_dtype, sp.n_entries);
  if (scratch_bytes < h.total) return MFAR_ERR_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  char* s = static_cast<char*>(scratch);
  if (n_dense > 0)
    MFAR_CUDA_OK(cudaMemcpyAsync(s + h.off_q, q_vecs_host, size_t(Q) * dim * 2, cudaMemcpyHostToDevice, st));
  if (query_cond)
    MFAR_CUDA_OK(cudaMemcpyAsync(s + h.off_qe, q_emb_host, size_t(Q) * E * 4, cudaMemcpyHostToDevice, st));
  if (sp.kind == kSparseRows) {   // [Q,Fs,N] host rows -> [Q,Fs,sparse_ld] device rows (aligned pitch)
    const size_t es = sp.dense_dtype == MFAR_F32 ? 4 : 2;
    const size_t width = size_t(n_docs) * es, dpitch = size_t(h.sparse_ld) * es;
    MFAR_CUDA_OK(cudaMemcpy2DAsync(s + h.off_sparse, dpitch, sp.dense, width, width, size_t(Q) * n_sparse,
                                   cudaMemcpyHostToDevice, st));
    if (dpitch > width)
      MFAR_CUDA_OK(cudaMemset2DAsync(s + h.off_sparse + width, dpitch, 0, dpitch - width, size_t(Q) * n_sparse, st));
    sp.dense = s + h.off_sparse;
    sp.dense_ld = h.sparse_ld;
  } else if (bm25) {
    if (sp.n_entries > 0)
      MFAR_CUDA_OK(cudaMemcpyAsync(s + h.off_sparse, sp.entries, sp.n_entries * 12, cudaMemcpyHostToDevice, st));
    sp.entries = reinterpret_cast<const int32_t*>(s + h.off_sparse);
  }
  float* w_dev = reinterpret_cast<float*>(s + h.off_w);
  // query_cond == 0: the shared weight row is replicated per query so the scoring kernels index w[q, f] uniformly
  if (int rc = launch_mixture_weights(query_cond ? reinterpret_cast<const float*>(s + h.off_qe) : nullptr, W, mask, Q,
                                      E, n_dense + n_sparse, query_cond, w_dev, st))
    return rc;
  float* sc = reinterpret_cast<float*>(s + h.off_scores);
  int64_t* ids = reinterpret_cast<int64_t*>(s + h.off_ids);
  int rc = score_topk_core(dense_operands(MFAR_BF16, corpus, nullptr, s + h.off_q, nullptr), n_docs, corpus_fields,
                           field_begin, n_dense, dim, Q, w_dev, sp, doc_id_base, k, nullptr, sc, ids,
                           s + h.off_ws, h.ws_bytes, impl, st);
  if (rc) return rc;
  t_last_launches += 1;
  MFAR_CUDA_OK(cudaMemcpyAsync(out_scores_host, sc, size_t(Q) * k * 4, cudaMemcpyDeviceToHost, st));
  MFAR_CUDA_OK(cudaMemcpyAsync(out_ids_host, ids, size_t(Q) * k * 8, cudaMemcpyDeviceToHost, st));
  MFAR_CUDA_OK(cudaStreamSynchronize(st));
  return MFAR_OK;
}

int mfar_search_host(const void* corpus, int64_t n_docs, int corpus_fields, int field_begin, int n_dense, int dim,
                     const void* q_vecs_host, const float* q_emb_host, int Q, int E, const float* W, const float* mask,
                     int query_cond, const void* sparse_host, int n_sparse, int sparse_dtype, int64_t doc_id_base,
                     int k, float* out_scores_host, int64_t* out_ids_host, void* scratch, size_t scratch_bytes,
                     int impl, void* stream) {
  return search_host_core(corpus, n_docs, corpus_fields, field_begin, n_dense, dim, q_vecs_host, q_emb_host, Q, E, W,
                          mask, query_cond, rows_input(sparse_host, n_sparse, sparse_dtype, n_docs), doc_id_base, k,
                          out_scores_host, out_ids_host, scratch, scratch_bytes, impl, stream);
}

int mfar_search_host_bm25(const void* corpus, int64_t n_docs, int corpus_fields, int field_begin, int n_dense, int dim,
                          const void* q_vecs_host, const float* q_emb_host, int Q, int E, const float* W,
                          const float* mask, int query_cond, const void* const* indptr_host,
                          const void* const* indices_host, const void* const* data_host, const int32_t* vocab_host,
                          int n_sparse, const int32_t* entries_host, int64_t n_entries, int64_t doc_id_base, int k,
                          float* out_scores_host, int64_t* out_ids_host, void* scratch, size_t scratch_bytes, int impl,
                          void* stream) {
  return search_host_core(corpus, n_docs, corpus_fields, field_begin, n_dense, dim, q_vecs_host, q_emb_host, Q, E, W,
                          mask, query_cond, bm25_input(indptr_host, indices_host, data_host, vocab_host, n_sparse,
                                                       entries_host, n_entries),
                          doc_id_base, k, out_scores_host, out_ids_host, scratch, scratch_bytes, impl, stream);
}

static int check_doc_layout(const float* q, int B, int E, const float* docs, int64_t N, int F, int64_t inner,
                            int64_t stride_p, int64_t stride_f, int64_t stride_s, float temperature) {
  if (!q || !docs || B <= 0 || N <= 0 || inner <= 0 || N % inner != 0 || !(temperature > 0.f)) return MFAR_ERR_ARG;
  if (F <= 0 || F > MFAR_MAX_FIELDS || E <= 0 || E % 4 != 0 || E > 1024) return MFAR_ERR_SHAPE;
  if (stride_p % 4 || stride_f % 4 || stride_s % 4 || reinterpret_cast<uintptr_t>(docs) % 16 ||
      reinterpret_cast<uintptr_t>(q) % 16)
    return MFAR_ERR_ARG;
  return MFAR_OK;
}

int mfar_field_components_fwd(const float* q, int B, int E, const float* docs, int64_t N, int F, int64_t inner,
                              int64_t stride_p, int64_t stride_f, int64_t stride_s, float temperature, float* comp,
                              void* stream) {
  if (int rc = check_doc_layout(q, B, E, docs, N, F, inner, stride_p, stride_f, stride_s, temperature)) return rc;
  if (!comp) return MFAR_ERR_ARG;
  if (int rc = check_arch()) return rc;
  const DocLayout L{inner, stride_p, stride_f, stride_s};
  return launch_field_components_fwd(q, B, E, docs, N, F, L, temperature, comp, static_cast<cudaStream_t>(stream));
}

int mfar_field_components_bwd(const float* q, int B, int E, const float* docs, int64_t N, int F, int64_t inner,
                              int64_t stride_p, int64_t stride_f, int64_t stride_s, float temperature,
                              const float* dcomp, float* dq, float* ddocs, void* stream) {
  if (int rc = check_doc_layout(q, B, E, docs, N, F, inner, stride_p, stride_f, stride_s, temperature)) return rc;
  if (!dcomp || (!dq && !ddocs)) return MFAR_ERR_ARG;
  if ((dq && reinterpret_cast<uintptr_t>(dq) % 16) || (ddocs && reinterpret_cast<uintptr_t>(ddocs) % 16))
    return MFAR_ERR_ARG;
  if (int rc = check_arch()) return rc;
  const DocLayout L{inner, stride_p, stride_f, stride_s};
  return launch_field_components_bwd(q, B, E, docs, N, F, L, temperature, dcomp, dq, ddocs,
                                     static_cast<cudaStream_t>(stream));
}

int mfar_mixture_bwd(const float* x, const float* q_emb, const float* W, const float* w, int w_rows, const float* g,
                     int B, int S, int E, int F, int query_cond, float* dx, float* dW, float* dq,
                     float* dlogit_scratch, void* stream) {
  if (!x || !W || !w || !g || !dW || !dlogit_scratch || B <= 0 || S < 0) return MFAR_ERR_ARG;
  if (query_cond && (!q_emb || E <= 0)) return MFAR_ERR_ARG;
  if (F <= 0 || F > MFAR_MAX_FIELDS || (w_rows != 1 && w_rows != B)) return MFAR_ERR_SHAPE;
  if (int rc = check_arch()) return rc;
  return launch_mixture_bwd(x, q_emb, W, w, w_rows, g, B, S, E, F, query_cond, dx, dW, query_cond ? dq : nullptr,
                            dlogit_scratch, static_cast<cudaStream_t>(stream));
}

int mfar_last_launch_count(void) { return t_last_launches; }

#ifdef MFAR_DEBUG_SEED
MFAR_API void mfar_debug_set_seed(const void* seed) { g_debug_seed = static_cast<const unsigned long long*>(seed); }
#endif

int mfar_profile_enable(int on) {
  if (on) {
    int dev = 0;
    MFAR_CUDA_OK(cudaGetDevice(&dev));
    if (g_prof_dev != dev) {                    // first use on this thread, or the thread moved to another device
      if (g_prof_dev >= 0)
        for (int i = 0; i < kProfRing; ++i)
          for (int j = 0; j < 2; ++j) cudaEventDestroy(g_prof_ev[i][j]);
      for (int i = 0; i < kProfRing; ++i)
        for (int j = 0; j < 2; ++j) MFAR_CUDA_OK(cudaEventCreate(&g_prof_ev[i][j]));
      g_prof_dev = dev;
    }
  }
  g_prof_on = on != 0;
  g_prof_n = 0;
  return MFAR_OK;
}

int mfar_profile_collect(float* out_ms_host, int max_n) {
  int n = g_prof_n < max_n ? g_prof_n : max_n;
  for (int i = 0; i < n; ++i) {
    if (cudaEventSynchronize(g_prof_ev[i][1]) != cudaSuccess) return -1;
    if (cudaEventElapsedTime(&out_ms_host[i], g_prof_ev[i][0], g_prof_ev[i][1]) != cudaSuccess) return -1;
  }
  g_prof_n = 0;
  return n;
}

long long mfar_profile_cluster4_ctas(void) { return qs_cluster4_ctas_collect(); }

}  // extern "C"
