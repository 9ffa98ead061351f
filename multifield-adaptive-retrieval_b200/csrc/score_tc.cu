// Fused multi-field scoring + streaming top-k on the 5th-gen tensor cores (sm_100a).
//
//   score[q, n] = sum_f w[q,f] * <q_vec[q], corpus[n, f, :]>  (+ base[q, n])  ->  per-CTA top-k
//
// Work decomposition
//   corpus tile  = 128 docs (UMMA M = 128, one TMEM lane per doc)
//   unit         = (tile, field): D_f[128 docs x QP queries] = A[128 x dim] . B[QP x dim]^T
//   A            = the (tile, field) block of the packed corpus, contiguous 128*dim bf16 in HBM,
//                  streamed by TMA in K-chunks of 64 (16 KB, SWIZZLE_128B) through a ring of stages
//   B            = the CTA's query tile (QP <= 64 rows), TMA-loaded ONCE and resident in shared
//                  memory for the whole kernel (QP*dim*2 B)
//   D            = fp32 accumulators in TMEM, double buffered (2 x QP columns)
//
// Warp roles (192 threads, 1 CTA / SM, persistent over tiles):
//   warp 0      TMA producer (one elected lane)
//   warp 1      TMEM allocator + tcgen05.mma issuer (one elected lane)
//   warps 2..5  epilogue: tcgen05.ld the finished D_f, acc[q] += w[q,f] * D_f[doc,q] in registers
//               (fp32 weights applied AFTER the fp32 accumulation - never folded into bf16 operands),
//               and after the last field: + pre-mixed sparse term, threshold filter, candidate push,
//               warp-level list compaction.  No [Q x N x F] (or [Q x N]) score tensor is ever written.
//
// grid = (workers, q_tiles): CTAs with the same blockIdx.x walk the same tile sequence for different
// query tiles, so a corpus tile is fetched from HBM once and re-read from L2 by the other q-tiles.
#include <cuda.h>

#include "common.cuh"
#include "kernels.h"
#include "tc_ptx.cuh"

namespace mfar {

constexpr int kTcThreads = 192;
constexpr int kABytes = kTileDocs * kChunkK * 2;  // 16 KB per stage

struct TcParams {
  int64_t n_docs;
  int n_tiles, corpus_fields, field_begin, n_dense, k_chunks;
  int Q;
  const float* w;
  int w_ld;
  const float* base;
  int64_t base_ld;
  const void* sparse;   // [Q, n_sparse, sparse_ld] f16/f32 gathered by the epilogue (exclusive with base), rows 32-B aligned
  int64_t sparse_ld;
  int64_t sparse_cols;  // columns addressable from `sparse` (<= sparse_ld)
  int n_sparse;
  int sparse_f16;
  const float* corpus_scales;   // E4M3 corpus: [tiles][corpus_fields][128] row scales
  const float* q_scales;        // E4M3 queries: [Q]
  int64_t doc_id_base;
  int k;
  int stages;
  TopkWorkspace ws;
  DocFilter filt;               // FILT only
};

// Sparse term of one corpus tile for the CTA's QP queries, gathered from the per-field score rows (index.py:111-118)
// and mixed (weighting.py:29) into a shared-memory block base_s[QP][128 docs] fp32 that seeds the accumulators:
//   base_s[c][n] = sum_j w[q0 + c, n_dense + j] * sparse[q0 + c, j, tile*128 + n]     (j ascending, fmaf)
// An epilogue THREAD of this kernel owns a doc (TMEM lane), but the score rows run along docs per (query, field) - so
// the gather has its own mapping and its own two STAGER WARPS (6, 7): a thread takes (query c, 32-byte group g)
// pairs, 8 lanes cover one query's 128 docs (256 contiguous bytes of f16), a warp four queries; loads of field j+1 are
// in flight while field j is mixed.  The stagers run one tile ahead of the epilogue (base_full / base_empty
// mbarriers; the epilogue copies base_s into its accumulators at tile start and hands the block back), so the DRAM
// latency of the gather never sits in front of an accumulator drain (done by the epilogue warps themselves it cost
// 17 % at Amazon-shaped Q=64).  The [Q, N] pre-mix block of round 1 (written to and re-read from HBM) is gone.
constexpr int kStagerThreads = 64;
constexpr int kStagerWarp0 = 6;
template <int QP, bool F16>
__device__ __forceinline__ void tc_stage_sparse(float* base_s, const TcParams& p, int q0, int nq, int64_t tile_doc0,
                                                const float* w_sp, int et) {   // et: 0 .. kStagerThreads-1
  constexpr int kEs = F16 ? 2 : 4;
  constexpr int kLoadDocs = 32 / kEs;               // 16 / 8 docs per 32-byte load
  constexpr int kGroups = kTileDocs / kLoadDocs;    // 8 / 16 groups per query row
  constexpr int kPairs = QP * kGroups / kStagerThreads;   // (query, group) pairs per thread: QP/8 (f16), QP/4 (f32)
  static_assert(kPairs >= 1, "tile too small");
  constexpr int kBatch = kPairs < 4 ? kPairs : 4;   // pairs processed together (loads in flight: 2 * kBatch)
  const int64_t row_bytes = p.sparse_ld * kEs;
  for (int b0 = 0; b0 < kPairs; b0 += kBatch) {
    const char* src[kBatch];
    bool live[kBatch];
    int cq[kBatch], gq[kBatch];
#pragma unroll
    for (int i = 0; i < kBatch; ++i) {
      const int pid = (b0 + i) * kStagerThreads + et;
      cq[i] = pid / kGroups; gq[i] = pid % kGroups;
      const int64_t d = tile_doc0 + gq[i] * kLoadDocs;
      live[i] = cq[i] < nq && d < p.sparse_cols;
      src[i] = static_cast<const char*>(p.sparse) + (int64_t(q0 + cq[i]) * p.n_sparse * p.sparse_ld + d) * kEs;
    }
    float acc[kBatch][kLoadDocs];
#pragma unroll
    for (int i = 0; i < kBatch; ++i)
#pragma unroll
      for (int e = 0; e < kLoadDocs; ++e) acc[i][e] = 0.f;
    uint32_t cur[kBatch][8], nxt[kBatch][8];
    auto load = [&](uint32_t (&b)[kBatch][8], int j) {
#pragma unroll
      for (int i = 0; i < kBatch; ++i) {
        if (live[i]) {
          ldg256_stream(src[i] + int64_t(j) * row_bytes, b[i]);
        } else {
#pragma unroll
          for (int e = 0; e < 8; ++e) b[i][e] = 0u;
        }
      }
    };
    load(cur, 0);
#pragma unroll 2
    for (int j = 0; j < p.n_sparse; ++j) {
      if (j + 1 < p.n_sparse) load(nxt, j + 1);
#pragma unroll
      for (int i = 0; i < kBatch; ++i) {
        const float wj = w_sp[j * QP + cq[i]];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          if (F16) {
            const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&cur[i][e]));
            acc[i][2 * e] = fmaf(wj, f.x, acc[i][2 * e]);
            acc[i][2 * e + 1] = fmaf(wj, f.y, acc[i][2 * e + 1]);
          } else {
            acc[i][e] = fmaf(wj, __uint_as_float(cur[i][e]), acc[i][e]);
          }
        }
      }
#pragma unroll
      for (int i = 0; i < kBatch; ++i)
#pragma unroll
        for (int e = 0; e < 8; ++e) cur[i][e] = nxt[i][e];
    }
#pragma unroll
    for (int i = 0; i < kBatch; ++i) {
      float4* dst = reinterpret_cast<float4*>(base_s + cq[i] * kTileDocs + gq[i] * kLoadDocs);
#pragma unroll
      for (int e = 0; e < kLoadDocs; e += 4) dst[e / 4] = make_float4(acc[i][e], acc[i][e + 1], acc[i][e + 2], acc[i][e + 3]);
    }
  }
}


// ------------------------------------------------------------------------------------ the kernel
// QP: query columns per CTA (UMMA N), one of 16 / 32 / 64.
// E8: E4M3 corpus and queries.  A K-chunk is still one 128-byte swizzled row span (128 elements instead of 64), so the
// ring, the descriptors and the producer are those of bf16; the MMA is kind::f8f6f4 (K = 32), and the epilogue applies
// the query scale (shared memory) and the doc's row scale (one coalesced 512-byte load per (tile, field)) to D_f.
// FILT: doc filter.  A thread owns a doc and tests QP queries' bits for it, so the tile's words of every query are
// staged in shared memory (s_filt, one tile ahead) and a pushed pair reads one of them next to the key compare.
template <int QP, bool SP, bool E8, bool FILT>   // SP: sparse fields gathered in-kernel (tc_stage_sparse, 2 more warps)
__global__ void __launch_bounds__(SP ? kTcThreads + kStagerThreads : kTcThreads, 1)
score_tc_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, TcParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // carve: [A stages][B resident][w_s][s_q (E8)][thr as float][thr][cnt][flags][base_s (SP)][s_filt (FILT)][barriers]
  // [tmem ptr]
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem_a + size_t(p.stages) * kABytes;
  constexpr int kChunkElems = E8 ? kChunkK8 : kChunkK;
  const int b_chunk_bytes = QP * 128;              // QP rows of one 128-byte K-chunk
  const int n_w = p.n_dense + (SP ? p.n_sparse : 0);   // weight rows kept in shared memory
  float* w_s = reinterpret_cast<float*>(smem_b + size_t(p.k_chunks) * b_chunk_bytes);     // [n_w][QP]
  float* sq_s = w_s + size_t(n_w) * QP;            // [QP] query scales (E8)
  float* s_thrf = sq_s + (E8 ? QP : 0);            // [QP] score of s_thr (float pre-filter), +inf for padding queries
  unsigned long long* s_thr = reinterpret_cast<unsigned long long*>(s_thrf + QP);
  int* s_cnt = reinterpret_cast<int*>(s_thr + QP);
  int* s_flags = s_cnt + QP;                       // reserved (keeps the shared-memory layout)
  float* base_s = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(s_flags + QP) + 15) & ~uintptr_t(15));   // [QP][128]
  constexpr int kFiltWords = QP * (kTileDocs / 32);   // one tile's filter words: [QP queries][4 x 32 docs]
  uint32_t* s_filt = reinterpret_cast<uint32_t*>(base_s + (SP ? QP * kTileDocs : 0));   // [2][kFiltWords]
  uint64_t* bars = reinterpret_cast<uint64_t*>(
      (reinterpret_cast<uintptr_t>(s_filt + (FILT ? 2 * kFiltWords : 0)) + 7) & ~uintptr_t(7));
  uint64_t* full_bar = bars;                       // [stages]
  uint64_t* empty_bar = bars + p.stages;           // [stages]
  uint64_t* tfull_bar = bars + 2 * p.stages;       // [2]
  uint64_t* tempty_bar = tfull_bar + 2;            // [2]
  uint64_t* bq_bar = tempty_bar + 2;               // [1]
  uint64_t* base_full = bq_bar + 1;                // [1]  stagers -> epilogue: base_s holds the next tile's sparse term
  uint64_t* base_empty = base_full + 1;            // [1]  epilogue -> stagers: base_s has been copied out
  uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(base_empty + 1);

  const int warp = __shfl_sync(0xffffffffu, int(threadIdx.x >> 5), 0);   // warp-uniform for the compiler too
  const int lane = threadIdx.x & 31;
  const int g = blockIdx.x;                        // worker (walks tiles g, g+G, ...)
  const int q0 = blockIdx.y * QP;                  // first query of this CTA's tile
  const int nq = min(QP, p.Q - q0);
  int* err = p.ws.err;
  constexpr uint32_t kTmemCols = (2 * QP < 32) ? 32 : 2 * QP;

  // ---- one-time setup
  for (int i = threadIdx.x; i < n_w * QP; i += int(blockDim.x)) {
    const int f = i / QP, c = i % QP;
    w_s[i] = (c < nq) ? p.w[int64_t(q0 + c) * p.w_ld + f] : 0.f;
  }
  if (E8 && threadIdx.x < QP) sq_s[threadIdx.x] = int(threadIdx.x) < nq ? p.q_scales[q0 + threadIdx.x] : 1.f;
  if (threadIdx.x < QP) {
    s_thr[threadIdx.x] = 0ull; s_cnt[threadIdx.x] = 0; s_flags[threadIdx.x] = 0;
    s_thrf[threadIdx.x] = int(threadIdx.x) < nq ? -INFINITY : INFINITY;
  }
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a);
    tma_prefetch_desc(&map_b);
    for (int s = 0; s < p.stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&tfull_bar[b], 1); mbar_init(&tempty_bar[b], kEpiThreads); }
    mbar_init(bq_bar, 1);
    mbar_init(base_full, kStagerThreads);
    mbar_init(base_empty, kEpiThreads);
    fence_barrier_init();
  }
  if (warp == 1) { tmem_alloc(tmem_ptr_s, kTmemCols); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_s;

  const int my_tiles = (p.n_tiles > g) ? (p.n_tiles - g + gridDim.x - 1) / gridDim.x : 0;
  const int units = my_tiles * p.n_dense;

  if (warp == 0) {
    // ===================================================================== TMA producer
    if (units > 0) {                                // whole warp walks the loop, one elected lane issues
      if (elect_one()) {
        mbar_expect_tx(bq_bar, uint32_t(p.k_chunks) * b_chunk_bytes);
        for (int kc = 0; kc < p.k_chunks; ++kc)
          tma_load_2d(&map_b, bq_bar, smem_b + size_t(kc) * b_chunk_bytes, kc * kChunkElems, q0);
      }
      __syncwarp();
      int stage = 0; uint32_t phase = 0;
      for (int i = 0; i < my_tiles; ++i) {
        const int t = g + i * gridDim.x;
        for (int f = 0; f < p.n_dense; ++f) {
          const int row0 = (t * p.corpus_fields + p.field_begin + f) * kTileDocs;
          for (int kc = 0; kc < p.k_chunks; ++kc) {
            mbar_wait(&empty_bar[stage], phase ^ 1, err, 1);
            if (elect_one()) {
              mbar_expect_tx(&full_bar[stage], kABytes);
              tma_load_2d(&map_a, &full_bar[stage], smem_a + size_t(stage) * kABytes, kc * kChunkElems, row0);
            }
            __syncwarp();
            if (++stage == p.stages) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================================================================== MMA issuer
    if (units > 0) {                                // whole warp walks the loop, one elected lane issues
      constexpr uint32_t idesc = E8 ? make_idesc_e4m3(kTileDocs, QP) : make_idesc(kTileDocs, QP);
      const uint32_t issue = elect_one() ? 1u : 0u;
      mbar_wait(bq_bar, 0, err, 2);
      tc_fence_after();
      int stage = 0; uint32_t phase = 0;
      for (int u = 0; u < units; ++u) {
        const int buf = u & 1;
        mbar_wait(&tempty_bar[buf], ((u >> 1) & 1) ^ 1, err, 3);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + uint32_t(buf * QP);
        for (int kc = 0; kc < p.k_chunks; ++kc) {
          mbar_wait(&full_bar[stage], phase, err, 4);
          tc_fence_after();
          const uint64_t a_desc = make_sw128_desc(smem_u32(smem_a + size_t(stage) * kABytes));
          const uint64_t b_desc = make_sw128_desc(smem_u32(smem_b + size_t(kc) * b_chunk_bytes));
#pragma unroll
          for (int kk = 0; kk < kChunkK / kUmmaK; ++kk) {
            // advance 32 B (16 bf16 / 32 E4M3 elements) along K inside the 128 B swizzle span: +2 in the >>4 address field
            if (E8) umma_e4m3_pred(d_tmem, a_desc + uint64_t(kk * 2), b_desc + uint64_t(kk * 2), idesc, (kc | kk) != 0, issue);
            else umma_bf16_pred(d_tmem, a_desc + uint64_t(kk * 2), b_desc + uint64_t(kk * 2), idesc, (kc | kk) != 0, issue);
          }
          __syncwarp();
          if (elect_one()) tc_commit(&empty_bar[stage]);   // smem stage reusable once these MMAs retire
          if (++stage == p.stages) { stage = 0; phase ^= 1; }
        }
        if (elect_one()) tc_commit(&tfull_bar[buf]);       // accumulator of this unit complete
        __syncwarp();
      }
    }
  } else if (SP && warp >= kStagerWarp0) {
    // ===================================================================== sparse stagers (warps 6, 7)
    const int st = int(threadIdx.x) - kStagerWarp0 * 32;
    for (int i = 0; i < my_tiles; ++i) {
      const int64_t tile_doc0 = int64_t(g + i * int(gridDim.x)) * kTileDocs;
      mbar_wait(base_empty, (i & 1) ^ 1, err, 6);
      if (p.sparse_f16) tc_stage_sparse<QP, true>(base_s, p, q0, nq, tile_doc0, w_s + p.n_dense * QP, st);
      else tc_stage_sparse<QP, false>(base_s, p, q0, nq, tile_doc0, w_s + p.n_dense * QP, st);
      mbar_arrive(base_full);                        // release: this thread's base_s stores
    }
  } else {
    // ===================================================================== epilogue (warps 2..5)
    const int lane_grp = warp & 3;                 // TMEM lanes 32*lane_grp .. +31 are this warp's
    const int doc_in_tile = lane_grp * 32 + lane;
    const int epi_warp = warp - 2;
    float acc[QP];
    int u = 0;
    // Query c's list, thresholds and counter are looked after by warp c % 4, one query per LANE: cq = this lane's query.
    const int cq = epi_warp + (kEpiThreads / 32) * lane;
    const bool cq_live = lane < QP / (kEpiThreads / 32) && cq < nq;
    if (cq_live) {                                   // the seed (capi.cu, threshold seeding), if any
      const unsigned long long gt = ld_relaxed_u64(p.ws.gthr + q0 + cq);
      if (gt > s_thr[cq]) { s_thr[cq] = gt; s_thrf[cq] = key_score(gt); }
    }
    // FILT: s_filt[b][c * 4 + w] = bits of docs 32w .. 32w + 31 of a tile for query c (0 for padding queries).  Tile
    // i + 1's words are loaded at the head of tile i and stored after its last accumulator drain into buffer (i + 1) & 1;
    // tile i's push reads buffer i & 1.  The block barriers that end tile i order those stores before tile i + 1's
    // reads, and tile i - 1's reads of the same buffer before them.
    constexpr int kFiltPer = (kFiltWords + kEpiThreads - 1) / kEpiThreads;
    const int fe0 = int(threadIdx.x) - 64;           // epilogue thread index 0 .. 127
    uint32_t fnext[kFiltPer];
    auto filt_load = [&](int tile) {
#pragma unroll
      for (int j = 0; j < kFiltPer; ++j) {
        const int e = fe0 + j * kEpiThreads, c = e >> 2;
        fnext[j] = (e < kFiltWords && c < nq)
                       ? filter_bits32(p.filt.bits + int64_t(q0 + c) * p.filt.stride, p.filt.words,
                                       p.doc_id_base + int64_t(tile) * kTileDocs + (e & 3) * 32)
                       : 0u;
      }
    };
    auto filt_store = [&](int b) {
#pragma unroll
      for (int j = 0; j < kFiltPer; ++j)
        if (fe0 + j * kEpiThreads < kFiltWords) s_filt[b * kFiltWords + fe0 + j * kEpiThreads] = fnext[j];
    };
    if (FILT && my_tiles > 0) { filt_load(g); filt_store(0); }
    epi_bar_sync();
    for (int i = 0; i < my_tiles; ++i) {
      const int t = g + i * gridDim.x;
      // the best threshold any CTA found for this lane's query (incl. the pooled bound, common.cuh): the load is issued
      // here and consumed after the tile's pushes, so its L2 round trip hides behind the accumulation (it used to sit,
      // with a block barrier, at the head of every tile - ~10 % of a single-field tile)
      unsigned long long gt_next = 0ull;
      if (cq_live) gt_next = ld_relaxed_u64(p.ws.gthr + q0 + cq);
      // Long tiles / few tiles per CTA (PRIME-shaped: 7 tiles of 22 fields): one tile of staleness costs a whole extra
      // round of compactions, so the value is applied BEFORE this tile's pushes (one more block barrier, nothing next
      // to a 100 us tile); short tiles apply it after the pushes, for the next tile.
      const bool adopt_before_push = p.n_dense >= 8 || my_tiles <= 32;
      if (FILT && i + 1 < my_tiles) filt_load(t + int(gridDim.x));   // consumed after the field loop
      // The accumulators start from the pre-mixed sparse term: its QP loads per doc (coalesced across the warp's
      // 32 docs) are issued here, ahead of the wait for the tile's first accumulator, instead of serialising with
      // the push loop after the last field.
      const int64_t doc_local = int64_t(t) * kTileDocs + doc_in_tile;
      if (SP) {
        mbar_wait(base_full, i & 1, err, 7);
#pragma unroll
        for (int c = 0; c < QP; ++c) acc[c] = base_s[c * kTileDocs + doc_in_tile];
        mbar_arrive(base_empty);                     // the stagers may fill base_s for the next tile
      } else if (p.base != nullptr && doc_local < p.n_docs) {
        const float* bp = p.base + int64_t(q0) * p.base_ld + doc_local;
#pragma unroll
        for (int c = 0; c < QP; ++c) acc[c] = (c < nq) ? __ldg(bp + int64_t(c) * p.base_ld) : 0.f;
      } else {
#pragma unroll
        for (int c = 0; c < QP; ++c) acc[c] = 0.f;
      }
      for (int f = 0; f < p.n_dense; ++f, ++u) {
        const int buf = u & 1;
        // the doc's row scale: 128 consecutive floats per (tile, field), loaded ahead of the wait for the accumulator
        const float sd = E8 ? __ldg(p.corpus_scales + (int64_t(t) * p.corpus_fields + p.field_begin + f) * kTileDocs +
                                    doc_in_tile)
                            : 1.f;
        mbar_wait(&tfull_bar[buf], (u >> 1) & 1, err, 5);
        tc_fence_after();
        const uint32_t taddr = tmem_base + (uint32_t(lane_grp * 32) << 16) + uint32_t(buf * QP);
        const float* wf = w_s + f * QP;
#pragma unroll
        for (int c0 = 0; c0 < QP; c0 += 16) {
          uint32_t v[16];
          tmem_ld16(taddr + c0, v);
          tmem_ld_wait();
#pragma unroll
          for (int c = 0; c < 16; c += 4) {
            const float4 w4 = *reinterpret_cast<const float4*>(wf + c0 + c);
            if (E8) {                                // w * ((D * s_q) * s_d): two roundings, never s_q * s_d first
#pragma unroll
              for (int j = 0; j < 4; ++j) v[c + j] = __float_as_uint((__uint_as_float(v[c + j]) * sq_s[c0 + c + j]) * sd);
            }
            acc[c0 + c + 0] = fmaf(w4.x, __uint_as_float(v[c + 0]), acc[c0 + c + 0]);
            acc[c0 + c + 1] = fmaf(w4.y, __uint_as_float(v[c + 1]), acc[c0 + c + 1]);
            acc[c0 + c + 2] = fmaf(w4.z, __uint_as_float(v[c + 2]), acc[c0 + c + 2]);
            acc[c0 + c + 3] = fmaf(w4.w, __uint_as_float(v[c + 3]), acc[c0 + c + 3]);
          }
        }
        tc_fence_before();
        mbar_arrive(&tempty_bar[buf]);             // 128 arrivals free the accumulator buffer
      }
      // ---- tile done: filter, push
      if (FILT && i + 1 < my_tiles) filt_store((i + 1) & 1);
      if (adopt_before_push) {
        if (cq_live && gt_next > s_thr[cq]) { s_thr[cq] = gt_next; s_thrf[cq] = key_score(gt_next); }
        epi_bar_sync();
      }
      if (doc_local < p.n_docs) {
        const uint32_t doc_id = uint32_t(p.doc_id_base + doc_local);
        const uint32_t* fw = s_filt + (i & 1) * kFiltWords + lane_grp;   // FILT: word c * 4 holds this warp's 32 docs
        // Float pre-filter per GROUP of 8 queries: max_j(score[c0+j] - score of query c0+j's threshold) >= 0 decides
        // with 8 FADD + 3 FMNMX3/FMNMX + 1 FSETP + 1 branch whether any of the 8 (doc, query) pairs can be admitted;
        // the exact (score, id) key is only built inside live groups.  With one epilogue warp per scheduler every
        // branch is a pipeline bubble: the former per-pair key compare (LDS + 2 ISETP + branch, x QP) made a single_
        // scorer at Q=64 epilogue-bound (ncu: 0.56 of HBM peak, tensor pipe 10 % active).
#pragma unroll
        for (int c0 = 0; c0 < QP; c0 += 8) {
          const float4 ta = *reinterpret_cast<const float4*>(s_thrf + c0);
          const float4 tb = *reinterpret_cast<const float4*>(s_thrf + c0 + 4);
          // NaN-propagating max and !(m < 0): a NaN score, or inf - inf of a score and threshold in the same infinite
          // class, reaches the key compare (fmaxf would drop it, and the answer would depend on the group's mates)
          const float m = fmax_nan(fmax_nan(fmax_nan(acc[c0] - ta.x, acc[c0 + 1] - ta.y), fmax_nan(acc[c0 + 2] - ta.z, acc[c0 + 3] - ta.w)),
                                   fmax_nan(fmax_nan(acc[c0 + 4] - tb.x, acc[c0 + 5] - tb.y), fmax_nan(acc[c0 + 6] - tb.z, acc[c0 + 7] - tb.w)));
          if (!(m < 0.f)) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const int c = c0 + j;
              const uint64_t key = make_key(acc[c], doc_id);
              if (key > s_thr[c] && c < nq && (!FILT || ((fw[c * 4] >> lane) & 1u))) {
                const int pos = atomicAdd(&s_cnt[c], 1);
                __stcg(p.ws.cand_keys + (int64_t(g) * p.ws.q_pad + q0 + c) * kCandCap + pos, key);
              }
            }
          }
        }
      }
      epi_bar_sync();
      // lists that could overflow during the next tile, found lane-parallel (a serial walk over the warp's 16 queries
      // with a shared-memory load and a branch each was ~20 % of a single-field tile's epilogue)
      unsigned need = __ballot_sync(0xffffffffu, cq_live && s_cnt[cq] > kCandCap - kTileDocs);
      if (!adopt_before_push && cq_live && gt_next > s_thr[cq]) { s_thr[cq] = gt_next; s_thrf[cq] = key_score(gt_next); }
      __syncwarp();
      while (need) {
        const int c = epi_warp + (kEpiThreads / 32) * (__ffs(need) - 1);
        need &= need - 1u;
        const int cnt = s_cnt[c];
        uint64_t* list = p.ws.cand_keys + (int64_t(g) * p.ws.q_pad + q0 + c) * kCandCap;
        int cnt_new = p.k;                             // every round: warp select (see score_qs.cu)
        const int r = pooled_rank(p.k, int(gridDim.x));
        uint64_t bound_r = 0ull;
        const uint64_t kth = warp_select_list(list, cnt, p.k, kCandCap - kTileDocs, lane, &cnt_new, r, &bound_r);
        __syncwarp();
        const unsigned long long pooled = pool_publish_and_min(p.ws.pool, int(gridDim.x), p.ws.q_pad, g, q0 + c,
                                                               bound_r, lane);
        if (lane == 0) {
          if (kth > s_thr[c]) s_thr[c] = kth;
          if (pooled > s_thr[c]) s_thr[c] = pooled;
          s_thrf[c] = key_score(s_thr[c]);
          s_cnt[c] = cnt_new;
          atomicMax(p.ws.gthr + q0 + c, s_thr[c]);
        }
      }
      epi_bar_sync();
    }
    const int et = threadIdx.x - 64;
    if (et < nq) {
      p.ws.cand_cnt[int64_t(g) * p.ws.q_pad + q0 + et] = s_cnt[et];
      p.ws.cand_thr[int64_t(g) * p.ws.q_pad + q0 + et] = s_thr[et];
    }
  }

  // ---- teardown
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 1) tmem_dealloc(tmem_base, kTmemCols);
}

// ------------------------------------------------------------------------------------ host side
bool score_tc_supported(const ScoreArgs& a) {
  const int chunk = a.corpus_dtype == MFAR_E4M3 ? kChunkK8 : kChunkK;
  return a.n_dense >= 1 && a.dim % chunk == 0 && a.dim >= chunk && a.dim <= 1024 &&
         (reinterpret_cast<uintptr_t>(a.corpus) % 16 == 0) && (reinterpret_cast<uintptr_t>(a.q_vecs) % 16 == 0) &&
         int64_t(a.n_tiles) * a.corpus_fields * kTileDocs < (int64_t(1) << 31);
}

PassPlan plan_score_tc(int Q, int n_tiles) {
  PassPlan p{};
  p.impl = MFAR_IMPL_TCGEN05;
  p.q_pad = Q <= 16 ? 16 : (Q <= 32 ? 32 : 64);
  p.q_tiles = (Q + p.q_pad - 1) / p.q_pad;
  p.q_pad_total = p.q_pad * p.q_tiles;
  int w = kNumSmsB200 / p.q_tiles;
  if (w < 1) w = 1;
  if (w > n_tiles) w = n_tiles;
  if (w < 1) w = 1;
  p.workers = p.lists = w;
  p.cg = 1;
  return p;
}

// n_weights: rows of [QP] floats next to the weights (E8: + the query scales); filt: two tiles of filter words
static size_t tc_smem_bytes(int qp, int n_weights, bool sparse, int k_chunks, int stages, bool filt) {
  return 1024 + size_t(stages) * kABytes + size_t(k_chunks) * qp * 128 + size_t(n_weights) * qp * 4 +
         size_t(qp) * 20 + 16 + (sparse ? size_t(qp) * kTileDocs * 4 : 0) + (filt ? size_t(qp) * kTileDocs / 4 : 0) + 8 +
         (2 * stages + 7) * 8 + 16;
}

template <int QP, bool SP, bool E8, bool FILT>
static int launch_tc_impl(const ScoreArgs& a, const PassPlan& plan, const TopkWorkspace& ws, cudaStream_t st) {
  TcParams p;
  p.n_docs = a.n_docs; p.n_tiles = a.n_tiles; p.corpus_fields = a.corpus_fields; p.field_begin = a.field_begin;
  p.n_dense = a.n_dense; p.k_chunks = a.dim / (E8 ? kChunkK8 : kChunkK);
  p.corpus_scales = a.corpus_scales; p.q_scales = a.q_scales; p.Q = a.Q; p.w = a.w; p.w_ld = a.w_ld; p.base = a.base;
  p.base_ld = a.base_ld; p.doc_id_base = a.doc_id_base; p.k = a.k;
  p.sparse = a.sparse; p.sparse_ld = a.sparse_ld; p.n_sparse = a.sparse ? a.n_sparse : 0;
  p.sparse_cols = a.sparse_cols ? a.sparse_cols : a.sparse_ld;
  p.sparse_f16 = a.sparse_dtype == MFAR_F16;
  const int n_w = a.n_dense + p.n_sparse + (E8 ? 1 : 0);
  p.ws = ws;
  p.filt = DocFilter{a.filter_bits, a.filter_stride, a.filter_words};
  int stages = 8;
  const size_t smem_cap = 227 * 1024;
  while (stages > 2 && tc_smem_bytes(QP, n_w, a.sparse != nullptr, p.k_chunks, stages, FILT) > smem_cap) --stages;
  if (tc_smem_bytes(QP, n_w, a.sparse != nullptr, p.k_chunks, stages, FILT) > smem_cap) return MFAR_ERR_SHAPE;
  p.stages = stages;
  const size_t smem = tc_smem_bytes(QP, n_w, a.sparse != nullptr, p.k_chunks, stages, FILT);

  CUtensorMap map_a, map_b;
  int rc = make_tensor_map_2d(&map_a, a.corpus, uint64_t(a.n_tiles) * a.corpus_fields * kTileDocs, a.dim, kTileDocs,
                       CU_TENSOR_MAP_L2_PROMOTION_L2_256B, E8);
  if (rc) return rc;
  rc = make_tensor_map_2d(&map_b, a.q_vecs, uint64_t(a.Q), a.dim, QP, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, E8);
  if (rc) return rc;

  static PerDeviceOnce attr_once;   // per template instantiation
  MFAR_CUDA_OK(attr_once.run([&] {
    return cudaFuncSetAttribute(score_tc_kernel<QP, SP, E8, FILT>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem_cap));
  }));
  dim3 grid(plan.workers, plan.q_tiles);
  score_tc_kernel<QP, SP, E8, FILT><<<grid, SP ? kTcThreads + kStagerThreads : kTcThreads, smem, st>>>(map_a, map_b, p);
  MFAR_CUDA_OK(cudaGetLastError());
  return MFAR_OK;
}

template <bool E8, bool FILT>
static int launch_tc_qp(const ScoreArgs& a, const PassPlan& plan, const TopkWorkspace& ws, cudaStream_t st) {
  switch (plan.q_pad) {
    case 16: return a.sparse ? launch_tc_impl<16, true, E8, FILT>(a, plan, ws, st)
                             : launch_tc_impl<16, false, E8, FILT>(a, plan, ws, st);
    case 32: return a.sparse ? launch_tc_impl<32, true, E8, FILT>(a, plan, ws, st)
                             : launch_tc_impl<32, false, E8, FILT>(a, plan, ws, st);
    case 64: return a.sparse ? launch_tc_impl<64, true, E8, FILT>(a, plan, ws, st)
                             : launch_tc_impl<64, false, E8, FILT>(a, plan, ws, st);
    default: return MFAR_ERR_SHAPE;
  }
}

int launch_score_tc(const ScoreArgs& a, const PassPlan& plan, const TopkWorkspace& ws, cudaStream_t st,
                    int* launches) {
  int rc;
  if (a.corpus_dtype == MFAR_E4M3)
    rc = a.filter_bits ? launch_tc_qp<true, true>(a, plan, ws, st) : launch_tc_qp<true, false>(a, plan, ws, st);
  else
    rc = a.filter_bits ? launch_tc_qp<false, true>(a, plan, ws, st) : launch_tc_qp<false, false>(a, plan, ws, st);
  if (rc == MFAR_OK) ++*launches;
  return rc;
}

}  // namespace mfar
