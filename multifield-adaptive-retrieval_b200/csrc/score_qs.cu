// Query-stationary fused multi-field scoring + streaming top-k for LARGE query batches (sm_100a).
//
//   score[q, n] = sum_f w[q,f] * <q_vec[q], corpus[n, f, :]>  (+ base[q, n])  ->  per-CTA top-k
//
// Why a second tensor-core kernel: with docs on the UMMA M axis (score_tc.cu) a CTA can keep at most 64
// queries resident in shared memory next to the corpus ring, so Q=512 re-streams the corpus 8x through L2
// and the M=128 x N=64 SS-MMAs need 192 B/cycle of shared-memory reads (port: 128 B/cycle) - ncu round 1:
// tensor pipe 18 % active, DRAM 4.3x the algorithmic bytes.  Here the roles are swapped:
//
//   A  = 128 QUERIES per CTA, bf16, resident in TENSOR MEMORY for the whole kernel
//        (lane = query, dim/2 columns: 384 of the 512 columns at d=768) -> no shared-memory reads for A
//   B  = 64 docs x (KC x 64) K-elements per stage (up to 48 KB, SWIZZLE_128B), ONE 3-D TMA box per stage: the
//        tensor map views a corpus row as [dim/64 chunks][64], so a box lands as KC consecutive [rows x 128 B]
//        K-major blocks - one mbarrier round trip and one tcgen05.commit per 4*KC MMAs instead of per 4
//   D  = [128 queries x 64 docs] fp32 in the remaining 128 TMEM columns, double buffered
//   CG = 2: CTA pairs (cta_group::2, M = 256 queries): each CTA TMA-loads HALF of every doc tile and the
//        pair's tensor cores share it - L2->SM traffic and shared-memory reads per SM are halved.
//
// Epilogue orientation: TMEM lane = query, so an epilogue THREAD owns one query: its field weights, its
// running mixture accumulators (64 docs), its top-k admission threshold and its candidate list - the
// threshold test is a register compare, no shared-memory traffic, no atomics.
//
// Warp roles (224 threads, 1 CTA / SM, persistent over doc tiles): warp 0 TMA producer, warp 1 TMEM
// allocator + MMA issuer for even units, warp 6 MMA issuer for odd units (leader CTA only when CG = 2),
// warps 2..5 epilogue.  ES = 2 (single-field scorers): a SECOND epilogue set, warps 7..10 (352 threads).  With one
// field every MMA unit ends in a push phase; one set is busy ~1.8k cycles per unit against 1.5k cycles of tensor time
// and the issuers wait on the accumulator hand-back.  Set s owns accumulator buffer s, i.e. the units of half-tile s
// of every tile, with its own candidate lists (list index g*ES + s), so each set has two unit times per unit.
// grid = (q_tiles, workers): CTAs with the same blockIdx.y walk the same doc tiles for different query
// tiles (adjacent in launch order -> co-resident in time, so re-reads hit L2).
#include <cuda.h>

#include "common.cuh"
#include "kernels.h"
#include "tc_ptx.cuh"

namespace mfar {

constexpr int kQsThreads = 224;   // ES = 1; ES = 2 adds 4 epilogue warps
constexpr int kQsEpiBWarp = 7;    // first warp of the second epilogue set
__host__ __device__ constexpr int qs_threads(int es, bool sp = false) { return kQsThreads + (es - 1) * 128 + (sp ? 32 : 0); }

constexpr int kQsIssuerBWarp = 6;   // second MMA-issuing warp (odd units)
constexpr int kQsQ = 128;        // queries per CTA (TMEM lanes)
constexpr int kQsDocs = 64;      // docs per unit (UMMA N)
constexpr int kQsTmemCols = 512;
constexpr int kQsDCol = 384;     // accumulator columns start here (A occupies [0, dim/2) <= 384)
constexpr int kSpSlotBytes = 128 * kQsQ;   // one sparse element: 128 queries x 128 bytes (64 f16 / 32 f32 docs)
constexpr int kSpMaxSlots = 4;

struct QsParams {
  int64_t n_docs;
  int n_tiles, corpus_fields, field_begin, n_dense, k_chunks;
  const __nv_bfloat16* q_vecs;
  int dim;
  int Q;
  const float* w;
  int w_ld;
  const float* base;
  int64_t base_ld;
  const void* sparse;  // [Q, n_sparse, sparse_ld] f16/f32 gathered by the epilogue (exclusive with base), rows 32-B aligned
  int64_t sparse_ld;
  int n_sparse;
  int sparse_f16;
  int sp_slots;        // sparse ring depth (SP kernels)
  int64_t doc_id_base;
  int k;
  int stages;          // ring depth
  int kc_per_stage;    // 64-element K chunks per stage (divides k_chunks)
  TopkWorkspace ws;
  DocFilter filt;      // FILT only
};

// Issue the 4*KC MMAs of one shared-memory stage (KC K-major [rows x 64] blocks) into accumulator d_tmem.
// Fully unrolled: every TMEM address / descriptor offset is an immediate added to one uniform base.
template <int CG, int KC>
__device__ __forceinline__ void qs_issue_stage(uint32_t d_tmem, uint32_t a0, uint64_t desc0, uint32_t idesc,
                                               bool overwrite_first, uint32_t issue) {
  constexpr int kChunkDesc = ((kQsDocs / CG) * kChunkK * 2) >> 4;   // descriptor address units (16 B) per block
#pragma unroll
  for (int c = 0; c < KC; ++c) {
#pragma unroll
    for (int kk = 0; kk < kChunkK / kUmmaK; ++kk) {
      const uint32_t a_tmem = a0 + uint32_t(c * (kChunkK / 2) + kk * (kUmmaK / 2));
      const uint64_t b_desc = desc0 + uint64_t(c * kChunkDesc + kk * 2);
      const uint32_t acc = (c == 0 && kk == 0) ? (overwrite_first ? 0u : 1u) : 1u;
      if (CG == 2) umma_bf16_ts_cg2_pred(d_tmem, a_tmem, b_desc, idesc, acc, issue);
      else umma_bf16_ts_pred(d_tmem, a_tmem, b_desc, idesc, acc, issue);
    }
  }
}

// Sparse term of one query's 64 docs, gathered from the per-field score rows (mfar/data/index.py:111-118: the
// score_batch gather) and mixed with the query's softmax weights (weighting.py:29) into the same accumulators as the
// dense fields:  acc[c] += w[q, n_dense + j] * sparse[q, j, doc0 + c] - nothing is written back to HBM.
//
// Data path: the [Q, n_sparse, ld] tensor is a 3-D TMA tensor (ld | n_sparse | Q); one ELEMENT = the 128-byte run
// (64 f16 / 32 f32 docs) of one field for the CTA's 128 queries = a (128 B, 1, 128) box, 16 KB, landing 128-byte
// swizzled in a small shared-memory ring filled by a dedicated producer warp that runs up to kSpMaxSlots elements
// ahead.  The epilogue thread of query r reads row r of the slot (8 x LDS.128 with the swizzle XOR - conflict-free,
// each quarter-warp covers all 32 banks) after each dense field's accumulator drain.  Why TMA and not per-thread
// global loads: a thread owns one query, so its loads touch one private 128-byte line per field - measured, LDG.256
// from 128 threads sustains only ~7 GB/s per SM at DRAM latency (the L1 miss path's concurrency), which capped the
// Amazon-shaped Q=512 kernel at 7.9 ms however deep the register pipeline was (1 or 2 elements ahead, with or
// without L2 prefetch); the TMA queue is deep enough to keep the 16 KB boxes streaming.
__device__ __forceinline__ void qs_sparse_consume(const uint8_t* slot, int qloc, bool f16, int e, float wj,
                                                  float (&acc)[kQsDocs]) {
  const uint8_t* row = slot + qloc * 128;
  const int sw = qloc & 7;
  if (f16) {
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const uint4 v = *reinterpret_cast<const uint4*>(row + ((c ^ sw) << 4));
      const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int x = 0; x < 4; ++x) {
        const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w4[x]));
        acc[c * 8 + 2 * x] = fmaf(wj, f.x, acc[c * 8 + 2 * x]);
        acc[c * 8 + 2 * x + 1] = fmaf(wj, f.y, acc[c * 8 + 2 * x + 1]);
      }
    }
  } else if ((e & 1) == 0) {
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const float4 v = *reinterpret_cast<const float4*>(row + ((c ^ sw) << 4));
      acc[c * 4 + 0] = fmaf(wj, v.x, acc[c * 4 + 0]); acc[c * 4 + 1] = fmaf(wj, v.y, acc[c * 4 + 1]);
      acc[c * 4 + 2] = fmaf(wj, v.z, acc[c * 4 + 2]); acc[c * 4 + 3] = fmaf(wj, v.w, acc[c * 4 + 3]);
    }
  } else {
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const float4 v = *reinterpret_cast<const float4*>(row + ((c ^ sw) << 4));
      acc[32 + c * 4 + 0] = fmaf(wj, v.x, acc[32 + c * 4 + 0]); acc[32 + c * 4 + 1] = fmaf(wj, v.y, acc[32 + c * 4 + 1]);
      acc[32 + c * 4 + 2] = fmaf(wj, v.z, acc[32 + c * 4 + 2]); acc[32 + c * 4 + 3] = fmaf(wj, v.w, acc[32 + c * 4 + 3]);
    }
  }
}

// Compaction of the candidate lists of one epilogue warp (lane = query) that could overflow on the next unit, one list
// at a time by the whole warp.  Every round is a warp SELECT (4-ary search on the score word; it also yields the
// rank-r bound that is published).  The loop is software-pipelined over the lists: the keys of the NEXT list and the
// other CTAs' pooled bounds of THIS list's query are requested before this list's select runs, so neither L2 round
// trip sits on the critical path.  Deliberately NOT inlined: inlined, its ~30 extra live registers changed the
// allocation of the drain / FMA loop around it and cost the 5-field MAG shape 7 % (2.71 -> 2.90 ms at Q=512).
struct QsCompacted { uint64_t thr; int cnt; };

__device__ __noinline__ QsCompacted qs_compact_lists(unsigned need, uint64_t* my_list, int cnt, int qrow, uint64_t thr,
                                                     int lane, unsigned long long* pool, unsigned long long* gthr,
                                                     int q_pad, int k, int GL, int gl) {
  const int r = pooled_rank(k, GL);
  uint64_t v_cur[8];
  {
    const int l0 = __ffs(need) - 1;
    __syncwarp();                                    // the list's last pushes (this warp's own lanes) are visible
    warp_list_load(my_list + int64_t(l0 - lane) * kCandCap, __shfl_sync(0xffffffffu, cnt, l0), lane, v_cur);
  }
  while (need) {
    const int l = __ffs(need) - 1;
    need &= need - 1;
    const int cnt_l = __shfl_sync(0xffffffffu, cnt, l);
    const int qrow_l = __shfl_sync(0xffffffffu, qrow, l);
    uint64_t* list_l = my_list + int64_t(l - lane) * kCandCap;
    unsigned long long pl[kPoolPerLane];
    pool_load_others(pool, GL, q_pad, gl, qrow_l, lane, pl);
    uint64_t v_next[8];
    if (need) {
      const int ln = __ffs(need) - 1;
      warp_list_load(my_list + int64_t(ln - lane) * kCandCap, __shfl_sync(0xffffffffu, cnt, ln), lane, v_next);
    }
    int cnt_new = k;
    uint64_t bound_r = 0ull;
    const uint64_t kth = warp_select_keys(v_cur, list_l, cnt_l, k, kCandCap - kQsDocs, lane, &cnt_new, r, &bound_r);
    const unsigned long long pooled = pool_publish_min(pool, GL, q_pad, gl, qrow_l, bound_r, lane, pl);
    if (lane == l) {
      thr = kth > thr ? kth : thr;
      thr = pooled > thr ? pooled : thr;
      cnt = cnt_new;
      atomicMax(gthr + qrow, thr);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) v_cur[j] = v_next[j];
    __syncwarp();
  }
  return QsCompacted{thr, cnt};
}

// CTAs that ran in 4-CTA clusters, since the last mfar_profile_cluster4_ctas() (one atomic per CTA)
__device__ unsigned long long g_qs_cluster4_ctas;

// SP: the epilogue gathers the sparse fields itself (qs_seed_sparse) - a separate instantiation, so the dense-only
// kernels keep their register allocation.  map_bh: the corpus view of map_b with half its K chunks per box (the
// multicast loads of a 4-CTA cluster).
// FILT: doc filter.  A thread owns a query over a half-tile of 64 docs: its 64-bit window of the query's row (3 words
// and a funnel shift at bit doc_id_base + doc0) is loaded at the head of the half-tile and tested next to the key
// compare.
template <int CG, int ES, bool SP, bool FILT>
__global__ void __launch_bounds__(qs_threads(ES, SP), 1)
score_qs_kernel(const __grid_constant__ CUtensorMap map_b, const __grid_constant__ CUtensorMap map_bh,
                const __grid_constant__ CUtensorMap map_sp, QsParams p) {
  constexpr int kRowsPerCta = kQsDocs / CG;               // doc rows this CTA loads per stage
  constexpr int kChunkBytes = kRowsPerCta * kChunkK * 2;  // one [rows x 64] K-major block: 8 KB (CG=1) / 4 KB (CG=2)
  const int kStageBytes = p.kc_per_stage * kChunkBytes;
  const int stages_per_unit = p.k_chunks / p.kc_per_stage;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_b = smem;
  uint8_t* smem_sp = smem_b + size_t(p.stages) * kStageBytes;                          // [sp_slots][16 KB], 1024-aligned
  const int sp_slots = SP ? p.sp_slots : 0;
  const int sp_ring = SP ? p.sp_slots : 1;           // ring arithmetic below (1: well-defined in the dense-only instantiations)
  float* w_s = reinterpret_cast<float*>(smem_sp + size_t(sp_slots) * kSpSlotBytes);    // [n_dense (+ n_sparse)][128]
  const int n_w = p.n_dense + (SP ? p.n_sparse : 0);   // weight rows kept in shared memory
  uint64_t* bars = reinterpret_cast<uint64_t*>(w_s + size_t(n_w) * kQsQ);
  uint64_t* full_bar = bars;                       // [stages]  (leader's are the ones waited on)
  uint64_t* empty_bar = bars + p.stages;           // [stages]
  uint64_t* tfull_bar = bars + 2 * p.stages;       // [2]
  uint64_t* tempty_bar = tfull_bar + 2;            // [2]       (leader's are the ones waited on)
  uint64_t* sfull_bar = tempty_bar + 2;            // [kSpMaxSlots] sparse ring: producer warp -> epilogue
  uint64_t* sempty_bar = sfull_bar + kSpMaxSlots;  // [kSpMaxSlots] epilogue (4 warps of the consuming set) -> producer
  uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(sempty_bar + kSpMaxSlots);

  const int warp = __shfl_sync(0xffffffffu, int(threadIdx.x >> 5), 0);   // warp-uniform for the compiler too
  const int lane = threadIdx.x & 31;
#ifdef MFAR_QS_TIMING
  const long long t_kernel0 = clock64();
#endif
  const int g = blockIdx.y;                        // worker: walks tiles g, g+G, ...
  const int G = gridDim.y;
  const int q0 = blockIdx.x * kQsQ;                // first query of this CTA
  const uint32_t cta_rank = (CG == 2) ? cluster_ctarank() : 0u;
  // A 4-CTA cluster (launched as the preferred cluster shape) is the two pairs of one worker column: ranks {0,1} and
  // {2,3}, each a cta_group::2 pair with its even rank as leader.  Where the GPC had no room, the hardware formed
  // 2-CTA clusters instead; a column can come up either way.
  const uint32_t cl_size = (CG == 2) ? cluster_nctarank() : 1u;
  const bool mc = CG == 2 && cl_size == 4;         // doc tiles shared between the pairs by TMA multicast
  const bool leader = (cta_rank & 1u) == 0;
  const uint32_t pair_mask = 0x3u << (cta_rank & 2u);
  int* err = p.ws.err;

  // ---- one-time setup
  for (int i = threadIdx.x; i < n_w * kQsQ; i += qs_threads(ES, SP)) {
    const int f = i / kQsQ, c = i % kQsQ;
    w_s[i] = (q0 + c < p.Q) ? p.w[int64_t(q0 + c) * p.w_ld + f] : 0.f;
  }
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_b);
    // multicast: a stage slot is written by both pairs' producers, so both pairs' MMAs must have consumed it
    for (int s = 0; s < p.stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], mc ? 2 : 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&tfull_bar[b], 1); mbar_init(&tempty_bar[b], 4 * CG); }
    for (int b = 0; b < kSpMaxSlots; ++b) { mbar_init(&sfull_bar[b], 1); mbar_init(&sempty_bar[b], 4); }
    if (SP) tma_prefetch_desc(&map_sp);
    if (mc) { tma_prefetch_desc(&map_bh); atomicAdd(&g_qs_cluster4_ctas, 1ull); }
    fence_barrier_init();
  }
  if (warp == 1) {
    if (CG == 2) { tmem_alloc_cg2(tmem_ptr_s, kQsTmemCols); tmem_relinquish_cg2(); }
    else { tmem_alloc(tmem_ptr_s, kQsTmemCols); tmem_relinquish(); }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  // The whole tensor memory (512 columns) is allocated, so the allocation can only start at lane 0 / column 0.
  // Using the literal keeps every TMEM address of the MMA issue loop in uniform registers (no per-instruction
  // R2UR of a value loaded from shared memory); anything else is a driver/hardware surprise -> trap.
  if (*tmem_ptr_s != 0u) {
    if (threadIdx.x == 0) atomicExch(err, 21);
    __threadfence_system();
    asm volatile("trap;");
  }
  constexpr uint32_t tmem_base = 0u;

  // ---- queries -> tensor memory (A operand): lane = query, column c holds elements 2c, 2c+1
  if (warp >= 2 && warp < 6) {
    const int lane_grp = warp & 3;
    const int qrow = q0 + lane_grp * 32 + lane;
    const uint4* src = reinterpret_cast<const uint4*>(p.q_vecs + int64_t(qrow) * p.dim);
    const uint32_t taddr = tmem_base + (uint32_t(lane_grp * 32) << 16);
    for (int c0 = 0; c0 < p.dim / 2; c0 += 16) {   // 16 columns = 32 bf16 = 4 x 16-byte loads
      uint32_t v[16];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint4 x = make_uint4(0, 0, 0, 0);
        if (qrow < p.Q) x = __ldg(src + c0 / 4 + j);
        v[4 * j + 0] = x.x; v[4 * j + 1] = x.y; v[4 * j + 2] = x.z; v[4 * j + 3] = x.w;
      }
      tmem_st16(taddr + c0, v);
    }
    tmem_st_wait();
  }
  tc_fence_before();
  if (CG == 2) cluster_sync_all(); else __syncthreads();
  tc_fence_after();

  const int my_tiles = (p.n_tiles > g) ? (p.n_tiles - g + G - 1) / G : 0;
  const int units = my_tiles * 2 * p.n_dense;      // (tile, half, field)
#ifdef MFAR_QS_TIMING
  const long long t_setup_done = clock64();
  if (threadIdx.x == 0 && blockIdx.x == 0 && blockIdx.y == 0)
    printf("[qs timing] setup (barriers, TMEM alloc, queries -> TMEM) %lld cycles\n", t_setup_done - t_kernel0);
#endif

  if (warp == 0) {
    // ===================================================================== TMA producer (every CTA)
    {                                               // whole warp walks the loop, one elected lane issues
      // Stage ownership: the two MMA-issuing warps alternate units, and a parity wait on an mbarrier is only sound for
      // a waiter that observes every phase of that barrier in turn - so each issuer owns HALF of the ring (stages
      // [b * S, (b + 1) * S) for the issuer of accumulator buffer b) and the producer fills unit u into the half of
      // issuer u & 1.  (With one shared ring an issuer's first visit to a stage could be for its SECOND fill and pass
      // the parity test before the first fill had landed: harmless for the 4-stage / 2-per-unit geometry round 1
      // shipped, where the split happens to coincide with ring order, fatal for others.)
      const int S_half = p.stages >> 1;
      int st0 = 0, st1 = 0;                        // next stage inside the half of issuer 0 / 1
      uint32_t ph0 = 0u, ph1 = 0u;
      int unit = 0;
      // Query groups (CTA pairs / CTAs with the same blockIdx.y) stream the SAME doc tiles.  They are kept within
      // one sync interval (a half-tile of >= 8 fields) of each other through per-group progress counters so that the second reader of a tile
      // hits L2 instead of HBM (ncu before: DRAM read 1.8x the corpus at Q=512).  Bounded spin: a group that is
      // not co-resident (SMs taken by another kernel) only costs lockstep, never a deadlock.
      const int n_groups = gridDim.x / CG;
      const int my_group = blockIdx.x / CG;
      int* prog = p.ws.progress + g * n_groups;
      // (the pairs of one cluster are already held together by the shared stage slots: a column that is one cluster
      // needs no counters)
      bool lockstep = n_groups > 1 && leader && gridDim.x > cl_size && (G * n_groups <= kProgressInts);
      // a sync point every ~8 MMA units (= every half-tile when n_dense >= 8): the global round trip must not sit
      // in front of every TMA issue of a few-field scorer
      const int sync_every = p.n_dense >= 8 ? 1 : (8 + p.n_dense - 1) / p.n_dense;
      for (int i = 0; i < my_tiles; ++i) {
        const int t = g + i * G;
        for (int h = 0; h < 2; ++h) {
          if (lockstep && ((2 * i + h) % sync_every) == 0) {
            if (lane == 0) {
              const int idx = (2 * i + h) / sync_every;               // sync point number
              st_release_gpu(prog + my_group, idx + 1);             // "I am past sync point idx"
              const unsigned long long t0 = clock64();
              for (int o = 0; o < n_groups && lockstep; ++o) {
                while (ld_acquire_gpu(prog + o) < idx) {            // o has not reached sync point idx - 1 yet
                  if (clock64() - t0 > 200000ull) { lockstep = false; break; }   // ~100 us: give up for good
                  __nanosleep(200);
                }
              }
            }
            lockstep = __shfl_sync(0xffffffffu, int(lockstep), 0) != 0;
          }
          for (int f = 0; f < p.n_dense; ++f) {
            const int row0 = (t * p.corpus_fields + p.field_begin + f) * kTileDocs + h * kQsDocs +
                             int(cta_rank & 1u) * kRowsPerCta;
            const int ib = unit & 1;                // issuer (= accumulator buffer) of this unit
            ++unit;
            for (int s = 0; s < stages_per_unit; ++s) {
              const int stage = ib ? S_half + st1 : st0;
              const uint32_t phase = ib ? ph1 : ph0;
              mbar_wait(&empty_bar[stage], phase ^ 1, err, 11);
              if (elect_one()) {
                if (mc) {
                  // CTA r and r ^ 2 need the same rows: each loads one K half of the stage into both of them
                  const int half = p.kc_per_stage >> 1;
                  const int kh = int(cta_rank >> 1) * half;
                  if (leader) mbar_expect_tx(&full_bar[stage], kStageBytes * 2);
                  tma_load_3d_cg2_mc(&map_bh, &full_bar[stage], smem_b + size_t(stage) * kStageBytes + size_t(kh) * kChunkBytes,
                                     0, row0, s * p.kc_per_stage + kh, uint16_t((1u << cta_rank) | (1u << (cta_rank ^ 2u))));
                } else if (CG == 2) {
                  if (leader) mbar_expect_tx(&full_bar[stage], kStageBytes * 2);
                  tma_load_3d_cg2(&map_b, &full_bar[stage], smem_b + size_t(stage) * kStageBytes, 0, row0,
                                  s * p.kc_per_stage);
                } else {
                  mbar_expect_tx(&full_bar[stage], kStageBytes);
                  tma_load_3d(&map_b, &full_bar[stage], smem_b + size_t(stage) * kStageBytes, 0, row0,
                              s * p.kc_per_stage);
                }
              }
              __syncwarp();
              if (ib) { if (++st1 == S_half) { st1 = 0; ph1 ^= 1u; } }
              else { if (++st0 == S_half) { st0 = 0; ph0 ^= 1u; } }
            }
          }
        }
      }
      // The MMAs of another pair release this CTA's stages through remote commits: wait until every stage has been
      // released after its last fill, so that no commit lands in this CTA's shared memory after it has exited.
      if (CG == 2) {
        for (int i = 0; i < S_half; ++i) {
          mbar_wait(&empty_bar[st0], ph0 ^ 1, err, 11);
          mbar_wait(&empty_bar[S_half + st1], ph1 ^ 1, err, 11);
          if (++st0 == S_half) { st0 = 0; ph0 ^= 1u; }
          if (++st1 == S_half) { st1 = 0; ph1 ^= 1u; }
        }
      }
    }
  } else if (SP && warp == qs_threads(ES) / 32) {
    // ===================================================================== sparse producer (last warp, every CTA)
    // elements in the order the epilogue sets consume them: ES = 1: (tile, half, element); ES = 2: (tile, element,
    // half) - the two sets then own the even / odd slots of the ring
    const int n_elems = p.n_sparse * (p.sparse_f16 ? 1 : 2);
    const int per_elem_docs = p.sparse_f16 ? 64 : 32;
    int seq = 0;
    for (int i = 0; i < my_tiles; ++i) {
      const int64_t tile_doc0 = int64_t(g + i * G) * kTileDocs;
      for (int a = 0; a < (ES == 2 ? n_elems : 2); ++a) {
        for (int b = 0; b < (ES == 2 ? 2 : n_elems); ++b) {
          const int h = ES == 2 ? b : a, e = ES == 2 ? a : b;
          const int64_t doc0 = tile_doc0 + h * kQsDocs;
          if (doc0 < p.n_docs) {                     // (the epilogue skips a half-tile past the last doc too)
            const int slot = seq % sp_ring;
            mbar_wait(&sempty_bar[slot], ((seq / sp_ring) & 1) ^ 1, err, 16);
            if (elect_one()) {
              mbar_expect_tx(&sfull_bar[slot], kSpSlotBytes);
              const int j = p.sparse_f16 ? e : (e >> 1);
              const int64_t d = doc0 + (p.sparse_f16 ? 0 : (e & 1) * per_elem_docs);
              tma_load_3d(&map_sp, &sfull_bar[slot], smem_sp + size_t(slot) * kSpSlotBytes, int(d), j, q0);
            }
            __syncwarp();
          }
          ++seq;
        }
      }
    }
  } else if (warp == 1 || warp == kQsIssuerBWarp) {
    // ===================================================================== MMA issuers (leader CTA)
    // TWO issuing warps: warp 1 owns the even units (accumulator buffer 0), warp 6 the odd units (buffer 1).
    // An M=256 x N=64 x K=16 MMA occupies the tensor pipe for 32 cycles but costs a single warp ~65 cycles of
    // issue work (descriptor arithmetic, elect, uniform-register moves) - measured 3330 cycles per 48-MMA unit
    // against a 1536-cycle floor.  Two warps feed the in-order tensor pipe from both sides; tcgen05.commit
    // tracks the issuing thread's own MMAs, so each warp releases exactly the stages / accumulator it consumed.
    if (leader) {                                   // whole warp walks the loop, one elected lane issues
      constexpr uint32_t idesc = make_idesc(kQsQ * CG, kQsDocs);
      const int buf = (warp == 1) ? 0 : 1;
      const uint32_t issue = elect_one() ? 1u : 0u;
      const uint32_t d_tmem = tmem_base + uint32_t(kQsDCol + buf * kQsDocs);
#ifdef MFAR_QS_TIMING
      long long t_tempty = 0, t_full = 0, t_issue = 0, t_prev = clock64();
#define QS_TICK(acc) { const long long _n = clock64(); acc += _n - t_prev; t_prev = _n; }
#else
#define QS_TICK(acc)
#endif
      for (int u = buf; u < units; u += 2) {
        mbar_wait(&tempty_bar[buf], ((u >> 1) & 1) ^ 1, err, 13);
        QS_TICK(t_tempty)
        tc_fence_after();
        for (int s = 0; s < stages_per_unit; ++s) {
          const int ring = (u >> 1) * stages_per_unit + s;   // position in this issuer's half of the ring
          const int S_half = p.stages >> 1;
          const int stage = buf * S_half + ring % S_half;
          const uint32_t phase = uint32_t(ring / S_half) & 1u;
          mbar_wait(&full_bar[stage], phase, err, 14);
          QS_TICK(t_full)
          tc_fence_after();
          const uint32_t stage_addr = smem_u32(smem_b + size_t(stage) * kStageBytes);
          const uint64_t desc0 = make_sw128_desc(stage_addr);
          const uint32_t a0 = tmem_base + uint32_t(s * p.kc_per_stage * (kChunkK / 2));
          const bool first_stage = (s == 0);
          if (p.kc_per_stage == 12) qs_issue_stage<CG, 12>(d_tmem, a0, desc0, idesc, first_stage, issue);
          else if (p.kc_per_stage == 6) qs_issue_stage<CG, 6>(d_tmem, a0, desc0, idesc, first_stage, issue);
          else
            for (int c = 0; c < p.kc_per_stage; ++c) qs_issue_stage<CG, 1>(d_tmem, a0 + uint32_t(c * (kChunkK / 2)),
                                                                            desc0 + uint64_t(c * (kChunkBytes >> 4)),
                                                                            idesc, first_stage && c == 0, issue);
          __syncwarp();
          if (elect_one()) {
            if (CG == 2) tc_commit_cg2(&empty_bar[stage], mc ? 0xF : pair_mask); else tc_commit(&empty_bar[stage]);
          }
        }
        if (elect_one()) { if (CG == 2) tc_commit_cg2(&tfull_bar[buf], pair_mask); else tc_commit(&tfull_bar[buf]); }
        __syncwarp();
        QS_TICK(t_issue)
      }
#ifdef MFAR_QS_TIMING
      if (lane == 0 && blockIdx.y == 0 && blockIdx.x == 0)
        printf("[qs timing] issuer %d: units %d  cycles/unit: wait_tempty %.0f wait_full %.0f issue %.0f\n", buf,
               (units + 1 - buf) / 2, double(t_tempty) / ((units + 1 - buf) / 2), double(t_full) / ((units + 1 - buf) / 2),
               double(t_issue) / ((units + 1 - buf) / 2));
#endif
    }
  } else {
    // ===================================================================== epilogue: thread = query
    const int lane_grp = warp & 3;
    const int qloc = lane_grp * 32 + lane;
    const int qrow = q0 + qloc;
    const bool q_valid = qrow < p.Q;
    const int eset = (ES == 2 && warp >= kQsEpiBWarp) ? 1 : 0;     // epilogue set = accumulator buffer it drains
    const int gl = g * ES + eset;                                  // candidate-list owner index (ES lists per CTA)
    const int GL = G * ES;
    uint64_t* my_list = p.ws.cand_keys + (int64_t(gl) * p.ws.q_pad + qrow) * kCandCap;
    const float* my_base = p.base ? p.base + int64_t(q_valid ? qrow : 0) * p.base_ld : nullptr;
    uint64_t thr = 0ull;
    int cnt = 0;
    const int refresh_mask = p.n_dense >= 8 ? 0 : (p.n_dense >= 4 ? 1 : (p.n_dense >= 2 ? 3 : 7));
    float acc[kQsDocs];
    int u = 0;
    // fused sparse gather (SP): position of this epilogue set in the sparse ring (see the producer warp)
    const int sp_elems = SP ? p.n_sparse * (p.sparse_f16 ? 1 : 2) : 0;
    int sp_seq = (ES == 2) ? eset : 0;               // ES = 2: set s consumes elements s, s + 2, ...
    auto sp_step = [&](int sp_e, float (&acc_)[kQsDocs]) {
      const int slot = sp_seq % sp_ring;
      mbar_wait(&sfull_bar[slot], (sp_seq / sp_ring) & 1, err, 17);
      const int j = p.sparse_f16 ? sp_e : (sp_e >> 1);
      qs_sparse_consume(smem_sp + size_t(slot) * kSpSlotBytes, qloc, p.sparse_f16 != 0, sp_e,
                        w_s[(p.n_dense + j) * kQsQ + qloc], acc_);
      __syncwarp();
      if (lane == 0) mbar_arrive(&sempty_bar[slot]);
      sp_seq += ES;
    };
#ifdef MFAR_QS_TIMING
    long long e_wait = 0, e_drain = 0, e_push = 0, e_compact = 0, e_prev = clock64();
    int n_compact = 0;
#define QS_ETICK(acc_) { const long long _n = clock64(); acc_ += _n - e_prev; e_prev = _n; }
#else
#define QS_ETICK(acc_)
#endif
    int n_push = 0;
    for (int i = 0; i < my_tiles; ++i) {
      const int t = g + i * G;
      for (int h = (ES == 2 ? eset : 0); h < (ES == 2 ? eset + 1 : 2); ++h) {
        if (ES == 2) u = 2 * i + h;                              // single field: unit index == half-tile index
        const int64_t doc0 = int64_t(t) * kTileDocs + h * kQsDocs;
        // accumulators start from the pre-mixed sparse term (16 x 16-byte loads per query row, issued ahead of the
        // wait for the half-tile's first accumulator; base_ld is a multiple of 128, so the row read stays in bounds)
        const bool sp_live = SP && doc0 < p.n_docs;   // warp-uniform: padding queries read TMA zero fill
        // the best threshold any CTA found for this query: requested now, used after the half-tile's last field (an L2
        // round trip that used to sit in front of every push phase)
        const bool refresh = q_valid && ((n_push++ & refresh_mask) == 0);
        unsigned long long gt_new = 0ull;
        if (refresh) gt_new = ld_relaxed_u64(p.ws.gthr + qrow);
        uint32_t fx[3] = {0u, 0u, 0u};               // FILT: words of docs doc0 .. doc0 + 63 (padding queries: none)
        if (FILT && q_valid && doc0 < p.n_docs) {
          const uint32_t* frow = p.filt.bits + int64_t(qrow) * p.filt.stride;
          const int64_t w0 = (p.doc_id_base + doc0) >> 5;
#pragma unroll
          for (int j = 0; j < 3; ++j) fx[j] = filter_ld_word(frow, p.filt.words, w0 + j);
        }
        int sp_e = 0;                                // next sparse element of this half-tile to consume
        if (sp_live) {
#pragma unroll
          for (int c = 0; c < kQsDocs; ++c) acc[c] = 0.f;
        } else if (my_base != nullptr && q_valid && doc0 < p.n_docs) {
          const float4* b4 = reinterpret_cast<const float4*>(my_base + doc0);
#pragma unroll
          for (int c = 0; c < kQsDocs; c += 4) {
            const float4 b = __ldg(b4 + c / 4);
            acc[c] = b.x; acc[c + 1] = b.y; acc[c + 2] = b.z; acc[c + 3] = b.w;
          }
        } else {
#pragma unroll
          for (int c = 0; c < kQsDocs; ++c) acc[c] = 0.f;
        }
        for (int f = 0; f < p.n_dense; ++f, ++u) {
          const int buf = u & 1;
          mbar_wait(&tfull_bar[buf], (u >> 1) & 1, err, 15);
          QS_ETICK(e_wait)
          tc_fence_after();
          const uint32_t taddr = tmem_base + (uint32_t(lane_grp * 32) << 16) + uint32_t(kQsDCol + buf * kQsDocs);
          const float wf = w_s[f * kQsQ + qloc];
          {
            // drain the whole accumulator into registers and hand the TMEM buffer back BEFORE the FMAs: the
            // release -> next MMA chain (cross-CTA in pair mode) is what bounds the unit rate, not the arithmetic
            uint32_t v[kQsDocs];
#pragma unroll
            for (int c0 = 0; c0 < kQsDocs; c0 += 16)
              tmem_ld16(taddr + c0, *reinterpret_cast<uint32_t(*)[16]>(&v[c0]));
            tmem_ld_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {                         // one arrival per epilogue warp frees the accumulator buffer
              if (CG == 2) mbar_arrive_cluster(&tempty_bar[buf], cta_rank & ~1u); else mbar_arrive(&tempty_bar[buf]);
            }
#pragma unroll
            for (int c = 0; c < kQsDocs; ++c) acc[c] = fmaf(wf, __uint_as_float(v[c]), acc[c]);
          }
          if (sp_live && sp_e < sp_elems) { sp_step(sp_e, acc); ++sp_e; }   // one sparse element per dense field
          QS_ETICK(e_drain)
        }
        while (sp_live && sp_e < sp_elems) { sp_step(sp_e, acc); ++sp_e; }  // more sparse elements than dense fields
        // ---- 64 docs scored under every field: threshold filter, push
        // adopt the best threshold any CTA found for this query - an L2 round trip, so not more often than once
        // per ~8 MMA units (every half-tile when n_dense >= 8, every 8th for a single_ scorer)
        thr = gt_new > thr ? gt_new : thr;                               // incl. the pooled bound, common.cuh
        if (q_valid && doc0 < p.n_docs) {
          const int64_t left = p.n_docs - doc0;
          const int nd = left < kQsDocs ? int(left) : kQsDocs;
          const uint32_t id0 = uint32_t(p.doc_id_base + doc0);
          // one float compare per doc rejects almost everything; the exact (score, id) key is only built for docs
          // whose score reaches the threshold's score (thr == 0: nothing established yet, admit all)
          const float thr_f = thr ? key_score(thr) : -INFINITY;
          const uint32_t fsh = uint32_t((p.doc_id_base + doc0) & 31);
          const uint64_t fwin =                                     // FILT: bit c <=> doc doc0 + c is eligible
              FILT ? (uint64_t(__funnelshift_r(fx[1], fx[2], fsh)) << 32) | __funnelshift_r(fx[0], fx[1], fsh) : 0ull;
          // ... and one compare per GROUP of 8 docs (max tree: 3 FMNMX/FMNMX3 + 1 FSETP instead of 8 FSETP + 8
          // branches) rejects almost every group once a threshold exists - with a single_ scorer this push phase runs
          // after every MMA unit.  (A branch-free 64-bit pass mask was measured too: its 3 instructions per doc cost
          // more than the 8 group branches it saves - single_ Q=512 8.2 ms vs 7.5 ms.)
#pragma unroll
          for (int c0 = 0; c0 < kQsDocs; c0 += 8) {
            // NaN-propagating max and !(x < thr_f): a NaN score (or a NaN threshold) reaches the key compare
            const float m = fmax_nan(fmax_nan(fmax_nan(acc[c0], acc[c0 + 1]), fmax_nan(acc[c0 + 2], acc[c0 + 3])),
                                     fmax_nan(fmax_nan(acc[c0 + 4], acc[c0 + 5]), fmax_nan(acc[c0 + 6], acc[c0 + 7])));
            if (!(m < thr_f)) {
#pragma unroll
              for (int c = c0; c < c0 + 8; ++c) {
                if (c < nd && !(acc[c] < thr_f)) {
                  const uint64_t key = make_key(acc[c], id0 + c);
                  if (key > thr && (!FILT || ((fwin >> c) & 1ull))) { __stcg(my_list + cnt, key); ++cnt; }
                }
              }
            }
          }
        }
        QS_ETICK(e_push)
        // ---- lists that could overflow on the next unit are compacted by the whole warp, one at a time
        unsigned need = __ballot_sync(0xffffffffu, cnt > kCandCap - kQsDocs);
#ifdef MFAR_QS_TIMING
        n_compact += __popc(need);
#endif
        if (need) {
          const QsCompacted c = qs_compact_lists(need, my_list, cnt, qrow, thr, lane, p.ws.pool, p.ws.gthr, p.ws.q_pad,
                                                 p.k, GL, gl);
          thr = c.thr;
          cnt = c.cnt;
        }
        QS_ETICK(e_compact)
      }
    }
#ifdef MFAR_QS_TIMING
    if (lane == 0 && blockIdx.y == 0 && blockIdx.x == 0)
      printf("[qs timing] epilogue warp %d: units %d kcycles: wait %lld drain %lld push %lld compact %lld (lists compacted %d)\n",
             warp, units, e_wait / 1000, e_drain / 1000, e_push / 1000, e_compact / 1000, n_compact);
#endif
    if (q_valid) {
      p.ws.cand_cnt[int64_t(gl) * p.ws.q_pad + qrow] = cnt;
      p.ws.cand_thr[int64_t(gl) * p.ws.q_pad + qrow] = thr;
    }
  }

  // ---- teardown
  tc_fence_before();
  if (CG == 2) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  if (warp == 1) {
    if (CG == 2) tmem_dealloc_cg2(tmem_base, kQsTmemCols); else tmem_dealloc(tmem_base, kQsTmemCols);
  }
}

// ------------------------------------------------------------------------------------ host side
bool score_qs_supported(const ScoreArgs& a) {
  return a.n_dense >= 1 && a.corpus_dtype != MFAR_E4M3 && a.dim % kChunkK == 0 && a.dim >= kChunkK && a.dim / 2 <= kQsDCol &&
         (reinterpret_cast<uintptr_t>(a.corpus) % 16 == 0) && (reinterpret_cast<uintptr_t>(a.q_vecs) % 16 == 0) &&
         int64_t(a.n_tiles) * a.corpus_fields * kTileDocs < (int64_t(1) << 31);
}

// n_dense = 0 plans the reservation of mfar_score_topk_workspace_bytes, which does not know n_dense: two lists per
// worker at every batch size
PassPlan plan_score_qs(int Q, int n_tiles, int n_dense) {
  PassPlan p{};
  p.impl = MFAR_IMPL_TCGEN05_QS;
  const int qt = (Q + kQsQ - 1) / kQsQ;
  p.cg = qt >= 2 ? 2 : 1;
  p.q_tiles = round_up(qt, p.cg);
  p.q_pad = kQsQ;
  p.q_pad_total = p.q_pad * p.q_tiles;
  int w = kNumSmsB200 / p.q_tiles;
  if (w > n_tiles) w = n_tiles;
  if (w < 1) w = 1;
  p.workers = w;
  // two epilogue sets, each with its own lists, only where the epilogue is the bound: single-field scorers in CTA-pair
  // mode (Q > 128); at Q <= 128 the kernel is HBM-bound and the extra warps measured ~3 % slower
  p.lists = (n_dense == 0 || (n_dense == 1 && p.cg == 2)) ? 2 * w : w;
  return p;
}

static size_t qs_smem_bytes(int n_weights, int stages, int stage_bytes, int sp_slots) {
  return 1024 + size_t(stages) * stage_bytes + size_t(sp_slots) * kSpSlotBytes + size_t(n_weights) * kQsQ * 4 +
         (2 * stages + 4 + 2 * kSpMaxSlots) * 8 + 16;
}

template <int CG, int ES, bool SP, bool FILT>
static int launch_qs_impl(const ScoreArgs& a, const PassPlan& plan, const TopkWorkspace& ws, cudaStream_t st) {
  constexpr int kChunkBytes = (kQsDocs / CG) * kChunkK * 2;
  QsParams p;
  p.n_docs = a.n_docs; p.n_tiles = a.n_tiles; p.corpus_fields = a.corpus_fields; p.field_begin = a.field_begin;
  p.n_dense = a.n_dense; p.k_chunks = a.dim / kChunkK; p.q_vecs = static_cast<const __nv_bfloat16*>(a.q_vecs);
  p.dim = a.dim; p.Q = a.Q; p.w = a.w; p.w_ld = a.w_ld; p.base = a.base; p.base_ld = a.base_ld;
  p.doc_id_base = a.doc_id_base; p.k = a.k;
  p.sparse = a.sparse; p.sparse_ld = a.sparse_ld; p.n_sparse = a.sparse ? a.n_sparse : 0;
  p.sparse_f16 = a.sparse_dtype == MFAR_F16;
  const int n_w = a.n_dense + p.n_sparse;
  p.ws = ws;
  p.filt = DocFilter{a.filter_bits, a.filter_stride, a.filter_words};
  const size_t smem_cap = 227 * 1024;
  // Shared memory: corpus ring + (SP) sparse ring of 16 KB slots + weights + barriers.  The corpus ring is split in two
  // halves, one per MMA-issuing warp (see the producer), so `stages` is even.  Dense-only: stages of up to 48 KB, 192 KB
  // of ring.  SP: stages of up to 24 KB so that three per issuer fit next to the sparse ring.
  const int stage_cap = SP ? 24 * 1024 : 48 * 1024;
  int kc = 1;                                       // largest divisor of k_chunks within the stage cap
  for (int d = 1; d <= p.k_chunks; ++d)
    if (p.k_chunks % d == 0 && d * kChunkBytes <= stage_cap) kc = d;
  p.kc_per_stage = kc;
  const int kStageBytes = kc * kChunkBytes;
  auto max_stages = [&](int slots) {                // largest even stage count that fits with `slots` sparse slots
    int st = int((192 * 1024) / kStageBytes) & ~1;
    while (st > 2 && qs_smem_bytes(n_w, st, kStageBytes, slots) > smem_cap) st -= 2;
    return st < 2 ? 2 : st;
  };
  int sp_slots = 0;
  if (SP) {                                         // deepest sparse ring that still leaves >= 3 corpus stages per issuer
    sp_slots = kSpMaxSlots;
    while (sp_slots > 2 && max_stages(sp_slots) * kStageBytes < 6 * 24 * 1024 &&
           max_stages(sp_slots - (ES == 2 ? 2 : 1)) > max_stages(sp_slots))
      sp_slots -= (ES == 2 ? 2 : 1);                // ES = 2: the two epilogue sets own the even / odd slots
  }
  const int stages = max_stages(sp_slots);
  p.stages = stages;
  p.sp_slots = sp_slots;
  const size_t smem = qs_smem_bytes(n_w, stages, kStageBytes, sp_slots);
  if (smem > smem_cap) return MFAR_ERR_SHAPE;

  // Two CTA pairs per cluster where they read the same doc tiles (grid x = query tiles: one cluster of 4 is two pairs
  // of one worker column) and a stage splits into two K halves: each doc tile then crosses from L2 to the SMs once per
  // column instead of once per pair.  A preferred cluster, not a required one: GPCs with no room for 4 CTAs get
  // 2-CTA clusters, so every SM stays busy.
  const bool cluster4 = CG == 2 && plan.q_tiles % 4 == 0 && kc % 2 == 0;
  const uint64_t corpus_rows = uint64_t(a.n_tiles) * a.corpus_fields * kTileDocs;
  CUtensorMap map_b;
  int rc = make_tensor_map_kchunked(&map_b, a.corpus, corpus_rows, a.dim, kQsDocs / CG, kc,
                                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B);
  if (rc) return rc;
  CUtensorMap map_bh = map_b;                       // unused unless cluster4
  if (cluster4) {
    rc = make_tensor_map_kchunked(&map_bh, a.corpus, corpus_rows, a.dim, kQsDocs / CG, kc / 2,
                                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B);
    if (rc) return rc;
  }
  CUtensorMap map_sp = map_b;                       // unused by the dense-only kernels
  if (SP) {
    rc = make_tensor_map_sparse_rows(&map_sp, a.sparse, a.sparse_dtype == MFAR_F16, uint64_t(a.sparse_ld),
                                     uint64_t(a.sparse_cols ? a.sparse_cols : a.sparse_ld), uint32_t(a.n_sparse),
                                     uint64_t(a.Q), kQsQ);
    if (rc) return rc;
  }
  static PerDeviceOnce attr_once;   // per template instantiation
  MFAR_CUDA_OK(attr_once.run([&] {
    return cudaFuncSetAttribute(score_qs_kernel<CG, ES, SP, FILT>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem_cap));
  }));
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(plan.q_tiles, plan.workers);
  cfg.blockDim = dim3(qs_threads(ES, SP));
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CG; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributePreferredClusterDimension;
  attr[1].val.preferredClusterDim.x = 4; attr[1].val.preferredClusterDim.y = 1; attr[1].val.preferredClusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = cluster4 ? 2 : 1;
  MFAR_CUDA_OK(cudaLaunchKernelEx(&cfg, score_qs_kernel<CG, ES, SP, FILT>, map_b, map_bh, map_sp, p));
  return MFAR_OK;
}

long long qs_cluster4_ctas_collect() {
  unsigned long long n = 0;
  const unsigned long long zero = 0;
  if (cudaMemcpyFromSymbol(&n, g_qs_cluster4_ctas, sizeof(n)) != cudaSuccess ||
      cudaMemcpyToSymbol(g_qs_cluster4_ctas, &zero, sizeof(zero)) != cudaSuccess)
    return -1;
  return static_cast<long long>(n);
}

template <bool FILT>
static int launch_qs_filt(const ScoreArgs& a, const PassPlan& plan, const TopkWorkspace& ws, cudaStream_t st) {
  const bool sp = a.sparse != nullptr;
  if (plan.lists == 2 * plan.workers)               // two epilogue sets (CTA pairs only)
    return sp ? launch_qs_impl<2, 2, true, FILT>(a, plan, ws, st) : launch_qs_impl<2, 2, false, FILT>(a, plan, ws, st);
  if (plan.cg == 2)
    return sp ? launch_qs_impl<2, 1, true, FILT>(a, plan, ws, st) : launch_qs_impl<2, 1, false, FILT>(a, plan, ws, st);
  return sp ? launch_qs_impl<1, 1, true, FILT>(a, plan, ws, st) : launch_qs_impl<1, 1, false, FILT>(a, plan, ws, st);
}

int launch_score_qs(const ScoreArgs& a, const PassPlan& plan, const TopkWorkspace& ws, cudaStream_t st,
                    int* launches) {
  const int rc = a.filter_bits ? launch_qs_filt<true>(a, plan, ws, st) : launch_qs_filt<false>(a, plan, ws, st);
  if (rc == MFAR_OK) ++*launches;
  return rc;
}

}  // namespace mfar
