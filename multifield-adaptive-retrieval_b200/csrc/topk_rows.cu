// Streaming top-k over pre-mixed score rows: the sparse-only scorers (all_sparse / single_sparse field sets, and
// bm25s-style retrieve over one field) have no dense contraction - their score[q, n] is the fp32 base[Q, N] block
// the sparse pre-mix / BM25 scatter kernels produce - so the whole scoring pass is "top-k of every row".
// Replaces torch.topk over the full score matrix (mfar/modeling/contrastive.py:696) / bm25s' argpartition
// (mfar/data/index.py:92,99) for that case.  HBM-bound: Q*N*4 bytes read once.
//
// One WARP per (row segment, query): it streams its segment with 16-byte loads, 512 docs (4 x float4 per lane) in
// flight per step, filters against its threshold in registers, appends survivors to its candidate list with
// ballot/popc slots (no shared memory, no atomics, no block barriers) and compacts the list with the warp select of
// common.cuh when it could overflow.  Lists land in the same workspace layout as the scoring kernels'
// ([segment][query][kCandCap]), so the same merge kernel finishes.  Segments of one query share their thresholds
// through gthr[q] like the CTAs of the tensor-core kernels.
#include "common.cuh"
#include "kernels.h"

namespace mfar {

constexpr int kRowsWarps = 8;
constexpr int kRowsStepDocs = 512;     // docs per warp step: 4 float4 per lane

// Threshold seed.  Every segment warp of a query starts at the same time with no threshold, so without help each
// admits its first ~200 docs and needs several compactions before the shared gthr[q] gets tight (measured: 160 us for
// 245 MB at Q=64).  One CTA per query scans a prefix of the row as 8192 disjoint 4-doc subsets, keeps each subset's
// maximum and finds the k-th largest of those maxima by a block binary search on the 32-bit score word: every
// maximum is a real doc, so at least k docs of the row score >= it - a valid admission bound, close to the exact
// k-th best of the prefix - and the segment warps start from it.
constexpr int kSeedThreads = 256;
constexpr int kSeedPerThread = 32;     // float4 subsets per thread: prefix = 256 * 32 * 4 = 32768 docs

// FILT: ineligible docs count as absent (-inf) in their subset's maximum, so every maximum above -inf is still an
// eligible doc and the bound stays one that k eligible docs reach.
template <bool FILT>
__global__ void __launch_bounds__(kSeedThreads)
topk_rows_seed_kernel(const float* __restrict__ base, long long base_ld, long long n_docs, int k,
                      unsigned long long* __restrict__ gthr, long long doc_id_base, DocFilter filt) {
  __shared__ int part[kSeedThreads / 32];
  __shared__ int total_s;
  const int q = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const float* row = base + (long long)q * base_ld;
  const uint32_t* frow = FILT ? filt.bits + (long long)q * filt.stride : nullptr;
  uint32_t hi[kSeedPerThread];
  const long long last_vec = ((n_docs - 1) / 4) * 4;       // base_ld is a multiple of 128: this 16-byte read is in bounds
#pragma unroll
  for (int i0 = 0; i0 < kSeedPerThread; i0 += 8) {         // 8 unconditional loads in flight, then the masking
    float4 v[8];
    uint32_t fb[8];                                        // FILT: eligibility of the subset's 4 docs (bits 0..3)
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const long long d = ((long long)(i0 + j) * kSeedThreads + tid) * 4;
      v[j] = __ldg(reinterpret_cast<const float4*>(row + (d < n_docs ? d : last_vec)));
      fb[j] = FILT ? filter_bits32(frow, filt.words, doc_id_base + d) : 0xFu;
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const long long d = ((long long)(i0 + j) * kSeedThreads + tid) * 4;
      float m = d < n_docs && (fb[j] & 1u) ? v[j].x : -INFINITY;
      m = d + 1 < n_docs && (fb[j] & 2u) ? fmaxf(m, v[j].y) : m;
      m = d + 2 < n_docs && (fb[j] & 4u) ? fmaxf(m, v[j].z) : m;
      m = d + 3 < n_docs && (fb[j] & 8u) ? fmaxf(m, v[j].w) : m;
      hi[i0 + j] = float_to_ordered(m);
    }
  }
  uint32_t lo = 0u, up = 0xFFFFFFFFu;                     // largest T with count(hi >= T) >= k
  while (lo < up) {
    const uint32_t mid = lo + ((up - lo) >> 1) + 1u;
    int c = 0;
#pragma unroll
    for (int i = 0; i < kSeedPerThread; ++i) c += (hi[i] >= mid) ? 1 : 0;
    c = __reduce_add_sync(0xffffffffu, c);
    if (lane == 0) part[wid] = c;
    __syncthreads();
    if (tid == 0) {
      int t = 0;
#pragma unroll
      for (int w = 0; w < kSeedThreads / 32; ++w) t += part[w];
      total_s = t;
    }
    __syncthreads();
    if (total_s >= k) lo = mid; else up = mid - 1u;
  }
  // subsets without docs carry -inf: if fewer than k subsets are real, T lands at or below -inf's word and admits all
  if (tid == 0 && lo > float_to_ordered(-INFINITY)) atomicMax(gthr + q, ((unsigned long long)lo << 32) - 1ull);
}

__device__ __forceinline__ void rows_load_step(const float* __restrict__ row, long long s0, long long d1, int lane,
                                               float4 (&v)[4]) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {                            // seg_docs, base_ld are multiples of 4: aligned, in bounds
    const long long d = s0 + j * 128 + lane * 4;
    v[j] = d < d1 ? __ldcs(reinterpret_cast<const float4*>(row + d)) : make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
  }
}

// FILT: a doc whose bit is clear is never pushed; its bits are read on the rare path, after the sub-step's ballot.
template <bool FILT>
__global__ void __launch_bounds__(kRowsWarps * 32, 3)
topk_rows_kernel(const float* __restrict__ base, long long base_ld, long long n_docs, int Q, int segments,
                 long long seg_docs, long long doc_id_base, int k, TopkWorkspace ws, DocFilter filt) {
  const int lane = threadIdx.x & 31;
  const long long task = (long long)blockIdx.x * kRowsWarps + (threadIdx.x >> 5);   // = seg * Q + q (q fastest)
  if (task >= (long long)segments * Q) return;
  const int seg = int(task / Q), q = int(task - (long long)seg * Q);
  const long long d0 = seg * seg_docs, d1 = min(n_docs, d0 + seg_docs);
  const float* row = base + (long long)q * base_ld;
  const uint32_t* frow = FILT ? filt.bits + (long long)q * filt.stride : nullptr;
  uint64_t* list = ws.cand_keys + ((long long)seg * ws.q_pad + q) * kCandCap;
  unsigned long long thr = 0ull;
  float thr_f = -INFINITY;
  int cnt = 0;
  const unsigned lt_mask = (1u << lane) - 1u;
  float4 cur[4], nxt[4];
  rows_load_step(row, d0, d1, lane, cur);
  for (long long s0 = d0; s0 < d1; s0 += kRowsStepDocs) {
    rows_load_step(row, s0 + kRowsStepDocs, d1, lane, nxt);          // next step's loads fly while this one is filtered
    {                                                      // best bound any segment of this query has published
      const unsigned long long gt = ws_ld_relaxed_u64(ws.gthr + q);
      if (gt > thr) { thr = gt; thr_f = key_score(gt); }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      // one compare per lane (max of its 4 docs) and one ballot reject the 128 docs of this sub-step in the common case
      // NaN-propagating max and !(x < thr_f): NaN scores (NaN > +inf in the key order) reach the key compare
      const float m = fmax_nan(fmax_nan(cur[j].x, cur[j].y), fmax_nan(cur[j].z, cur[j].w));
      if (__ballot_sync(0xffffffffu, !(m < thr_f)) == 0u) continue;
      const long long d = s0 + j * 128 + lane * 4;
      const float x[4] = {cur[j].x, cur[j].y, cur[j].z, cur[j].w};
      const uint32_t fb = FILT ? filter_bits32(frow, filt.words, doc_id_base + d) : 0xFu;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const unsigned long long key = make_key(x[e], uint32_t(doc_id_base + d + e));
        const bool pass = (d + e < d1) && !(x[e] < thr_f) && key > thr && ((fb >> e) & 1u);
        const unsigned b = __ballot_sync(0xffffffffu, pass);
        if (b) {
          if (pass) __stcg(list + cnt + __popc(b & lt_mask), key);
          cnt += __popc(b);
        }
      }
      if (cnt > kCandCap - 128) {                          // the next 128 docs could overflow the list
        __syncwarp();
        int cnt_new = k;
        uint64_t bound_r = 0ull;
        const uint64_t kth = warp_select_list(list, cnt, k, kCandCap - 128, lane, &cnt_new, 1, &bound_r);
        __syncwarp();
        cnt = cnt_new;
        if (kth > thr) { thr = kth; thr_f = key_score(kth); }
        if (lane == 0) atomicMax(ws.gthr + q, thr);
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) cur[j] = nxt[j];
  }
  if (lane == 0) {
    ws.cand_cnt[(long long)seg * ws.q_pad + q] = cnt;
    ws.cand_thr[(long long)seg * ws.q_pad + q] = thr;
  }
}

// segments per row: enough warps to fill the machine (148 SMs x 64 warps), at least 2048 docs each
PassPlan plan_topk_rows(int Q, long long n_docs) {
  long long want = (long long)kNumSmsB200 * 64 / (Q > 0 ? Q : 1);
  if (want < 1) want = 1;
  long long cap = (n_docs + 2047) / 2048;
  if (cap < 1) cap = 1;
  long long s = want < cap ? want : cap;
  if (s > 1024) s = 1024;
  long long per = (n_docs + s - 1) / s;
  per = (per + kRowsStepDocs - 1) / kRowsStepDocs * kRowsStepDocs;     // whole steps: 16-byte aligned segment starts
  s = (n_docs + per - 1) / per;
  PassPlan p{};
  p.impl = kImplRows;
  p.workers = p.lists = int(s < 1 ? 1 : s);
  p.seg_docs = per;
  p.q_tiles = p.cg = 1;
  p.q_pad = p.q_pad_total = round_up(Q, 4);
  return p;
}

int launch_topk_rows(const ScoreArgs& a, const PassPlan& plan, const TopkWorkspace& ws, cudaStream_t st,
                     int* launches) {
  if (!a.base || a.base_ld % 4 != 0 || reinterpret_cast<uintptr_t>(a.base) % 16 != 0) return MFAR_ERR_ARG;
  const DocFilter filt{a.filter_bits, a.filter_stride, a.filter_words};
  const bool f = filt.bits != nullptr;
  const bool seeded = a.n_docs >= 4096;                    // tiny shards: a few steps per warp, nothing to seed
  if (seeded) {
    auto seed = f ? topk_rows_seed_kernel<true> : topk_rows_seed_kernel<false>;
    seed<<<a.Q, kSeedThreads, 0, st>>>(a.base, a.base_ld, a.n_docs, a.k, ws.gthr, a.doc_id_base, filt);
  }
  const long long tasks = (long long)plan.workers * a.Q;
  const unsigned blocks = unsigned((tasks + kRowsWarps - 1) / kRowsWarps);
  auto rows = f ? topk_rows_kernel<true> : topk_rows_kernel<false>;
  rows<<<blocks, kRowsWarps * 32, 0, st>>>(a.base, a.base_ld, a.n_docs, a.Q, plan.workers, plan.seg_docs,
                                           a.doc_id_base, a.k, ws, filt);
  MFAR_CUDA_OK(cudaGetLastError());
  *launches += seeded ? 2 : 1;
  return MFAR_OK;
}

}  // namespace mfar
