// Shared device/host helpers for the mFAR B200 scoring path.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/mfar_b200.h"

namespace mfar {

constexpr int kTileDocs = MFAR_TILE_DOCS;  // docs per corpus tile == UMMA M
constexpr int kMaxK = MFAR_MAX_K;
constexpr int kCandCap = 256;              // per-(worker, query) candidate slots; >= kMaxK + kTileDocs
constexpr int kNumSmsB200 = 148;
constexpr int kProgressInts = 1024;        // cross-CTA progress counters (score_qs lockstep), one per (worker, query group)

__host__ __device__ inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

#define MFAR_CUDA_OK(expr)                                                                   \
  do {                                                                                       \
    cudaError_t _e = (expr);                                                                 \
    if (_e != cudaSuccess) {                                                                 \
      fprintf(stderr, "[mfar_b200] %s failed: %s (%s:%d)\n", #expr, cudaGetErrorString(_e),  \
              __FILE__, __LINE__);                                                           \
      return MFAR_ERR_CUDA;                                                                  \
    }                                                                                        \
  } while (0)

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is per (function, device): remembered per device so that a process
// driving several GPUs raises the limit on each of them.  `done` is a static per call site / template instantiation.
struct PerDeviceOnce {
  bool done[64] = {};
  template <class Fn>
  cudaError_t run(Fn&& fn) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev >= 0 && dev < 64 && done[dev]) return cudaSuccess;
    e = fn();
    if (e == cudaSuccess && dev >= 0 && dev < 64) done[dev] = true;
    return e;
  }
};

// ---------------------------------------------------------------------------------------
// (score, doc id) <-> order-preserving 64-bit key.
//   high 32 bits: float score mapped so that unsigned order == float order
//   low  32 bits: ~doc_id, so that among equal scores the LOWER doc id is the LARGER key
// max-key-first order therefore is (score desc, doc id asc): the deterministic tie-break the
// oracle's topk_sorted() uses.  Every NaN, whatever its sign or payload, maps to ONE word above +inf's
// (kNanOrdered, the word of the canonical +NaN 0x7FC00000), so the full order is
//   NaN > +inf > finite scores (desc) > -inf, then doc id asc inside each class
// - torch.topk's order (NaN counts as the largest value), which the reference ranks with (contrastive.py:696).
// A NaN doc reports the canonical NaN.  (-0.0 would rank just below +0.0, but every score is a sum started at +0.0,
// which never yields -0.0.)  Key 0 is never produced by any score: it marks "empty".
// ---------------------------------------------------------------------------------------
constexpr uint32_t kNanOrdered = 0xFFC00000u;
__host__ __device__ __forceinline__ uint32_t float_to_ordered(float f) {
#ifdef __CUDA_ARCH__
  uint32_t u = __float_as_uint(f);
#else
  union { float f; uint32_t u; } c; c.f = f; uint32_t u = c.u;
#endif
  const uint32_t o = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
  return f != f ? kNanOrdered : o;
}
__host__ __device__ __forceinline__ float ordered_to_float(uint32_t o) {
  uint32_t u = (o & 0x80000000u) ? (o & 0x7FFFFFFFu) : ~o;
#ifdef __CUDA_ARCH__
  return __uint_as_float(u);
#else
  union { float f; uint32_t u; } c; c.u = u; return c.f;
#endif
}
__host__ __device__ __forceinline__ uint64_t make_key(float score, uint32_t doc_id) {
  return (uint64_t(float_to_ordered(score)) << 32) | uint64_t(~doc_id);
}
__host__ __device__ __forceinline__ float key_score(uint64_t key) { return ordered_to_float(uint32_t(key >> 32)); }
__host__ __device__ __forceinline__ uint32_t key_doc(uint64_t key) { return ~uint32_t(key & 0xFFFFFFFFull); }

// max that PROPAGATES NaN (fmaxf drops it).  The float pre-filters of the scoring kernels take a group maximum and
// test it with !(m < thr): a NaN anywhere in the group (a NaN score, or -inf - -inf, +inf - +inf in score_tc's
// differences) then passes to the exact key compare instead of being rejected - the filters stay conservative.
__device__ __forceinline__ float fmax_nan(float a, float b) {
  float d;
  asm("max.NaN.f32 %0, %1, %2;" : "=f"(d) : "f"(a), "f"(b));
  return d;
}

// Doc filter of the *_filtered entry points (DESIGN §4.5): a uint32 bitmap over GLOBAL doc ids, bit d of word d >> 5
// set <=> doc d may enter the top-k.  One row shared by every query (stride 0) or one row of `ld` words per query
// (stride == ld).  Only the first `words` = ceil((doc_id_base + n_docs) / 32) words of a row hold docs of the shard
// (<= 2^27, and <= ld): a word index past them reads as 0, so tile tails never read past the row.
struct DocFilter {
  const uint32_t* bits;   // nullptr: no filter
  long long stride;       // words between the rows of consecutive queries: 0 (one shared row) or ld
  int words;              // words of a row that are read
};
__device__ __forceinline__ uint32_t filter_ld_word(const uint32_t* row, int words, long long w) {
  return w < words ? __ldg(row + w) : 0u;
}
// bits [b, b + 32) of a row: bit j of the result is the eligibility of global doc b + j (funnel shift across words)
__device__ __forceinline__ uint32_t filter_bits32(const uint32_t* row, int words, long long b) {
  const long long w = b >> 5;
  const uint32_t lo = filter_ld_word(row, words, w), hi = filter_ld_word(row, words, w + 1);
  return __funnelshift_r(lo, hi, uint32_t(b & 31));
}

// Workspace carve-up shared by the scoring kernels and the merge.
//   cand_keys [G][Qp][kCandCap] u64 | cand_thr [G][Qp] u64 | cand_cnt [G][Qp] i32 | err flag (256 B) |
//   progress counters (kProgressInts i32) | gthr [Qp] u64 | pool [G][Qp] u64
//   (the tail from the progress counters on is zeroed before every scoring pass that reads it)
// gthr[q] = best admission threshold any CTA has established for query q (atomicMax of a k-th key).  The k-th key
// of ANY subset of the shard is a lower bound of the shard's k-th key, so every CTA may filter with it: the
// admitted-candidate count (and with it the list compactions) drops from k*ln(N_cta/k) per CTA to ~that in total.
struct TopkWorkspace {
  uint64_t* cand_keys;
  int* cand_cnt;
  uint64_t* cand_thr;
  int* err;
  int* progress;
  unsigned long long* gthr;
  unsigned long long* pool;    // [G][Qp]: latest rank-r key bound of each CTA's list, r = ceil(k / G) (0 = none yet)
  int workers;  // G
  int q_pad;    // Qp
};


inline size_t topk_workspace_bytes(int workers, int q_pad) {
  size_t n = size_t(workers) * q_pad;
  return n * kCandCap * 8 + n * 8 + round_up(int(n * 4), 256) + 256 + kProgressInts * 4 + size_t(q_pad) * 8 + n * 8;
}
// bytes of the zero-initialised tail (progress + gthr + pool), starting at TopkWorkspace::progress
inline size_t workspace_zero_bytes(int workers, int q_pad) {
  return size_t(kProgressInts) * 4 + size_t(q_pad) * 8 + size_t(workers) * q_pad * 8;
}
inline TopkWorkspace carve_workspace(void* base, int workers, int q_pad) {
  TopkWorkspace w;
  size_t n = size_t(workers) * q_pad;
  char* p = static_cast<char*>(base);
  w.cand_keys = reinterpret_cast<uint64_t*>(p); p += n * kCandCap * 8;
  w.cand_thr = reinterpret_cast<uint64_t*>(p);  p += n * 8;
  w.cand_cnt = reinterpret_cast<int*>(p);       p += round_up(int(n * 4), 256);
  w.err = reinterpret_cast<int*>(p);            p += 256;
  w.progress = reinterpret_cast<int*>(p);       p += kProgressInts * 4;
  w.gthr = reinterpret_cast<unsigned long long*>(p);   p += size_t(q_pad) * 8;
  w.pool = reinterpret_cast<unsigned long long*>(p);
  w.workers = workers;
  w.q_pad = q_pad;
  return w;
}

// --------------------------------------------------------------------------------------
// Warp-level bitonic sort, descending, of 256 u64 keys held 8 per lane (element e = lane*8+j).
// Compare distances 1,2,4 stay inside a lane; 8..128 are one 64-bit shuffle each.
// --------------------------------------------------------------------------------------
__device__ __forceinline__ void warp_sort256_desc(uint64_t (&v)[8], int lane) {
#pragma unroll
  for (int s = 2; s <= 256; s <<= 1) {
#pragma unroll
    for (int d = s >> 1; d > 0; d >>= 1) {
      if (d >= 8) {
        const int lane_d = d >> 3;
        const bool upper = (lane & lane_d) != 0;              // this lane holds the higher index of the pair
        const bool desc = ((lane * 8) & s) == 0 || s == 256;  // block direction (same for all 8 elems: s > 8)
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          uint64_t o = __shfl_xor_sync(0xffffffffu, v[j], lane_d);
          uint64_t mx = v[j] > o ? v[j] : o, mn = v[j] > o ? o : v[j];
          v[j] = (desc != upper) ? mx : mn;                   // lower index keeps max when descending
        }
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          if ((j & d) == 0) {
            const int e = lane * 8 + j;
            const bool desc = ((e & s) == 0) || s == 256;
            uint64_t a = v[j], b = v[j | d];
            uint64_t mx = a > b ? a : b, mn = a > b ? b : a;
            v[j] = desc ? mx : mn;
            v[j | d] = desc ? mn : mx;
          }
        }
      }
    }
  }
}

// Pooled threshold.  If every one of the G CTAs scanning a query's shard holds at least r = ceil(k/G) keys >= x_g,
// then min_g(x_g) has at least G*r >= k keys above it shard-wide: a valid admission threshold that is far tighter
// than any single CTA's own k-th key (it tracks roughly the k-th best of ALL docs scanned so far by all CTAs, not of
// one CTA's slice).  Every CTA re-publishes x_g = a lower bound of the rank-r key of its list at EVERY compaction
// (pool[g][q], single writer, monotone), then takes the min over the G slots and raises the shared gthr[q] with it
// (atomicMax of valid bounds stays a valid bound).  Readers keep reading just gthr[q].
__host__ __device__ inline int pooled_rank(int k, int G) {
#ifdef MFAR_FAULT_POOLED   // fault injection, never defined in the shipped build (profiles/r2_fault_injection.md): rank r-1
  const int r = (k + G - 1) / G;   // makes G*r < k, so the pooled bound can exceed the shard's true k-th key
  return r > 1 ? r - 1 : 1;
#else
  return (k + G - 1) / G;
#endif
}

__device__ __forceinline__ unsigned long long ws_ld_relaxed_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

// Whole warp: publish this CTA's bound for query q and return min over all G CTAs' bounds (0 while any is missing).
__device__ __forceinline__ unsigned long long pool_publish_and_min(unsigned long long* pool, int G, int q_pad, int g,
                                                                   int q, unsigned long long mine, int lane) {
  if (lane == 0) asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" :: "l"(pool + (long long)g * q_pad + q), "l"(mine) : "memory");
  unsigned long long m = mine;
  for (int gg = lane; gg < G; gg += 32) {
    if (gg != g) {
      const unsigned long long v = ws_ld_relaxed_u64(pool + (long long)gg * q_pad + q);
#ifdef MFAR_FAULT_POOLED   // fault injection (never defined in the shipped build): CTAs that have not published
      if (v == 0ull) continue;  // yet are skipped, so the "G*r >= k keys above the bound" argument no longer holds -
#endif                          // tests/test_gpu_parity_at_scale.py must FAIL against such a library (profiles/r2_fault_injection.md)
      m = v < m ? v : m;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long v = __shfl_xor_sync(0xffffffffu, m, o);
    m = v < m ? v : m;
  }
  return m;
}

// One warp compacts the candidate list of one (worker, query): keep the best k keys (sorted
// descending), return the k-th key (new admission threshold).  `list` points at kCandCap slots
// in global memory written earlier by threads of this CTA (made visible by a CTA barrier).
__device__ __forceinline__ uint64_t warp_compact_list(uint64_t* list, int count, int k, int lane) {
  uint64_t v[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    int e = lane * 8 + j;
    v[j] = (e < count) ? __ldcg(list + e) : 0ull;
  }
  warp_sort256_desc(v, lane);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    int e = lane * 8 + j;
    if (e < k) __stcg(list + e, v[j]);
  }
  // k-th key lives in lane (k-1)/8, register (k-1)%8
  uint64_t kth = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j)
    if (((k - 1) & 7) == j) kth = v[j];
  return __shfl_sync(0xffffffffu, kth, (k - 1) >> 3);
}

// Compaction by SELECTION instead of sorting: search the 32-bit score word for the largest T with
// count(score >= T) >= k, stop as soon as k <= count <= k + kSelectSlack, and keep exactly those keys (ballot-compacted,
// unsorted).  The search is 4-ary: three thresholds per round, their three warp-wide counts packed into ONE REDUX
// (10 bits each: a list holds at most 256 keys), so a round costs 24 compares + 1 REDUX and the range shrinks 4x -
// about half the dependent REDUX round trips of the bisection round 1 used (a compaction was ~9.4k cycles, of which
// the two searches ~2.5k).  Returns the admission threshold "(T << 32) - 1" (key > thr  <=>  score word >= T) and the
// new count through *new_count; the same search continued upwards for rank r <= k gives the pooled bound.  Falls back
// to the exact sort when score ties keep too many keys.
constexpr int kSelectSlack = 24;

__device__ __forceinline__ void warp_list_load(const uint64_t* list, int count, int lane, uint64_t (&v)[8]) {
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int e = lane * 8 + j;
    v[j] = (e < count) ? __ldcg(list + e) : 0ull;
  }
}

// largest T in [lo, up] with count(hi >= T) >= rank, given count(hi >= lo) >= rank; stops early once the count at the
// running lower end is <= rank + slack (slack < 0: run to the exact answer).  *c_lo_io: count(hi >= lo) in / out.
__device__ __forceinline__ uint32_t warp_rank_search(const uint32_t (&hi)[8], uint32_t lo, uint32_t up, int rank, int slack,
                                                     int* c_lo_io) {
  int c_lo = *c_lo_io;
  while (lo < up && (slack < 0 || c_lo > rank + slack)) {
    const uint32_t span = up - lo;                      // >= 1
    const uint32_t m2 = lo + (span >> 1) + (span & 1u); // lo < m2 <= up
    const uint32_t m1 = lo + ((m2 - lo) >> 1) + ((m2 - lo) & 1u);                 // lo < m1 <= m2
    const uint32_t m3 = m2 + ((up - m2) >> 1) + ((up - m2) & 1u);                 // m2 <= m3 <= up
    uint32_t c = 0u;
#pragma unroll
    for (int j = 0; j < 8; ++j)
      c += (hi[j] >= m1 ? 1u : 0u) + (hi[j] >= m2 ? 1u << 10 : 0u) + (hi[j] >= m3 ? 1u << 20 : 0u);
    c = __reduce_add_sync(0xffffffffu, c);
    const int c1 = int(c & 1023u), c2 = int((c >> 10) & 1023u), c3 = int(c >> 20);
    if (c3 >= rank) { lo = m3; c_lo = c3; }
    else if (c2 >= rank) { lo = m2; c_lo = c2; up = m3 - 1u; }
    else if (c1 >= rank) { lo = m1; c_lo = c1; up = m2 - 1u; }
    else { up = m1 - 1u; }
  }
  *c_lo_io = c_lo;
  return lo;
}

// v: the list's keys, 8 per lane (warp_list_load).  max_keep: the list may hold at most this many keys afterwards.
__device__ __forceinline__ uint64_t warp_select_keys(const uint64_t (&v)[8], uint64_t* list, int count, int k, int max_keep,
                                                     int lane, int* new_count, int r, uint64_t* rank_r_bound) {
  const int slack = min(kSelectSlack, max_keep - k);
  uint32_t hi[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) hi[j] = uint32_t(v[j] >> 32);       // 0 for empty slots: below every real score word
  uint32_t mx = 0u, mn = 0xFFFFFFFFu;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    mx = max(mx, hi[j]);
    if (v[j] != 0ull) mn = min(mn, hi[j]);
  }
  mx = __reduce_max_sync(0xffffffffu, mx);
  mn = __reduce_min_sync(0xffffffffu, mn);
  int c_lo = count;                                     // invariant: count(>= lo) = c_lo >= k; answer in [lo, up]
  const uint32_t lo = warp_rank_search(hi, mn, mx, k, slack, &c_lo);
  if (c_lo > k + slack) {                               // a big tie group straddles rank k (or no slack): exact path
    *new_count = k;
    uint64_t w[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) w[j] = v[j];
    warp_sort256_desc(w, lane);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int e = lane * 8 + j;
      if (e < k) __stcg(list + e, w[j]);
    }
    uint64_t kth = 0, rth = 0;                          // rank x lives in lane (x-1)/8, register (x-1)%8
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (((k - 1) & 7) == j) kth = w[j];
      if (((r - 1) & 7) == j) rth = w[j];
    }
    *rank_r_bound = __shfl_sync(0xffffffffu, rth, (r - 1) >> 3);
    return __shfl_sync(0xffffffffu, kth, (k - 1) >> 3);
  }
  {                                                     // same search for rank r <= k on [lo, mx], to the exact word
    int c2 = c_lo;
    const uint32_t lo2 = warp_rank_search(hi, lo, mx, r, -1, &c2);
    *rank_r_bound = (uint64_t(lo2) << 32) - 1ull;       // >= r keys have score word >= lo2, i.e. key > this bound
  }
  int base = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const bool keep = hi[j] >= lo && v[j] != 0ull;
    const unsigned b = __ballot_sync(0xffffffffu, keep);
    if (keep) __stcg(list + base + __popc(b & ((1u << lane) - 1u)), v[j]);
    base += __popc(b);
  }
  *new_count = base;
  return (uint64_t(lo) << 32) - 1ull;
}

__device__ __forceinline__ uint64_t warp_select_list(uint64_t* list, int count, int k, int max_keep, int lane,
                                                     int* new_count, int r, uint64_t* rank_r_bound) {
  uint64_t v[8];
  warp_list_load(list, count, lane, v);
  return warp_select_keys(v, list, count, k, max_keep, lane, new_count, r, rank_r_bound);
}

// Pooled bounds, split so that the loads of the other CTAs' slots can be issued BEFORE the select of the list at hand
// (their L2 round trip then hides behind the search): pool_load_others, later pool_publish_min.  Reading the others'
// bounds a little early is harmless - every slot only ever grows, an older value is a weaker but still valid bound.
constexpr int kPoolPerLane = 5;                         // up to 160 lists per query (148 CTAs, or 74 pairs x 2 sets)

__device__ __forceinline__ void pool_load_others(const unsigned long long* pool, int G, int q_pad, int g, int q, int lane,
                                                 unsigned long long (&pl)[kPoolPerLane]) {
#pragma unroll
  for (int i = 0; i < kPoolPerLane; ++i) {
    const int gg = lane + 32 * i;
    pl[i] = (gg < G && gg != g) ? ws_ld_relaxed_u64(pool + (long long)gg * q_pad + q) : ~0ull;
  }
}

__device__ __forceinline__ unsigned long long pool_publish_min(unsigned long long* pool, int G, int q_pad, int g, int q,
                                                               unsigned long long mine, int lane,
                                                               const unsigned long long (&pl)[kPoolPerLane]) {
  if (G > 32 * kPoolPerLane) return pool_publish_and_min(pool, G, q_pad, g, q, mine, lane);   // not prefetched
  if (lane == 0) asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" :: "l"(pool + (long long)g * q_pad + q), "l"(mine) : "memory");
  unsigned long long m = mine;
#pragma unroll
  for (int i = 0; i < kPoolPerLane; ++i) {
#ifdef MFAR_FAULT_POOLED
    if (pl[i] == 0ull) continue;
#endif
    m = pl[i] < m ? pl[i] : m;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long v = __shfl_xor_sync(0xffffffffu, m, o);
    m = v < m ? v : m;
  }
  return m;
}

// Two E4M3 bytes (the low byte is element 0) -> fp32.  Every E4M3 value is exact in f16, so the one conversion
// instruction (cvt.rn.f16x2.e4m3x2) and the widening are exact.
__device__ __forceinline__ float2 e4m3x2_to_float2(uint32_t two_bytes) {
  uint32_t h;
  asm("cvt.rn.f16x2.e4m3x2 %0, %1;" : "=r"(h) : "h"(uint16_t(two_bytes)));
  return __half22float2(*reinterpret_cast<const __half2*>(&h));
}
// 8 E4M3 bytes -> 8 fp32
__device__ __forceinline__ void e4m3x8_to_f32(const uint2& v, float (&f)[8]) {
  float2 a = e4m3x2_to_float2(v.x), b = e4m3x2_to_float2(v.x >> 16), c = e4m3x2_to_float2(v.y),
         d = e4m3x2_to_float2(v.y >> 16);
  f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y; f[4] = c.x; f[5] = c.y; f[6] = d.x; f[7] = d.y;
}

}  // namespace mfar
