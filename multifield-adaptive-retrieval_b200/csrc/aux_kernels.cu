// Corpus pack/unpack, field-mixture weights, candidate re-scoring, sparse pre-mix and the
// top-k merge.  All small / bandwidth-trivial next to the scoring pass; plain CUDA-core code.
#include <algorithm>

#include "common.cuh"
#include "kernels.h"

namespace mfar {

// ---------------------------------------------------------------------------------------
// pack: one warp per source row.  row-major [n_rows, dim] fp32|bf16 -> packed bf16
// [tile][field][128][dim].  Optional L2 normalisation x / max(||x||_2, 1e-12), what
// sentence-transformers' Normalize() applies (reference: mfar/modeling/util.py:50-51), computed
// in fp64 and rounded ONCE to bf16: the squares of fp32 values are exact in fp64, the sum cannot
// overflow (a row of |x| ~ 1e19 packs as itself over its norm, not as zeros), and the quotient
// goes straight to nearest-even bf16.  Queries go through the same kernel (prepare_queries).
// ---------------------------------------------------------------------------------------
template <typename SrcT>
__global__ void pack_rows_kernel(const SrcT* __restrict__ src, int64_t n_rows, int64_t row_begin,
                                 __nv_bfloat16* __restrict__ packed, int n_fields, int field, int dim,
                                 int normalize) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  if (r >= n_rows) return;
  const SrcT* s = src + r * dim;
  const int64_t doc = row_begin + r;
  const int64_t tile = doc / kTileDocs;
  const int in_tile = int(doc % kTileDocs);
  __nv_bfloat16* d = packed + ((tile * n_fields + field) * kTileDocs + in_tile) * int64_t(dim);
  if (!normalize) {
    for (int i = lane; i < dim; i += 32) d[i] = __float2bfloat16_rn(float(s[i]));
    return;
  }
  double ss = 0.0;
  for (int i = lane; i < dim; i += 32) {
    const double v = double(float(s[i]));
    ss = fma(v, v, ss);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  const double norm = fmax(sqrt(ss), double(1e-12f));   // F.normalize's eps on an fp32 tensor
  for (int i = lane; i < dim; i += 32) d[i] = __double2bfloat16(double(float(s[i])) / norm);
}

__global__ void unpack_rows_kernel(const __nv_bfloat16* __restrict__ packed, int n_fields, int field, int dim,
                                   int64_t row_begin, int64_t n_rows, float* __restrict__ dst) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  if (r >= n_rows) return;
  const int64_t doc = row_begin + r;
  const __nv_bfloat16* s =
      packed + (((doc / kTileDocs) * n_fields + field) * kTileDocs + (doc % kTileDocs)) * int64_t(dim);
  for (int i = lane; i < dim; i += 32) dst[r * dim + i] = __bfloat162float(s[i]);
}

// ---------------------------------------------------------------------------------------
// E4M3 pack: one warp per source row -> payload bytes [tile][field][128][dim] + one fp32 scale per row
// [tile][field][128].  The row (after the optional float64 normalisation above) gets s = 2^e,
// e = clamp(ceil(log2(amax / 448)), -117, 119): the lower bound keeps the smallest E4M3 subnormal times s at 2^-126 (a
// normal fp32 / bf16 number), the upper bound keeps 448 * s finite in bf16.  Each element is rounded ONCE, from
// float64, to the nearest E4M3 value of x / s (ties to even, saturating to +-448 - reached only when the clamp at 119
// binds).  Zero rows store s = 1, rows holding a NaN / infinity s = NaN; both store payload 0.
// ---------------------------------------------------------------------------------------
constexpr int kE4m3MinScaleExp = -117;
constexpr int kE4m3MaxScaleExp = 119;

// nearest E4M3 value of v (ties to even, saturating at 448), as its byte
__device__ __forceinline__ uint8_t e4m3_rne_byte(double v) {
  const double a = fabs(v);
  int k;
  frexp(a, &k);                                      // a = m 2^k, m in [0.5, 1): 4 significant bits -> spacing 2^(k-4)
  const int q = max(k - 4, -9);                      // -9: the subnormal spacing
  double r = ldexp(rint(ldexp(a, -q)), q);           // exact scalings; rint rounds half to even
  if (r > 448.0) r = 448.0;
  uint32_t b;
  if (r < 0.015625) {                                // below 2^-6: subnormal (or zero), mantissa = r * 2^9
    b = uint32_t(r * 512.0);
  } else {
    int k2;
    const double m = frexp(r, &k2);                  // r = (2m) 2^(k2-1), 2m = 1 + mant/8
    b = (uint32_t(k2 + 6) << 3) | uint32_t(m * 16.0 - 8.0);
  }
  return uint8_t(b | (signbit(v) ? 0x80u : 0u));
}

template <typename SrcT>
__global__ void pack_rows_e4m3_kernel(const SrcT* __restrict__ src, int64_t n_rows, int64_t row_begin,
                                      uint8_t* __restrict__ payload, float* __restrict__ scales, int n_fields,
                                      int field, int dim, int normalize) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  if (r >= n_rows) return;
  const SrcT* s = src + r * dim;
  const int64_t doc = row_begin + r;
  const int64_t row = ((doc / kTileDocs) * n_fields + field) * kTileDocs + doc % kTileDocs;
  uint8_t* d = payload + row * int64_t(dim);
  double ss = 0.0, amax = 0.0;
  bool bad = false;
  for (int i = lane; i < dim; i += 32) {
    const double v = double(float(s[i]));
    bad |= !isfinite(v);
    ss = fma(v, v, ss);
    amax = fmax(amax, fabs(v));
  }
  bad = __any_sync(0xffffffffu, bad);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ss += __shfl_xor_sync(0xffffffffu, ss, o);
    amax = fmax(amax, __shfl_xor_sync(0xffffffffu, amax, o));
  }
  // F.normalize's eps on an fp32 tensor; division is exact-rounded, so amax / norm is the largest |quotient|
  const double norm = normalize ? fmax(sqrt(ss), double(1e-12f)) : 1.0;
  if (normalize) amax = amax / norm;
  if (bad || amax == 0.0) {
    for (int i = lane; i < dim; i += 32) d[i] = 0;
    if (lane == 0) scales[row] = bad ? __int_as_float(0x7fc00000) : 1.f;
    return;
  }
  int k;
  const double m = frexp(amax, &k);                  // amax <= 448 2^e  <=>  e >= k - 9 + (m > 0.875)
  const int e = min(max(k - 9 + (m > 0.875 ? 1 : 0), kE4m3MinScaleExp), kE4m3MaxScaleExp);
  for (int i = lane; i < dim; i += 32) {
    double v = double(float(s[i]));
    if (normalize) v = v / norm;
    d[i] = e4m3_rne_byte(ldexp(v, -e));
  }
  if (lane == 0) scales[row] = ldexpf(1.f, e);
}

__device__ __forceinline__ float e4m3_to_float(uint8_t b) { return e4m3x2_to_float2(b).x; }

__global__ void unpack_rows_e4m3_kernel(const uint8_t* __restrict__ payload, const float* __restrict__ scales,
                                        int n_fields, int field, int dim, int64_t row_begin, int64_t n_rows,
                                        float* __restrict__ dst) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  if (r >= n_rows) return;
  const int64_t doc = row_begin + r;
  const int64_t row = ((doc / kTileDocs) * n_fields + field) * kTileDocs + doc % kTileDocs;
  const float sc = scales[row];
  const uint8_t* s = payload + row * int64_t(dim);
  for (int i = lane; i < dim; i += 32) dst[r * dim + i] = e4m3_to_float(s[i]) * sc;
}

// ---------------------------------------------------------------------------------------
// mixture weights: one CTA per query (or one CTA total when !query_cond).
// logits[f] = sum_e q[e] * W[e*F + f];  w = softmax(logits) * mask.   weighting.py:25-28
// ---------------------------------------------------------------------------------------
__global__ void mixture_weights_kernel(const float* __restrict__ q_emb, const float* __restrict__ W,
                                       const float* __restrict__ mask, int E, int F, int query_cond,
                                       float* __restrict__ out_w) {
  __shared__ float s_logit[MFAR_MAX_FIELDS];
  const int q = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
  if (query_cond) {
    const float* qe = q_emb + int64_t(q) * E;
    for (int f = warp; f < F; f += nwarp) {
      float acc = 0.f;
      for (int e = lane; e < E; e += 32) acc = fmaf(qe[e], W[int64_t(e) * F + f], acc);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      if (lane == 0) s_logit[f] = acc;
    }
  } else {
    for (int f = threadIdx.x; f < F; f += blockDim.x) s_logit[f] = W[f];  // W is [F,1]
  }
  __syncthreads();
  if (warp == 0) {
    float m = -INFINITY;
    for (int f = lane; f < F; f += 32) m = fmaxf(m, s_logit[f]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    float s = 0.f;
    for (int f = lane; f < F; f += 32) s += expf(s_logit[f] - m);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    for (int f = lane; f < F; f += 32) {
      float w = expf(s_logit[f] - m) / s;
      out_w[int64_t(q) * F + f] = mask ? w * mask[f] : w;
    }
  }
}

// out[b,s] = sum_f w[b or 0, f] * x[b,s,f]                                weighting.py:29
__global__ void mixture_apply_kernel(const float* __restrict__ x, const float* __restrict__ w, int64_t BS,
                                     int S, int F, int w_rows, float* __restrict__ out) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= BS) return;
  const int b = int(i / S);
  const float* wr = w + (w_rows == 1 ? 0 : int64_t(b) * F);
  const float* xr = x + i * F;
  float acc = 0.f;
  for (int f = 0; f < F; ++f) acc = fmaf(wr[f], xr[f], acc);
  out[i] = acc;
}

// ---------------------------------------------------------------------------------------
// candidate re-scoring: one warp per (candidate, field); loops over queries.
// out[f, q, c] = <q_vec[q], corpus[rows[c], field_begin + f]>;  rows[c] < 0 -> 0
// ---------------------------------------------------------------------------------------
// E4M3 (E8): D of the payload rows, then (D * s_q) * s_d as the scoring kernels apply it.
template <bool E8>
__global__ void score_candidates_kernel(const void* __restrict__ corpus_v, const float* __restrict__ corpus_scales,
                                        int64_t n_docs, int corpus_fields, int field_begin, int n_fields, int dim,
                                        const void* __restrict__ q_vecs_v, const float* __restrict__ q_scales, int Q,
                                        const int64_t* __restrict__ rows, int C, float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t wid = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  if (wid >= int64_t(C) * n_fields) return;
  const int c = int(wid % C), f = int(wid / C);
  const int64_t row = rows[c];
  if (row < 0 || row >= n_docs) {
    for (int q = lane; q < Q; q += 32) out[(int64_t(f) * Q + q) * C + c] = 0.f;
    return;
  }
  const int64_t crow = ((row / kTileDocs) * corpus_fields + field_begin + f) * kTileDocs + (row % kTileDocs);
  if (E8) {
    const uint8_t* v = static_cast<const uint8_t*>(corpus_v) + crow * int64_t(dim);
    const float sd = corpus_scales[crow];
    for (int q = 0; q < Q; ++q) {
      const uint8_t* qv = static_cast<const uint8_t*>(q_vecs_v) + int64_t(q) * dim;
      float acc = 0.f;
      for (int i = lane; i < dim; i += 32) acc = fmaf(e4m3_to_float(qv[i]), e4m3_to_float(v[i]), acc);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      if (lane == 0) out[(int64_t(f) * Q + q) * C + c] = (acc * q_scales[q]) * sd;
    }
    return;
  }
  const __nv_bfloat16* v = static_cast<const __nv_bfloat16*>(corpus_v) + crow * int64_t(dim);
  for (int q = 0; q < Q; ++q) {
    const __nv_bfloat16* qv = static_cast<const __nv_bfloat16*>(q_vecs_v) + int64_t(q) * dim;
    float acc = 0.f;
    for (int i = lane; i < dim; i += 32) acc = fmaf(__bfloat162float(qv[i]), __bfloat162float(v[i]), acc);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) out[(int64_t(f) * Q + q) * C + c] = acc;
  }
}

// ---------------------------------------------------------------------------------------
// sparse pre-mix: base[q, n] = sum_j w[q, n_dense + j] * sparse[q, j, n]   (fp32)
// Coalesced along n; 2 (f16) or 1 (f32) elements... kept simple: one thread per (q, 2 docs).
// The scoring epilogue then gathers ONE value per (query, doc) instead of n_sparse.
// ---------------------------------------------------------------------------------------
template <typename ST>
__global__ void sparse_premix_kernel(const ST* __restrict__ sparse, int64_t sparse_ld, int n_sparse,
                                     const float* __restrict__ w, int w_ld, int w_off, int64_t n_docs,
                                     float* __restrict__ base, int64_t base_ld) {
  const int q = blockIdx.y;
  const int64_t n = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (n >= n_docs) return;
  const float* wq = w + int64_t(q) * w_ld + w_off;
  const ST* sp = sparse + int64_t(q) * n_sparse * sparse_ld + n;
  float acc = 0.f;
#pragma unroll 4
  for (int j = 0; j < n_sparse; ++j) acc = fmaf(wq[j], float(sp[int64_t(j) * sparse_ld]), acc);
  base[int64_t(q) * base_ld + n] = acc;
}

// COO variant (the reference's precomputed-BM25 file format, precompute_bm25s_scores.py:21-30: int32 (query, doc)
// pairs + one value per pair, one segment per sparse field): base[q, doc - doc_id_base] += w[q, F_d + j] * val.
// base is zeroed by the launcher; atomics only collide between different fields of the same (query, doc).
struct CooFieldOffsets { long long off[MFAR_MAX_FIELDS + 1]; };

template <typename VT>
__global__ void sparse_premix_coo_kernel(const int2* __restrict__ keys, const VT* __restrict__ vals, CooFieldOffsets fo,
                                         int n_sparse, const float* __restrict__ w, int w_ld, int w_off, int Q,
                                         int64_t doc_id_base, int64_t n_docs, float* __restrict__ base,
                                         int64_t base_ld) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= fo.off[n_sparse]) return;
  int lo = 0, hi = n_sparse;                       // field j with off[j] <= i < off[j+1]
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (fo.off[mid] <= i) lo = mid; else hi = mid;
  }
  const int2 key = __ldg(keys + i);
  const int64_t doc = int64_t(key.y) - doc_id_base;
  if (key.x < 0 || key.x >= Q || doc < 0 || doc >= n_docs) return;      // other shard / other batch
  atomicAdd(base + int64_t(key.x) * base_ld + doc, __ldg(w + int64_t(key.x) * w_ld + w_off + lo) * float(vals[i]));
}

// Vectorised f16 variant: one thread mixes 8 consecutive docs per 16-byte load (n_sparse loads in flight, unrolled
// by 4), writes two float4.  Needs sparse_ld % 8 == 0 and 16-byte aligned rows (the launcher checks).
__global__ void sparse_premix_h8_kernel(const uint4* __restrict__ sparse, int64_t ld8, int n_sparse,
                                        const float* __restrict__ w, int w_ld, int w_off, int64_t n_docs,
                                        float* __restrict__ base, int64_t base_ld) {
  const int q = blockIdx.y;
  const int64_t n8 = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;     // group of 8 docs
  if (n8 * 8 >= n_docs) return;
  const float* wq = w + int64_t(q) * w_ld + w_off;
  const uint4* sp = sparse + int64_t(q) * n_sparse * ld8 + n8;
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
  for (int j = 0; j < n_sparse; ++j) {
    uint4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(sp + int64_t(j) * ld8));
    const float wj = __ldg(wq + j);
    const __half2* h = reinterpret_cast<const __half2*>(&v);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 f = __half22float2(h[e]);
      acc[2 * e] = fmaf(wj, f.x, acc[2 * e]);
      acc[2 * e + 1] = fmaf(wj, f.y, acc[2 * e + 1]);
    }
  }
  float* dst = base + int64_t(q) * base_ld + n8 * 8;                     // base_ld is a multiple of 128: in bounds
  *reinterpret_cast<float4*>(dst) = make_float4(acc[0], acc[1], acc[2], acc[3]);
  *reinterpret_cast<float4*>(dst + 4) = make_float4(acc[4], acc[5], acc[6], acc[7]);
}

// ---------------------------------------------------------------------------------------
// merge: one CTA (512 threads) per query.  Streams every candidate key of that query from the
// L lists through a 1024-slot shared buffer: admit keys >= running threshold, and whenever the
// buffer may overflow bitonic-sort it, keep the best k, raise the threshold.
// ---------------------------------------------------------------------------------------
constexpr int kMergeThreads = 512;
constexpr int kMergeBuf = 1024;

// block bitonic sort, descending, of the first n (power of two, <= kMergeBuf) slots
__device__ __forceinline__ void block_sort_desc(uint64_t* buf, int n) {
  for (int s = 2; s <= n; s <<= 1) {
    for (int d = s >> 1; d > 0; d >>= 1) {
      __syncthreads();
      const int t = threadIdx.x;                       // n/2 compare-exchanges per stage
      if (t < (n >> 1)) {
        const int lo = ((t & ~(d - 1)) << 1) | (t & (d - 1));
        const int hi = lo | d;
        const bool desc = (lo & s) == 0 || s == n;
        uint64_t a = buf[lo], b = buf[hi];
        if ((a < b) == desc) { buf[lo] = b; buf[hi] = a; }
      }
    }
  }
  __syncthreads();
}
__device__ __forceinline__ void block_sort1024_desc(uint64_t* buf) { block_sort_desc(buf, kMergeBuf); }
__device__ __forceinline__ int pow2_at_least(int c, int floor_) {
  int n = floor_;
  while (n < c) n <<= 1;
  return n;
}

// A many-list merge sees ~L*k candidates above the best per-list threshold (a CTA's k-th key is a weak bound
// shard-wide: ~L*k docs beat it), far more than the 1024-slot sort buffer.  So:
//   A. sweep the lists (a warp per list, coalesced, valid entries only), keep the 32-bit SCORE WORD of every key
//      >= max-threshold in dynamic shared memory (sc_cap words);
//   B. binary-search those words for a cut T with k <= count(score >= T) <= 1024 (one shared-memory pass + block
//      count per probe, ~12 probes);
//   C. sweep the lists again (L2 hits), gather the full keys with score >= T, bitonic-sort, emit the top k.
// If A overflows sc_cap the kernel falls back to the streaming path (stream through the 1024-slot buffer, sort,
// raise the threshold, repeat).
template <class F>
__device__ __forceinline__ void merge_sweep(const uint64_t* __restrict__ keys, const int* __restrict__ counts, int L,
                                            int q_stride, int slots, int q, F&& f) {
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31, nwarp = kMergeThreads >> 5;
  for (int l0 = warp; l0 < L; l0 += nwarp * 4) {
    int cnt[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int l = l0 + u * nwarp;
      cnt[u] = (l < L) ? (counts ? __ldg(counts + int64_t(l) * q_stride + q) : slots) : 0;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int l = l0 + u * nwarp;
      const uint64_t* list = keys + (int64_t(l) * q_stride + q) * slots;
      for (int s0 = 0; s0 < cnt[u]; s0 += 256) {
        uint64_t key[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int sl = s0 + j * 32 + lane;
          key[j] = (sl < cnt[u]) ? __ldcg(list + sl) : 0ull;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (key[j] != 0ull) f(key[j]);
      }
    }
  }
}

__global__ void __launch_bounds__(kMergeThreads)
merge_kernel(const uint64_t* __restrict__ keys, const int* __restrict__ counts, const uint64_t* __restrict__ thr,
             int L, int q_stride, int slots, int k, int sc_cap, uint64_t* __restrict__ out_keys,
             float* __restrict__ out_scores, int64_t* __restrict__ out_ids, const uint64_t* __restrict__ extra,
             int extra_n) {
  extern __shared__ uint32_t sc[];                     // [sc_cap] score words of the candidates
  __shared__ uint64_t buf[kMergeBuf];
  __shared__ int s_cnt, s_probe;
  __shared__ unsigned int s_max;
  __shared__ unsigned long long s_thr;
  const int q = blockIdx.x;
  const int t = threadIdx.x;
  if (t == 0) { s_cnt = 0; s_thr = 0ull; s_max = 0u; s_probe = 0; }
  __syncthreads();
  if (thr != nullptr) {                                // a list that was compacted holds >= k keys >= its thr
    unsigned long long m = 0ull;
    for (int l = t; l < L; l += kMergeThreads) {
      unsigned long long v = thr[int64_t(l) * q_stride + q];
      m = v > m ? v : m;
    }
    if (m) atomicMax(&s_thr, m);
  }
  __syncthreads();
  // ---- A: score words of everything above the threshold
  {
    const unsigned long long thr0 = s_thr;
    unsigned int mx = 0u;
    auto take = [&](uint64_t key) {
      if (key >= thr0) {
        const int pos = atomicAdd(&s_cnt, 1);
        const uint32_t w = uint32_t(key >> 32);
        if (pos < sc_cap) sc[pos] = w;
        mx = w > mx ? w : mx;
      }
    };
    merge_sweep(keys, counts, L, q_stride, slots, q, take);
    for (int j = t; j < extra_n; j += kMergeThreads) {   // the extra list (e.g. the top k of a prefix scored earlier)
      const uint64_t key = extra[int64_t(q) * extra_n + j];
      if (key != 0ull) take(key);
    }
    mx = __reduce_max_sync(0xffffffffu, mx);
    if ((t & 31) == 0 && mx) atomicMax(&s_max, mx);
  }
  __syncthreads();
  const int c = s_cnt;
  if (c <= sc_cap) {
    // ---- B: cut T with k <= count(score >= T) <= kMergeBuf (score ties can make that impossible: then the widest
    // count above kMergeBuf falls back to streaming below)
    uint32_t lo = uint32_t(s_thr >> 32), up = s_max;   // count(>= lo) = c; answer in [lo, up]
    int c_lo = c;
    while (c_lo > kMergeBuf && lo < up) {
      const uint32_t mid = lo + ((up - lo + 1u) >> 1);
      int n = 0;
      for (int i = t; i < c; i += kMergeThreads) n += (sc[i] >= mid) ? 1 : 0;
      n = __reduce_add_sync(0xffffffffu, n);
      __syncthreads();                                 // everyone has read s_probe's previous value
      if (t == 0) s_probe = 0;
      __syncthreads();
      if ((t & 31) == 0 && n) atomicAdd(&s_probe, n);
      __syncthreads();
      const int cm = s_probe;
      if (cm >= k) { lo = mid; c_lo = cm; } else { up = mid - 1u; }
    }
    if (c_lo <= kMergeBuf) {
      // ---- C: gather the full keys above the cut, sort, emit
      __syncthreads();
      if (t == 0) s_cnt = 0;
      __syncthreads();
      const unsigned long long thr0 = s_thr;
      auto gather = [&](uint64_t key) {
        if (key >= thr0 && uint32_t(key >> 32) >= lo) buf[atomicAdd(&s_cnt, 1)] = key;
      };
      merge_sweep(keys, counts, L, q_stride, slots, q, gather);
      for (int j = t; j < extra_n; j += kMergeThreads) {
        const uint64_t key = extra[int64_t(q) * extra_n + j];
        if (key != 0ull) gather(key);
      }
      __syncthreads();
      const int cc = s_cnt;
      const int n = pow2_at_least(cc > k ? cc : k, 128);
      for (int j = cc + t; j < n; j += kMergeThreads) buf[j] = 0ull;
      block_sort_desc(buf, n);
      for (int j = t; j < k; j += kMergeThreads) {
        const uint64_t key = buf[j];
        if (out_keys) out_keys[int64_t(q) * k + j] = key;
        if (out_scores) out_scores[int64_t(q) * k + j] = key ? key_score(key) : -INFINITY;
        if (out_ids) out_ids[int64_t(q) * k + j] = key ? int64_t(key_doc(key)) : int64_t(-1);
      }
      return;
    }
  }
  __syncthreads();
  if (t == 0) s_cnt = 0;
  __syncthreads();
  // ---- streaming path
  const int total = L * slots;
  for (int base = 0; base < total + extra_n; base += kMergeThreads) {
    const int i = base + t;
    if (i < total) {
      const int l = i / slots, sl = i % slots;
      const int cnt = counts ? counts[int64_t(l) * q_stride + q] : slots;
      if (sl < cnt) {
        const uint64_t key = keys[(int64_t(l) * q_stride + q) * slots + sl];
        if (key != 0ull && key >= s_thr) buf[atomicAdd(&s_cnt, 1)] = key;
      }
    } else if (i < total + extra_n) {
      const uint64_t key = extra[int64_t(q) * extra_n + (i - total)];
      if (key != 0ull && key >= s_thr) buf[atomicAdd(&s_cnt, 1)] = key;
    }
    __syncthreads();
    const int cs = s_cnt;                              // snapshot, then barrier: the branch below must be
    __syncthreads();                                   // uniform even if fast threads start the next round
    if (cs > kMergeBuf - kMergeThreads) {
      for (int j = cs + t; j < kMergeBuf; j += kMergeThreads) buf[j] = 0ull;
      block_sort1024_desc(buf);
      if (t == 0) {
        s_cnt = cs < k ? cs : k;
        if (cs >= k) s_thr = buf[k - 1];
      }
      __syncthreads();
    }
  }
  const int cs = s_cnt;
  for (int j = cs + t; j < kMergeBuf; j += kMergeThreads) buf[j] = 0ull;
  block_sort1024_desc(buf);
  for (int j = t; j < k; j += kMergeThreads) {
    const uint64_t key = buf[j];
    if (out_keys) out_keys[int64_t(q) * k + j] = key;
    if (out_scores) out_scores[int64_t(q) * k + j] = key ? key_score(key) : -INFINITY;
    if (out_ids) out_ids[int64_t(q) * k + j] = key ? int64_t(key_doc(key)) : int64_t(-1);
  }
}

// ---------------------------------------------------------------------------------------
// Cross-GPU exchange + merge in ONE kernel over NVLink peer memory (replaces ncclAllGather + merge).
// Every rank owns a buffer [flags: S][world][q_cap] i32 | [keys: S][world][q_cap][k_cap] u64 (S = 4 slots) that all peers have
// mapped (CUDA VMM / torch symmetric memory).  A grid of min(Q, 296) CTAs - all co-resident (2 per SM) - walks the
// queries b, b + grid, ... in TWO sweeps:
//   1. PUSH   for each of its queries, the rank's local top-k keys go into slot [parity][rank][q] of EVERY rank's
//             buffer (st.global on peer-mapped addresses -> NVLink) and, after a system-scope fence, the flag = epoch;
//   2. WAIT + MERGE  for each of its queries, until the flags of all ranks show `epoch` in the LOCAL buffer
//             (ld.acquire.sys), then the world * k_in keys (now local) are ranked by the block bitonic sort.
// No CTA waits before it has pushed everything it owns, and every CTA of the grid is resident, so every push of every
// rank is issued regardless of how the hardware orders CTAs: the wait always terminates once all ranks have launched
// (round 1 used one CTA per query and relied on CTAs being scheduled in index order when Q exceeded the resident
// capacity).  Slots rotate with the epoch (epoch % 4).  Complete exchanges: a peer can only be one call ahead (it needs
// this rank's next push to finish its next call).  Pipelined exchanges (push epoch e, merge epoch e-1 in the same
// step): a peer's push of e+2 can precede this rank's merge of e-1, its push of e+3 cannot (that needs this rank's
// push of e+1, which follows the merge of e-1 in stream order) - hence four slots.
// ---------------------------------------------------------------------------------------
constexpr int kMaxPeers = 8;
constexpr int kExchangeMaxCtas = 2 * kNumSmsB200;
struct PeerBufs { unsigned long long base[kMaxPeers]; };

__device__ __forceinline__ void st_release_sys(int* p, int v) {
  asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ int ld_acquire_sys(const int* p) {
  int v;
  asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

constexpr int kExchangeSlots = MFAR_EXCHANGE_SLOTS;   // key / flag slots per (rank, query), indexed by epoch % slots

// sweep 1: this CTA's queries -> every rank's buffer, then the flags
__device__ __forceinline__ void exchange_push(const uint64_t* __restrict__ local_keys, int Q, int k_in,
                                              const PeerBufs& peers, int rank, int world, int q_cap, int k_cap, int epoch) {
  const int t = threadIdx.x;
  const int sl = epoch % kExchangeSlots;
  const size_t flag_bytes = size_t(kExchangeSlots) * world * q_cap * sizeof(int);
  for (int q = blockIdx.x; q < Q; q += gridDim.x) {
    const size_t slot = (size_t(sl) * world + rank) * q_cap + q;              // [slot][rank][q]
    for (int i = t; i < world * k_in; i += kMergeThreads) {
      const int r = i / k_in, j = i % k_in;
      uint64_t* dst = reinterpret_cast<uint64_t*>(peers.base[r] + flag_bytes) + slot * k_cap + j;
      *dst = __ldg(local_keys + int64_t(q) * k_in + j);
    }
    __threadfence_system();
    __syncthreads();
    if (t < world) st_release_sys(reinterpret_cast<int*>(peers.base[t]) + slot, epoch);
  }
}

// sweep 2: wait (bounded: a peer that never arrives becomes an error, not a hang) and merge the keys of `epoch`
__device__ __forceinline__ void exchange_wait_merge(uint64_t* buf, int Q, int q_pushed, int k_in, const PeerBufs& peers, int rank,
                                                    int world, int q_cap, int k_cap, int epoch, int k,
                                                    uint64_t* __restrict__ out_keys, float* __restrict__ out_scores,
                                                    int64_t* __restrict__ out_ids, int* __restrict__ err) {
  const int t = threadIdx.x;
  const int sl = epoch % kExchangeSlots;
  const size_t flag_bytes = size_t(kExchangeSlots) * world * q_cap * sizeof(int);
  const uint64_t* mine = reinterpret_cast<const uint64_t*>(peers.base[rank] + flag_bytes);
  for (int q = blockIdx.x; q < Q; q += gridDim.x) {
    const bool live = epoch >= 1 && q < q_pushed;                              // else: nothing was pushed for this query
    if (live && t < world) {
      const int* f = reinterpret_cast<const int*>(peers.base[rank]) + (size_t(sl) * world + t) * q_cap + q;
      const unsigned long long t0 = clock64();
      while (ld_acquire_sys(f) != epoch) {
        if (clock64() - t0 > 20000000000ull) {                                // ~10 s
#ifdef MFAR_TIMEOUT_EXIT   // debug build: say what was being waited for, then leave instead of trapping
          printf("[mfar_b200] exchange wait timed out: rank %d waits for rank %d, query %d, epoch %d (slot %d), flag %d\n",
                 rank, t, q, epoch, sl, ld_acquire_sys(f));
          asm volatile("exit;");
#endif
          atomicExch(err, 31);
          __threadfence_system();
          asm volatile("trap;");
        }
        __nanosleep(100);
      }
    }
    __syncthreads();
    for (int i = t; i < kMergeBuf; i += kMergeThreads) {                      // all data is in this rank's own buffer now
      uint64_t key = 0ull;
      if (live && i < world * k_in) {
        const int r = i / k_in, j = i % k_in;
        key = __ldcg(mine + ((size_t(sl) * world + r) * q_cap + q) * k_cap + j);
      }
      buf[i] = key;
    }
    block_sort1024_desc(buf);
    for (int j = t; j < k; j += kMergeThreads) {
      const uint64_t key = buf[j];
      if (out_keys) out_keys[int64_t(q) * k + j] = key;
      if (out_scores) out_scores[int64_t(q) * k + j] = key ? key_score(key) : -INFINITY;
      if (out_ids) out_ids[int64_t(q) * k + j] = key ? int64_t(key_doc(key)) : int64_t(-1);
    }
    __syncthreads();                                                          // buf is reused by the next query
  }
}

// mode 0: push + wait + merge of the same epoch (one call = one complete exchange);
// mode 1: push only;  mode 2: wait + merge of epoch - lag (the PIPELINED exchange: a step pushes its keys and merges
// the previous step's, whose peer pushes landed a whole step ago - no rank waits for the slowest one any more)
__global__ void __launch_bounds__(kMergeThreads, 2)
exchange_merge_kernel(const uint64_t* __restrict__ local_keys, int Q, int k_in, PeerBufs peers, int rank, int world,
                      int q_cap, int k_cap, int epoch_arg, const int* __restrict__ epoch_dev, int mode, int lag, int k,
                      uint64_t* __restrict__ out_keys, float* __restrict__ out_scores, int64_t* __restrict__ out_ids,
                      int* __restrict__ err) {
  __shared__ uint64_t buf[kMergeBuf];
  // the call counter: a kernel argument, or - so that the launch can be replayed from a CUDA graph - a device word
  // that bump_epoch_kernel (same stream, in front of the push) increments
  const int epoch = epoch_dev ? *epoch_dev : epoch_arg;
  if (mode != 2) exchange_push(local_keys, Q, k_in, peers, rank, world, q_cap, k_cap, epoch);
  // how many queries the epoch being merged was pushed with (recorded by bump_epoch_kernel): a pipelined merge right
  // after a change of batch size must not wait for queries nobody pushed
  int q_pushed = Q;
  if (epoch_dev && mode == 2 && epoch - lag >= 1) q_pushed = min(Q, epoch_dev[1 + (epoch - lag) % kExchangeSlots]);
  if (mode != 1)
    exchange_wait_merge(buf, Q, q_pushed, k_in, peers, rank, world, q_cap, k_cap, epoch - lag, k, out_keys, out_scores,
                        out_ids, err);
}

// epoch_dev: int32 [1 + slots] = the call counter, then the batch size each slot's epoch was pushed with
__global__ void bump_epoch_kernel(int* epoch_dev, int Q) {
  const int e = *epoch_dev + 1;
  *epoch_dev = e;
  epoch_dev[1 + e % kExchangeSlots] = Q;
}

__global__ void seed_gthr_kernel(unsigned long long* gthr, const unsigned long long* seed, int Q) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q < Q) gthr[q] = seed[q];
}
// key > (kth - 1)  <=>  key >= kth: the k-th best doc of the prefix itself must still be admitted by the main pass
__global__ void seed_from_keys_kernel(const uint64_t* keys, int Q, int k, unsigned long long* seed) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q < Q) {
    const uint64_t kth = keys[int64_t(q) * k + (k - 1)];
    seed[q] = kth ? kth - 1ull : 0ull;
  }
}

// index.py:192-193 quirk: running top-k starts as (0.0, row 0) entries.  They replace the negative scores only: a NaN
// entry outranks them under torch.topk's order (NaN largest) and stays.
__global__ void zero_init_kernel(float* scores, int64_t* ids, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && scores[i] < 0.0f) { scores[i] = 0.0f; ids[i] = 0; }
}

// ---------------------------------------------------------------------------------------
// host launchers
// ---------------------------------------------------------------------------------------
int launch_pack_rows(const void* src, int src_dtype, int64_t n_rows, int64_t row_begin, void* packed,
                     int n_fields, int field, int dim, int normalize, cudaStream_t st) {
  if (n_rows == 0) return MFAR_OK;
  const int threads = 256;
  const int64_t blocks = (n_rows * 32 + threads - 1) / threads;
  if (src_dtype == MFAR_F32)
    pack_rows_kernel<float><<<(unsigned)blocks, threads, 0, st>>>(static_cast<const float*>(src), n_rows, row_begin,
                                                                 static_cast<__nv_bfloat16*>(packed), n_fields, field,
                                                                 dim, normalize);
  else if (src_dtype == MFAR_BF16)
    pack_rows_kernel<__nv_bfloat16><<<(unsigned)blocks, threads, 0, st>>>(
        static_cast<const __nv_bfloat16*>(src), n_rows, row_begin, static_cast<__nv_bfloat16*>(packed), n_fields,
        field, dim, normalize);
  else
    return MFAR_ERR_ARG;
  MFAR_CUDA_OK(cudaGetLastError());
  return MFAR_OK;
}

int launch_unpack_rows(const void* packed, int n_fields, int field, int dim, int64_t row_begin, int64_t n_rows,
                       float* dst, cudaStream_t st) {
  if (n_rows == 0) return MFAR_OK;
  const int threads = 256;
  const int64_t blocks = (n_rows * 32 + threads - 1) / threads;
  unpack_rows_kernel<<<(unsigned)blocks, threads, 0, st>>>(static_cast<const __nv_bfloat16*>(packed), n_fields, field,
                                                           dim, row_begin, n_rows, dst);
  MFAR_CUDA_OK(cudaGetLastError());
  return MFAR_OK;
}

int launch_pack_rows_e4m3(const void* src, int src_dtype, int64_t n_rows, int64_t row_begin, uint8_t* payload,
                          float* scales, int n_fields, int field, int dim, int normalize, cudaStream_t st) {
  if (n_rows == 0) return MFAR_OK;
  const int threads = 256;
  const unsigned blocks = unsigned((n_rows * 32 + threads - 1) / threads);
  if (src_dtype == MFAR_F32)
    pack_rows_e4m3_kernel<float><<<blocks, threads, 0, st>>>(static_cast<const float*>(src), n_rows, row_begin, payload,
                                                             scales, n_fields, field, dim, normalize);
  else if (src_dtype == MFAR_BF16)
    pack_rows_e4m3_kernel<__nv_bfloat16><<<blocks, threads, 0, st>>>(static_cast<const __nv_bfloat16*>(src), n_rows,
                                                                     row_begin, payload, scales, n_fields, field, dim,
                                                                     normalize);
  else
    return MFAR_ERR_ARG;
  MFAR_CUDA_OK(cudaGetLastError());
  return MFAR_OK;
}

int launch_unpack_rows_e4m3(const uint8_t* payload, const float* scales, int n_fields, int field, int dim,
                            int64_t row_begin, int64_t n_rows, float* dst, cudaStream_t st) {
  if (n_rows == 0) return MFAR_OK;
  const int threads = 256;
  const unsigned blocks = unsigned((n_rows * 32 + threads - 1) / threads);
  unpack_rows_e4m3_kernel<<<blocks, threads, 0, st>>>(payload, scales, n_fields, field, dim, row_begin, n_rows, dst);
  MFAR_CUDA_OK(cudaGetLastError());
  return MFAR_OK;
}

int launch_mixture_weights(const float* q_emb, const float* W, const float* mask, int Q, int E, int F,
                           int query_cond, float* out_w, cudaStream_t st) {
  mixture_weights_kernel<<<Q, 256, 0, st>>>(q_emb, W, mask, E, F, query_cond, out_w);
  MFAR_CUDA_OK(cudaGetLastError());
  return MFAR_OK;
}

int launch_mixture_apply(const float* x, const float* w, int B, int S, int F, int w_rows, float* out,
                         cudaStream_t st) {
  const int64_t BS = int64_t(B) * S;
  if (BS == 0) return MFAR_OK;
  mixture_apply_kernel<<<(unsigned)((BS + 255) / 256), 256, 0, st>>>(x, w, BS, S, F, w_rows, out);
  MFAR_CUDA_OK(cudaGetLastError());
  return MFAR_OK;
}

int launch_score_candidates(const void* corpus, const float* corpus_scales, int64_t n_docs, int corpus_fields,
                            int field_begin, int n_fields, int dim, const void* q_vecs, const float* q_scales, int Q,
                            const int64_t* rows, int C, float* out, cudaStream_t st) {
  if (C == 0 || n_fields == 0) return MFAR_OK;
  const int64_t warps = int64_t(C) * n_fields;
  const unsigned blocks = unsigned((warps * 32 + 255) / 256);
  if (corpus_scales)
    score_candidates_kernel<true><<<blocks, 256, 0, st>>>(corpus, corpus_scales, n_docs, corpus_fields, field_begin,
                                                          n_fields, dim, q_vecs, q_scales, Q, rows, C, out);
  else
    score_candidates_kernel<false><<<blocks, 256, 0, st>>>(corpus, nullptr, n_docs, corpus_fields, field_begin,
                                                           n_fields, dim, q_vecs, nullptr, Q, rows, C, out);
  MFAR_CUDA_OK(cudaGetLastError());
  return MFAR_OK;
}

int launch_sparse_premix(const void* sparse, int sparse_dtype, int64_t sparse_ld, int n_sparse, const float* w,
                         int w_ld, int w_off, int Q, int64_t n_docs, float* base, int64_t base_ld,
                         cudaStream_t st) {
  dim3 grid((unsigned)((n_docs + 255) / 256), Q);
  if (sparse_dtype == MFAR_F32)
    sparse_premix_kernel<float><<<grid, 256, 0, st>>>(static_cast<const float*>(sparse), sparse_ld, n_sparse, w, w_ld,
                                                      w_off, n_docs, base, base_ld);
  else if (sparse_dtype == MFAR_F16) {
    if (sparse_ld % 8 == 0 && reinterpret_cast<uintptr_t>(sparse) % 16 == 0 && base_ld % 8 == 0 &&
        reinterpret_cast<uintptr_t>(base) % 16 == 0) {
      dim3 g8((unsigned)(((n_docs + 7) / 8 + 255) / 256), Q);
      sparse_premix_h8_kernel<<<g8, 256, 0, st>>>(static_cast<const uint4*>(sparse), sparse_ld / 8, n_sparse, w, w_ld,
                                                  w_off, n_docs, base, base_ld);
    } else {
      sparse_premix_kernel<__half><<<grid, 256, 0, st>>>(static_cast<const __half*>(sparse), sparse_ld, n_sparse, w,
                                                         w_ld, w_off, n_docs, base, base_ld);
    }
  }
  else
    return MFAR_ERR_ARG;
  MFAR_CUDA_OK(cudaGetLastError());
  return MFAR_OK;
}

int launch_sparse_premix_coo(const int32_t* keys, const void* vals, int val_dtype, const int64_t* field_offsets_host,
                             int n_sparse, const float* w, int w_ld, int w_off, int Q, int64_t doc_id_base,
                             int64_t n_docs, float* base, int64_t base_ld, cudaStream_t st) {
  CooFieldOffsets fo{};
  for (int j = 0; j <= n_sparse; ++j) {
    fo.off[j] = field_offsets_host[j];
    if (j > 0 && fo.off[j] < fo.off[j - 1]) return MFAR_ERR_ARG;
  }
  const long long nnz = fo.off[n_sparse];
  if (nnz == 0) return MFAR_OK;
  const unsigned blocks = unsigned((nnz + 255) / 256);
  if (val_dtype == MFAR_F16)
    sparse_premix_coo_kernel<__half><<<blocks, 256, 0, st>>>(reinterpret_cast<const int2*>(keys),
                                                             static_cast<const __half*>(vals), fo, n_sparse, w, w_ld,
                                                             w_off, Q, doc_id_base, n_docs, base, base_ld);
  else if (val_dtype == MFAR_F32)
    sparse_premix_coo_kernel<float><<<blocks, 256, 0, st>>>(reinterpret_cast<const int2*>(keys),
                                                            static_cast<const float*>(vals), fo, n_sparse, w, w_ld,
                                                            w_off, Q, doc_id_base, n_docs, base, base_ld);
  else
    return MFAR_ERR_ARG;
  MFAR_CUDA_OK(cudaGetLastError());
  return MFAR_OK;
}

int launch_merge(const uint64_t* keys, const int* counts, const uint64_t* thr, int L, int q_stride, int slots, int Q,
                 int k, uint64_t* out_keys, float* out_scores, int64_t* out_ids, cudaStream_t st, const uint64_t* extra,
                 int extra_n) {
  if (int64_t(L) * slots > (int64_t(1) << 30)) return MFAR_ERR_SHAPE;
  if (extra == nullptr) extra_n = 0;
  // score-word scratch: every slot of every list if that fits ~150 KB, else a cap (overflow -> streaming path)
  int sc_cap = int(std::min<int64_t>(int64_t(L) * slots + extra_n, 38 * 1024));
  sc_cap = (sc_cap + 3) & ~3;
  const size_t smem = size_t(sc_cap) * sizeof(uint32_t);
  static PerDeviceOnce attr_once;
  MFAR_CUDA_OK(attr_once.run([&] {
    return cudaFuncSetAttribute(merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
  }));
  merge_kernel<<<Q, kMergeThreads, smem, st>>>(keys, counts, thr, L, q_stride, slots, k, sc_cap, out_keys, out_scores,
                                              out_ids, extra, extra_n);
  MFAR_CUDA_OK(cudaGetLastError());
  return MFAR_OK;
}

int launch_exchange_merge(const uint64_t* local_keys, int Q, int k_in, int k, int rank, int world,
                          const unsigned long long* peer_bases, int q_cap, int k_cap, int epoch, int* epoch_dev, int mode,
                          int lag, uint64_t* out_keys, float* out_scores, int64_t* out_ids, cudaStream_t st) {
  if (world < 1 || world > kMaxPeers || world * k_in > kMergeBuf || Q > q_cap || k_in > k_cap) return MFAR_ERR_SHAPE;
  PeerBufs pb{};
  for (int r = 0; r < world; ++r) pb.base[r] = peer_bases[r];
  // the error word lives at the very end of this rank's buffer
  int* err = reinterpret_cast<int*>(pb.base[rank] + size_t(kExchangeSlots) * world * q_cap * sizeof(int) +
                                    size_t(kExchangeSlots) * world * q_cap * k_cap * sizeof(uint64_t));
  if (epoch_dev && mode != 2) bump_epoch_kernel<<<1, 1, 0, st>>>(epoch_dev, Q);   // a push opens a new epoch
  const int ctas = Q < kExchangeMaxCtas ? Q : kExchangeMaxCtas;               // all resident: 2 x 512 threads per SM
  exchange_merge_kernel<<<ctas, kMergeThreads, 0, st>>>(local_keys, Q, k_in, pb, rank, world, q_cap, k_cap, epoch,
                                                        epoch_dev, mode, lag, k, out_keys, out_scores, out_ids, err);
  MFAR_CUDA_OK(cudaGetLastError());
  return MFAR_OK;
}

int launch_seed_gthr(unsigned long long* gthr, const unsigned long long* seed, int Q, cudaStream_t st) {
  seed_gthr_kernel<<<(Q + 255) / 256, 256, 0, st>>>(gthr, seed, Q);
  MFAR_CUDA_OK(cudaGetLastError());
  return MFAR_OK;
}

int launch_seed_from_keys(const uint64_t* keys, int Q, int k, unsigned long long* seed, cudaStream_t st) {
  seed_from_keys_kernel<<<(Q + 255) / 256, 256, 0, st>>>(keys, Q, k, seed);
  MFAR_CUDA_OK(cudaGetLastError());
  return MFAR_OK;
}

int launch_zero_init(float* scores, int64_t* ids, int n, cudaStream_t st) {
  if (n == 0) return MFAR_OK;
  zero_init_kernel<<<(n + 255) / 256, 256, 0, st>>>(scores, ids, n);
  MFAR_CUDA_OK(cudaGetLastError());
  return MFAR_OK;
}

}  // namespace mfar
