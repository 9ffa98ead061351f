// CUDA-core streaming scoring pass (small query batches; also the on-GPU cross-check of the
// tcgen05 path at sizes the CPU oracle cannot reach).
//
// One CTA = 4 warps = one 128-doc corpus tile at a time (persistent, tiles strided by grid).
// A warp owns 32 docs of the tile.  For each doc and field the 32 lanes read the row with
// 16-byte loads (coalesced, 512 B per request), FMA against the fp32 query slice they keep in
// registers, butterfly-reduce, and fold w[q,f] * s_f into the doc's running mixture score.
// Scores never leave registers: lane j keeps doc j's final score, adds the pre-mixed sparse
// term, and pushes (score,id) keys that beat the CTA's per-query threshold into its candidate
// list (threshold + compaction logic in common.cuh).
// E4M3 corpus (E8): the same mapping with 8-byte vectors of 8 elements, decoded by cvt.rn.f16x2.e4m3x2 (exact); the
// payload dot product D is then scaled as the tensor-core path does it, w * ((D * s_q) * s_d) - the CUDA-core
// cross-check of the kind::f8f6f4 kernel.
#include "common.cuh"
#include "kernels.h"

namespace mfar {

constexpr int kSimtThreads = 128;
constexpr int kSimtMaxVec = 4;  // 16-byte vectors per lane per row: dim <= 4*32*8 = 1024

struct SimtParams {
  const void* corpus;
  int64_t n_docs;
  int n_tiles, corpus_fields, field_begin, n_dense, dim;
  const void* q_vecs;
  const float* corpus_scales;   // E8 only
  const float* q_scales;        // E8 only
  int Q;
  const float* w;
  int w_ld;
  const float* base;
  int64_t base_ld;
  int64_t doc_id_base;
  int k;
  TopkWorkspace ws;
  DocFilter filt;               // FILT only
};

__device__ __forceinline__ void bf16x8_to_f32(const uint4& v, float (&f)[8]) {
  f[0] = __uint_as_float(v.x << 16); f[1] = __uint_as_float(v.x & 0xffff0000u);
  f[2] = __uint_as_float(v.y << 16); f[3] = __uint_as_float(v.y & 0xffff0000u);
  f[4] = __uint_as_float(v.z << 16); f[5] = __uint_as_float(v.z & 0xffff0000u);
  f[6] = __uint_as_float(v.w << 16); f[7] = __uint_as_float(v.w & 0xffff0000u);
}

__device__ __forceinline__ uint4 ld_stream(const uint4* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}

// QB = queries handled per corpus pass (their slices live in registers)
// FILT: doc filter; the lane's filter word of each query is loaded at the tile's start and tested after the key compare
template <int QB, bool E8, bool FILT>
__global__ void __launch_bounds__(kSimtThreads) score_simt_kernel(SimtParams p) {
  extern __shared__ float s_w[];                      // [QB][n_dense]
  __shared__ unsigned long long s_thr[QB];
  __shared__ int s_cnt[QB];

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = blockIdx.x;
  const int nvec = p.dim / 8;                         // 16-byte vectors per row
  const int vec_per_lane = (nvec + 31) / 32;

  for (int q0 = 0; q0 < p.Q; q0 += QB) {
    const int nq = min(QB, p.Q - q0);
    __syncthreads();
    for (int i = threadIdx.x; i < QB * p.n_dense; i += kSimtThreads) {
      const int qi = i / p.n_dense, f = i % p.n_dense;
      s_w[i] = qi < nq ? p.w[int64_t(q0 + qi) * p.w_ld + f] : 0.f;
    }
    if (threadIdx.x < QB) { s_thr[threadIdx.x] = 0ull; s_cnt[threadIdx.x] = 0; }
    // query slices -> registers (fp32)
    float qreg[QB][kSimtMaxVec][8];
    float sq[QB];
#pragma unroll
    for (int qi = 0; qi < QB; ++qi) sq[qi] = (E8 && qi < nq) ? p.q_scales[q0 + qi] : 1.f;
#pragma unroll
    for (int qi = 0; qi < QB; ++qi)
#pragma unroll
      for (int v = 0; v < kSimtMaxVec; ++v) {
        const int vi = lane + 32 * v;
        if (p.n_dense > 0 && v < vec_per_lane && vi < nvec && qi < nq) {
          if constexpr (E8) {
            e4m3x8_to_f32(*reinterpret_cast<const uint2*>(static_cast<const uint8_t*>(p.q_vecs) + int64_t(q0 + qi) * p.dim +
                                                          vi * 8), qreg[qi][v]);
          } else {
            uint4 raw = *reinterpret_cast<const uint4*>(static_cast<const __nv_bfloat16*>(p.q_vecs) +
                                                        int64_t(q0 + qi) * p.dim + vi * 8);
            bf16x8_to_f32(raw, qreg[qi][v]);
          }
        } else {
#pragma unroll
          for (int e = 0; e < 8; ++e) qreg[qi][v][e] = 0.f;
        }
      }
    __syncthreads();

    for (int t = g; t < p.n_tiles; t += gridDim.x) {
      const int64_t fbit = p.doc_id_base + int64_t(t) * kTileDocs + warp * 32 + lane;   // global id of the lane's doc
      uint32_t fw[QB];
#pragma unroll
      for (int qi = 0; qi < QB; ++qi) {
        const uint32_t* frow = p.filt.bits + int64_t(q0 + qi) * p.filt.stride;
        fw[qi] = (FILT && qi < nq) ? filter_ld_word(frow, p.filt.words, fbit >> 5) : 0u;
      }
      float mine[QB];
#pragma unroll
      for (int qi = 0; qi < QB; ++qi) mine[qi] = 0.f;

      for (int j = 0; j < 32; ++j) {
        float acc[QB];
#pragma unroll
        for (int qi = 0; qi < QB; ++qi) acc[qi] = 0.f;
        for (int f = 0; f < p.n_dense; ++f) {
          const int64_t row_idx = (int64_t(t) * p.corpus_fields + p.field_begin + f) * kTileDocs + warp * 32 + j;
          float part[QB];
#pragma unroll
          for (int qi = 0; qi < QB; ++qi) part[qi] = 0.f;
          float sd = 1.f;
          if constexpr (E8) {
            const uint2* row = static_cast<const uint2*>(p.corpus) + row_idx * nvec;
            uint2 raw[kSimtMaxVec];
#pragma unroll
            for (int v = 0; v < kSimtMaxVec; ++v) {
              const int vi = lane + 32 * v;
              if (v < vec_per_lane && vi < nvec) {
                asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];"
                             : "=r"(raw[v].x), "=r"(raw[v].y) : "l"(row + vi));
              } else {
                raw[v] = make_uint2(0, 0);
              }
            }
            sd = __ldg(p.corpus_scales + row_idx);
#pragma unroll
            for (int v = 0; v < kSimtMaxVec; ++v) {
              float x[8];
              e4m3x8_to_f32(raw[v], x);
#pragma unroll
              for (int qi = 0; qi < QB; ++qi)
#pragma unroll
                for (int e = 0; e < 8; ++e) part[qi] = fmaf(x[e], qreg[qi][v][e], part[qi]);
            }
          } else {
            const uint4* row = static_cast<const uint4*>(p.corpus) + row_idx * nvec;
            uint4 raw[kSimtMaxVec];
#pragma unroll
            for (int v = 0; v < kSimtMaxVec; ++v) {
              const int vi = lane + 32 * v;
              raw[v] = (v < vec_per_lane && vi < nvec) ? ld_stream(row + vi) : make_uint4(0, 0, 0, 0);
            }
#pragma unroll
            for (int v = 0; v < kSimtMaxVec; ++v) {
              float x[8];
              bf16x8_to_f32(raw[v], x);
#pragma unroll
              for (int qi = 0; qi < QB; ++qi)
#pragma unroll
                for (int e = 0; e < 8; ++e) part[qi] = fmaf(x[e], qreg[qi][v][e], part[qi]);
            }
          }
#pragma unroll
          for (int qi = 0; qi < QB; ++qi) {
            float s = part[qi];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            if (E8) s = (s * sq[qi]) * sd;
            acc[qi] = fmaf(s_w[qi * p.n_dense + f], s, acc[qi]);
          }
        }
#pragma unroll
        for (int qi = 0; qi < QB; ++qi)
          if (lane == j) mine[qi] = acc[qi];
      }

      // lane owns doc (tile*128 + warp*32 + lane)
      const int64_t doc_local = int64_t(t) * kTileDocs + warp * 32 + lane;
      if (doc_local < p.n_docs) {
#pragma unroll
        for (int qi = 0; qi < QB; ++qi) {
          if (qi < nq) {
            float s = mine[qi];
            if (p.base) s += p.base[int64_t(q0 + qi) * p.base_ld + doc_local];
            const uint64_t key = make_key(s, uint32_t(p.doc_id_base + doc_local));
            if (key > s_thr[qi] && (!FILT || ((fw[qi] >> (fbit & 31)) & 1u))) {
              const int pos = atomicAdd(&s_cnt[qi], 1);
              __stcg(p.ws.cand_keys + (int64_t(g) * p.ws.q_pad + q0 + qi) * kCandCap + pos, key);
            }
          }
        }
      }
      __syncthreads();
      for (int qi = warp; qi < nq; qi += kSimtThreads / 32) {
        const int cnt = s_cnt[qi];
        if (cnt > kCandCap - kTileDocs) {
          uint64_t* list = p.ws.cand_keys + (int64_t(g) * p.ws.q_pad + q0 + qi) * kCandCap;
          const uint64_t kth = warp_compact_list(list, cnt, p.k, lane);
          if (lane == 0) { s_thr[qi] = kth; s_cnt[qi] = p.k; }
        }
      }
      __syncthreads();
    }
    if (threadIdx.x < nq) {
      p.ws.cand_cnt[int64_t(g) * p.ws.q_pad + q0 + threadIdx.x] = s_cnt[threadIdx.x];
      p.ws.cand_thr[int64_t(g) * p.ws.q_pad + q0 + threadIdx.x] = s_thr[threadIdx.x];
    }
  }
}

PassPlan plan_score_simt(int Q, int n_tiles) {
  PassPlan p{};
  p.impl = MFAR_IMPL_SIMT;
  p.q_tiles = p.cg = 1;
  p.q_pad = p.q_pad_total = round_up(Q, 4);
  int w = (Q <= 8) ? kNumSmsB200 * 4 : kNumSmsB200;   // bounded so the candidate workspace stays small
  if (w > n_tiles) w = n_tiles;
  if (w < 1) w = 1;
  p.workers = p.lists = w;
  return p;
}

template <bool E8, bool FILT>
static void launch_simt_qb(const SimtParams& p, int Q, int n_dense, int workers, cudaStream_t st) {
  if (Q == 1) {
    score_simt_kernel<1, E8, FILT><<<workers, kSimtThreads, 1 * n_dense * sizeof(float) + 16, st>>>(p);
  } else if (Q == 2) {
    score_simt_kernel<2, E8, FILT><<<workers, kSimtThreads, 2 * n_dense * sizeof(float) + 16, st>>>(p);
  } else {
    score_simt_kernel<4, E8, FILT><<<workers, kSimtThreads, 4 * n_dense * sizeof(float) + 16, st>>>(p);
  }
}

int launch_score_simt(const ScoreArgs& a, const PassPlan& plan, const TopkWorkspace& ws, cudaStream_t st,
                      int* launches) {
  if (a.dim % 8 != 0 || a.dim > kSimtMaxVec * 32 * 8) return MFAR_ERR_SHAPE;
  const bool e8 = a.corpus_dtype == MFAR_E4M3;
  if (e8 && (reinterpret_cast<uintptr_t>(a.corpus) % 8 || reinterpret_cast<uintptr_t>(a.q_vecs) % 8))
    return MFAR_ERR_ARG;
  SimtParams p;
  p.corpus = a.corpus; p.corpus_scales = a.corpus_scales; p.q_scales = a.q_scales;
  p.n_docs = a.n_docs; p.n_tiles = a.n_tiles; p.corpus_fields = a.corpus_fields; p.field_begin = a.field_begin;
  p.n_dense = a.n_dense; p.dim = a.dim; p.q_vecs = a.q_vecs; p.Q = a.Q;
  p.w = a.w; p.w_ld = a.w_ld; p.base = a.base; p.base_ld = a.base_ld; p.doc_id_base = a.doc_id_base; p.k = a.k;
  p.ws = ws;
  p.filt = DocFilter{a.filter_bits, a.filter_stride, a.filter_words};
  const bool f = a.filter_bits != nullptr;
  auto launch = e8 ? (f ? launch_simt_qb<true, true> : launch_simt_qb<true, false>)
                   : (f ? launch_simt_qb<false, true> : launch_simt_qb<false, false>);
  launch(p, a.Q, a.n_dense, plan.workers, st);
  MFAR_CUDA_OK(cudaGetLastError());
  ++*launches;
  return MFAR_OK;
}

}  // namespace mfar
