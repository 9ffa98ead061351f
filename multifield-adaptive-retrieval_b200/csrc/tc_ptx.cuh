// Inline-PTX wrappers for the sm_100a tensor-core kernels (TMA, mbarrier, tcgen05 / TMEM, clusters) and the
// host-side TMA descriptor helper.  Shared by score_tc.cu (doc-stationary M) and score_qs.cu (query-stationary).
#pragma once
#include <cuda.h>

#include "common.cuh"

namespace mfar {

constexpr int kChunkK = 64;   // bf16 elements per K-chunk = 128 B = swizzle span
constexpr int kChunkK8 = 128; // E4M3 elements per K-chunk: the same 128 B span, consumed by 4 MMAs of K = 32
constexpr int kUmmaK = 16;
constexpr int kEpiThreads = 128;   // 4 epilogue warps: one per 32-lane TMEM sub-partition
#ifdef MFAR_TIMEOUT_EXIT
constexpr unsigned long long kWaitTimeoutCycles = 200000000ull;
#else
constexpr unsigned long long kWaitTimeoutCycles = 4000000000ull;
#endif  // ~2 s: turn a pipeline bug into a trap, not a hang

// ------------------------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, int* err, int code) {
  if (mbar_try_wait(bar, parity)) return;
  const unsigned long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > kWaitTimeoutCycles) {
#ifdef MFAR_TIMEOUT_EXIT   // debug build: report and leave instead of trapping (a trap loses the printf buffer)
      if ((threadIdx.x & 31) == 0)
        printf("[mfar_b200] mbarrier wait timed out: code %d, block (%d,%d), warp %d, parity %u\n", code, int(blockIdx.x),
               int(blockIdx.y), int(threadIdx.x >> 5), parity);
      asm volatile("exit;");
#endif
      if (err) atomicExch(err, code);
      __threadfence_system();
      asm volatile("trap;");
    }
  }
}
// One lane of a converged warp.  Issue tcgen05 / TMA instructions as `if (elect_one()) asm(...)` from
// warp-UNIFORM control flow: operands computed outside the `if` stay in uniform registers, so the issuing
// loop is not slowed by per-instruction vote/R2UR "waterfall" sequences.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ int ld_relaxed_s32(const int* p) {
  int v;
  asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu(int* p, int v) {
  asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ int ld_acquire_gpu(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// 32-byte global load (LDG.E.256, sm_100+), read-only path, no L1 allocation: used where a thread streams a private
// row (one query's sparse scores) and every 32-byte sector is consumed exactly once
__device__ __forceinline__ void ldg256_stream(const void* p, uint32_t (&v)[8]) {
  asm volatile("ld.global.nc.L1::no_allocate.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "l"(p));
}
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void tma_load_2d(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]^T, bf16 x bf16 -> fp32
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t addr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(addr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory"); }

// K-major, SWIZZLE_128B shared-memory matrix descriptor (sm_100 format):
//   [0,14) start address >> 4 | [16,30) LBO >> 4 (unused for swizzled K-major: 1) | [32,46) SBO >> 4
//   (8 rows * 128 B = 1024 B between 8-row groups) | [46,48) version = 1 | [61,64) layout = 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_sw128_desc(uint32_t smem_addr) {
  return uint64_t((smem_addr & 0x3FFFFu) >> 4) | (uint64_t(1) << 16) | (uint64_t(1024 >> 4) << 32) |
         (uint64_t(1) << 46) | (uint64_t(2) << 61);
}
// kind::f16 instruction descriptor: D=f32 (bit 4), A=B=bf16 (bits 7,10), K-major both, N>>3 @17, M>>4 @24
__host__ __device__ constexpr uint32_t make_idesc(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (uint32_t(N >> 3) << 17) | (uint32_t(M >> 4) << 24);
}
// kind::f8f6f4 instruction descriptor: D=f32 (bit 4), A=B=E4M3 (format 0 in bits [7,10) and [10,13)), K-major both
__host__ __device__ constexpr uint32_t make_idesc_e4m3(int M, int N) {
  return (1u << 4) | (uint32_t(N >> 3) << 17) | (uint32_t(M >> 4) << 24);
}


// ------------------------------------------------------------------------------------ CTA pairs (cta_group::2)
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;   // clears the CTA-rank bit of a shared::cluster address -> rank 0

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t cluster_nctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_alloc_cg2(uint32_t* dst_smem, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish_cg2() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_cg2(uint32_t addr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
// both CTAs of the pair load their half of the tile; the transaction bytes land on CTA 0's mbarrier
__device__ __forceinline__ void tma_load_2d_cg2(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_load_3d_cg2(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
// the same, multicast: the box lands at the same offset in every CTA of cta_mask, and each destination's transaction
// bytes land on the mbarrier of that destination's pair leader (even rank)
__device__ __forceinline__ void tma_load_3d_cg2_mc(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1, int c2,
                                                   uint16_t cta_mask) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes.multicast::cluster"
      " [%0], [%1, {%3, %4, %5}], [%2], %6;"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1), "r"(c2), "h"(cta_mask)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tc_commit_cg2(uint64_t* bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"(cta_mask) : "memory");
}
// arrive on the mbarrier at the same offset in the shared memory of cluster CTA `rank`
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar, uint32_t rank) {
  asm volatile(
      "{\n\t.reg .b32 a;\n\t"
      "mapa.shared::cluster.u32 a, %0, %1;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [a];\n\t}"
      ::"r"(smem_u32(bar)), "r"(rank) : "memory");
}

// ------------------------------------------------------------------------------------ A operand in tensor memory
// D[tmem] (+)= A[tmem] * B[smem desc]^T, bf16 x bf16 -> fp32; A: lane = row, 16-bit elements packed 2 per column
__device__ __forceinline__ void umma_bf16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_bf16_ts_cg2(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// Predicated forms: `issue` is the elect_one() result of the calling lane.  The predicate travels INTO the asm
// (PTX @e) instead of wrapping the call in a C++ `if`, so the operand arithmetic stays in warp-uniform control
// flow and the compiler keeps descriptors / TMEM addresses in uniform registers.
__device__ __forceinline__ void umma_bf16_pred(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                               uint32_t accumulate, uint32_t issue) {
  asm volatile(
      "{\n\t.reg .pred p, e;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "setp.ne.b32 e, %5, 0;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(issue) : "memory");
}
// E4M3 x E4M3 -> fp32 (kind::f8f6f4, K = 32 per instruction: the same 32 bytes of a K-chunk as one bf16 MMA)
__device__ __forceinline__ void umma_e4m3_pred(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                               uint32_t accumulate, uint32_t issue) {
  asm volatile(
      "{\n\t.reg .pred p, e;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "setp.ne.b32 e, %5, 0;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(issue) : "memory");
}
__device__ __forceinline__ void umma_bf16_ts_pred(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                                  uint32_t accumulate, uint32_t issue) {
  asm volatile(
      "{\n\t.reg .pred p, e;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "setp.ne.b32 e, %5, 0;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(issue) : "memory");
}
__device__ __forceinline__ void umma_bf16_ts_cg2_pred(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc,
                                                      uint32_t idesc, uint32_t accumulate, uint32_t issue) {
  asm volatile(
      "{\n\t.reg .pred p, e;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "setp.ne.b32 e, %5, 0;\n\t"
      "@e tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(issue) : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t addr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
      ::"r"(addr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
        "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ------------------------------------------------------------------------------------ host: TMA descriptors
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static inline PFN_encodeTiled get_encode_fn() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess)
      return nullptr;
    fn = reinterpret_cast<PFN_encodeTiled>(p);
  }
  return fn;
}

// 2-D row-major [rows, cols] tensor, box = [box_rows, 128 bytes of cols], 128-byte swizzle: bf16 (64 cols) or, with
// e4m3, bytes (128 cols).
static inline int make_tensor_map_2d(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint32_t box_rows,
                       CUtensorMapL2promotion promo, bool e4m3 = false) {
  PFN_encodeTiled enc = get_encode_fn();
  if (!enc) return MFAR_ERR_CUDA;
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstride[1] = {cols * (e4m3 ? 1 : 2)};
  cuuint32_t box[2] = {cuuint32_t(e4m3 ? kChunkK8 : kChunkK), box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, e4m3 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    fprintf(stderr, "[mfar_b200] cuTensorMapEncodeTiled failed: %d\n", int(r));
    return MFAR_ERR_CUDA;
  }
  return MFAR_OK;
}


// 3-D "K-chunked" view of a bf16 row-major [rows, cols] tensor: dims (64 | rows | cols/64) with strides
// (2 B | cols*2 B | 128 B).  A box (64, box_rows, kc) lands in shared memory as kc consecutive
// [box_rows x 128 B] blocks, each 128-byte swizzled: exactly the K-major SWIZZLE_128B operand layout
// tcgen05.mma consumes, for kc*64 K-elements, with ONE TMA instruction.
static inline int make_tensor_map_kchunked(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols,
                                           uint32_t box_rows, uint32_t kc, CUtensorMapL2promotion promo) {
  PFN_encodeTiled enc = get_encode_fn();
  if (!enc) return MFAR_ERR_CUDA;
  cuuint64_t gdim[3] = {cuuint64_t(kChunkK), rows, cols / kChunkK};
  cuuint64_t gstride[2] = {cols * 2, cuuint64_t(kChunkK) * 2};
  cuuint32_t box[3] = {cuuint32_t(kChunkK), box_rows, kc};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), gdim, gstride, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    fprintf(stderr, "[mfar_b200] cuTensorMapEncodeTiled (k-chunked) failed: %d\n", int(r));
    return MFAR_ERR_CUDA;
  }
  return MFAR_OK;
}


// 3-D view of a [Q, n_sparse, ld] f16/f32 score tensor: dims (ld | n_sparse | Q), box = (128 bytes of docs, 1 field,
// box_q queries), 128-byte swizzled: the rows of one field for a tile of queries, one row per 128-byte line.
// Out-of-range docs / queries are zero-filled by the TMA unit.  Needs a 16-byte aligned base and row pitch.
// ld: row pitch in elements; cols <= ld: columns addressable from `base` (reads past them are zero-filled)
static inline int make_tensor_map_sparse_rows(CUtensorMap* map, const void* base, bool f16, uint64_t ld, uint64_t cols,
                                              uint32_t n_sparse, uint64_t Q, uint32_t box_q) {
  PFN_encodeTiled enc = get_encode_fn();
  if (!enc) return MFAR_ERR_CUDA;
  const uint64_t es = f16 ? 2 : 4;
  cuuint64_t gdim[3] = {cols, n_sparse, Q};
  cuuint64_t gstride[2] = {ld * es, ld * es * n_sparse};
  cuuint32_t box[3] = {cuuint32_t(128 / es), 1, box_q};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(map, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3,
                   const_cast<void*>(base), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    fprintf(stderr, "[mfar_b200] cuTensorMapEncodeTiled (sparse rows) failed: %d\n", int(r));
    return MFAR_ERR_CUDA;
  }
  return MFAR_OK;
}

}  // namespace mfar
