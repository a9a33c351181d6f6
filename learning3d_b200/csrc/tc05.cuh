// tcgen05 / TMEM / TMA / mbarrier PTX wrappers shared by the tensor-core kernels (softcorr.cu, edgeconv.cu).
// sm_100a only.  Every mbarrier wait is bounded (SC_SPIN_LIMIT polls): a protocol bug surfaces as an error
// word, never as a hung GPU.
#pragma once
#include "common.cuh"

#include <cuda.h>

namespace l3d {

constexpr int SC_BM = 128;                 // rows per CTA (UMMA M)
constexpr int SC_UK = 8;                   // UMMA K for kind::tf32 (32 bytes)
constexpr uint32_t SC_SPIN_LIMIT = 1u << 22;

// ---- PTX wrappers ---------------------------------------------------------------------------
__device__ __forceinline__ bool mbar_wait_bounded(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
#pragma unroll 1
  for (uint32_t spin = 0; spin < SC_SPIN_LIMIT; ++spin) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(addr), "r"(parity)
        : "memory");
    if (ok) return true;
  }
  return false;
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// ---- CTA-pair (cluster of 2) variants -----------------------------------------------------------
// wait on a barrier whose phase is completed by arrivals from the peer CTA as well (same PTX as the
// CTA-local wait, like cutlass::arch::ClusterBarrier::wait; kept separate to mark the cross-CTA sites)
__device__ __forceinline__ bool mbar_wait_bounded_cluster(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
#pragma unroll 1
  for (uint32_t spin = 0; spin < SC_SPIN_LIMIT; ++spin) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(addr), "r"(parity)
        : "memory");
    if (ok) return true;
  }
  return false;
}
// arrive on the barrier at the same shared-memory offset in CTA `rank` of the cluster.  Default semantics, as
// cutlass::arch::ClusterBarrier::arrive(cta_id): the writes it publishes were already forced into shared memory
// by fence.proxy.async; an explicit .release.cluster here stalled every splitter warp ~1.5k cycles per stage
// (266 us vs 152 us for the C3 kernel).
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar, uint32_t rank) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}"
      ::"r"(smem_u32(bar)), "r"(rank)
      : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tc_commit_pair(uint64_t* bar) {   // arrives on the barrier in BOTH CTAs
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"((unsigned short)3)
      : "memory");
}
__device__ __forceinline__ void tc_mma_tf32_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                                 uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tc_mma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                            uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// 32 lanes x 32 consecutive fp32 columns: thread t of the warp reads TMEM lane (warp%4)*32 + t
__device__ __forceinline__ void tc_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]),
        "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]),
        "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]),
        "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// tf32 rounding (nearest, ties away) on the bit pattern: two integer instructions
__device__ __forceinline__ uint32_t rna_tf32_bits(uint32_t u) { return (u + 0x1000u) & 0xffffe000u; }

__device__ __forceinline__ void sts128(uint32_t saddr, uint4 v) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)
               : "memory");
}
__device__ __forceinline__ uint4 lds128(uint32_t saddr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(saddr)
               : "memory");
  return v;
}
__device__ __forceinline__ void tma_load_3d(uint32_t smem_dst, const CUtensorMap* tmap, int c0, int c1, int c2,
                                            uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_dst), "l"(tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

// 4-D variant for the chunked view of make_dn_tmap4 (coordinates: n inside the 32-chunk, channel, chunk, item)
__device__ __forceinline__ void tma_load_4d(uint32_t smem_dst, const CUtensorMap* tmap, int c0, int c1, int c2, int c3,
                                            uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_dst), "l"(tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

// L2 prefetch of one box (no shared memory, no barrier): hides HBM latency for tiles further ahead than the
// shared-memory ring can hold (SASS: UTMAPF.L2)

// Shared-memory matrix descriptors (cute::UMMA::SmemDescriptor, sm_100 "version 1"), SWIZZLE_128B.
//   K-major  (generic path): rows of 32 fp32 (128 B), 8-row groups 1024 B apart (SBO).
//   MN-major (TMA path): 128 B of n per channel row, 8-channel groups 1024 B apart (SBO), the next
//            32 points 4096 B further (LBO).
__device__ __forceinline__ uint64_t sc_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                             uint32_t layout_type) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);       // start address            bits [0,14)
  d |= (uint64_t)(lbo_bytes >> 4) << 16;           // leading byte offset      bits [16,30)
  d |= (uint64_t)(sbo_bytes >> 4) << 32;           // stride byte offset       bits [32,46)
  d |= (uint64_t)1 << 46;                          // descriptor version 1     bits [46,48)
  d |= (uint64_t)layout_type << 61;                // 2 = SWIZZLE_128B, 1 = SWIZZLE_128B_BASE32B
  return d;
}
// instruction descriptor (cute::UMMA::InstrDescriptor): D = F32, A = B = TF32, M = 128, N = bn;
// mn_major sets a_major = b_major = MN
__host__ __device__ constexpr uint32_t sc_idesc(int bn, bool mn_major, int m = SC_BM) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(bn >> 3) << 17) | ((uint32_t)(m >> 4) << 24) |
         (mn_major ? ((1u << 15) | (1u << 16)) : 0u);
}

// ---- host: cuTensorMapEncodeTiled through the runtime's driver entry point (no -lcuda) -----------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)f;
  }
  return fn;
}

// fp32 tensor [B, D, N] (n fastest) as a 3-D map; boxes of 32 n x box_d channels, SWIZZLE_128B_ATOM_32B
// (= UMMA layout 1, the MN-major tf32 operand layout); out-of-range elements read as 0
inline bool make_dn_tmap(CUtensorMap* m, const float* base, int B, int D, int N, int box_d) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn) return false;
  cuuint64_t dims[3] = {(cuuint64_t)N, (cuuint64_t)D, (cuuint64_t)B};
  cuuint64_t strides[2] = {(cuuint64_t)N * 4, (cuuint64_t)N * (cuuint64_t)D * 4};
  cuuint32_t box[3] = {32, (cuuint32_t)box_d, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  return fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, (void*)base, dims, strides, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// The same tensor seen as [B, N/32, D, 32] (N % 32 == 0): dims (n_in = 32, d, chunk = n / 32, b) with strides
// (4, 4N, 128, 4ND) bytes.  One box of (32, box_d, chunks, 1) lands in shared memory as `chunks` consecutive
// [box_d x 32] atoms — byte for byte what `chunks` separate make_dn_tmap boxes at 32-point steps produce — so a whole
// operand tile is ONE bulk-tensor instruction instead of 4-8 (the per-instruction cost of the TMA unit, not L2 or HBM
// bandwidth, is what bounded the pipelines: profiles/r02/README.md).  Chunks beyond N/32 and channels beyond D read 0.
inline bool make_dn_tmap4(CUtensorMap* m, const float* base, int B, int D, int N, int box_d, int chunks) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn || (N & 31) || chunks < 1 || chunks > 256) return false;
  cuuint64_t dims[4] = {32, (cuuint64_t)D, (cuuint64_t)(N / 32), (cuuint64_t)B};
  cuuint64_t strides[3] = {(cuuint64_t)N * 4, 128, (cuuint64_t)N * (cuuint64_t)D * 4};
  cuuint32_t box[4] = {32, (cuuint32_t)box_d, (cuuint32_t)chunks, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  return fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (void*)base, dims, strides, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace l3d
