// Shared device helpers for the learning3d_b200 kernels (sm_100a only).
//
// Everything in this tree is compiled with -fmad=false: a*b+c is NEVER contracted
// behind our back.  Where the reference arithmetic is fused (MKL / cuBLAS K=3 GEMM,
// nvcc-contracted pointnet2 kernels) the kernels call fmaf() explicitly, so the
// rounding sequence of every distance is spelled out in the source and mirrored
// one-to-one by oracle/l3d_oracle.c.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <mutex>

#define L3D_FULL_MASK 0xffffffffu

// ---- error codes shared with include/l3d_b200.h ------------------------------------
#define L3D_OK 0
#define L3D_ERR_INVALID (-1)      // bad argument (null pointer, k > N, negative size ...)
#define L3D_ERR_UNSUPPORTED (-2)  // shape outside what the kernels were built for

#define L3D_LAUNCH_CHECK()                              \
  do {                                                  \
    cudaError_t e__ = cudaGetLastError();               \
    if (e__ != cudaSuccess) return (int)e__;            \
  } while (0)

namespace l3d {

// ---- host launch set-up ----------------------------------------------------------------
// Number of SMs of device `dev`, cached per host thread (148, a B200's count, if the query fails).
inline int sm_count(int dev) {
  static thread_local int c_dev = -1, c_n = 148;
  if (dev != c_dev) {
    int n = 0;
    c_n = (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0) ? n : 148;
    c_dev = dev;
  }
  return c_n;
}

// Opts kernel Kern in to `bytes` of dynamic shared memory on device `dev`, once per (kernel, device).  The
// attribute is shared by every host thread, so it is set under a process-wide lock and never lowered: a size
// per call would let a thread with a smaller problem lower it under a launch that still needs the larger one.
// Keyed by the kernel itself, not by its type (every kNN kernel is a void(KnnParams)).
template <auto Kern>
cudaError_t raise_smem_once(int dev, size_t bytes) {
  static std::mutex mu;
  static uint64_t done_mask = 0;   // bit = device ordinal (ordinals >= 64 set the attribute on every call)
  std::lock_guard<std::mutex> lock(mu);
  if (dev < 64 && (done_mask >> dev & 1)) return cudaSuccess;
  const cudaError_t e = cudaFuncSetAttribute(Kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e == cudaSuccess && dev < 64) done_mask |= (uint64_t)1 << dev;
  return e;
}

__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ int warp_id() { return threadIdx.x >> 5; }

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---- mbarrier + 1-D bulk async copy (TMA engine, SASS: UBLKCP) ---------------------
// A tensor-map (tiled) TMA box cannot express a 12-byte inner row, so point clouds are
// moved as flat 16-byte-aligned byte ranges with cp.async.bulk and an mbarrier.
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes,
                                         uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
          "r"(smem_u32(smem_dst)),
      "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "DONE:\n\t"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}

// ---- packed fp32 (sm_100 FFMA2 / FMUL2 / FADD2): two independent IEEE fp32 lanes per instruction, each
// rounded exactly like the scalar op, so a key computed in a packed lane is bit-identical to knn_key<>.
__device__ __forceinline__ unsigned long long f2_pack(float lo, float hi) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void f2_unpack(unsigned long long v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ unsigned long long f2_mul(unsigned long long a, unsigned long long b) {
  unsigned long long d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ unsigned long long f2_fma(unsigned long long a, unsigned long long b, unsigned long long c) {
  unsigned long long d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
// NOTE (measured on ptxas 12.9): a packed multiply feeding a packed add IS contracted into FFMA2 even with explicit
// .rn on both instructions and -fmad=false, and fma(a, b, -0) is first simplified back to a multiply.  Code that
// needs separately rounded products (Chamfer's (dx*dx + dy*dy) + dz*dz) therefore stays scalar; the packed helpers
// are only used where the reference arithmetic itself is an fma chain (kNN expansion keys, EMD distances).
__device__ __forceinline__ unsigned long long f2_add(unsigned long long a, unsigned long long b) {
  unsigned long long d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
// ---- ordering used by every selection kernel ---------------------------------------
// "better" = larger key first; equal keys -> lower index first.  All kNN flavours map
// their distance to a key whose LARGEST values are the nearest neighbours, so one
// comparator serves knn(), knn_point(), pointnet2 knn / three_nn and Chamfer's argmin.
__device__ __forceinline__ bool better(float av, uint32_t ai, float bv, uint32_t bi) {
  return (av > bv) || (av == bv && ai < bi);
}

// Bitonic sort of 32*S (key, idx) pairs held S-per-lane; position p = s*32 + lane.
// After the call position 0 holds the best pair, position 32*S-1 the worst.
template <int S>
__device__ __forceinline__ void warp_bitonic_sort(float (&v)[S], uint32_t (&ix)[S], int lane) {
  constexpr int NTOT = 32 * S;
#pragma unroll
  for (int k2 = 2; k2 <= NTOT; k2 <<= 1) {
#pragma unroll
    for (int j = k2 >> 1; j > 0; j >>= 1) {
      if (j >= 32) {
        const int js = j >> 5;
#pragma unroll
        for (int s = 0; s < S; ++s) {
          const int sp = s ^ js;
          if (sp > s) {
            const bool up = (((s * 32) & k2) == 0);  // lane bits < 32 <= k2 never matter here
            const bool b = better(v[sp], ix[sp], v[s], ix[s]);
            if (b == up) {
              float tv = v[s]; v[s] = v[sp]; v[sp] = tv;
              uint32_t ti = ix[s]; ix[s] = ix[sp]; ix[sp] = ti;
            }
          }
        }
      } else {
#pragma unroll
        for (int s = 0; s < S; ++s) {
          const float pv = __shfl_xor_sync(L3D_FULL_MASK, v[s], j);
          const uint32_t pi = __shfl_xor_sync(L3D_FULL_MASK, ix[s], j);
          const int p = s * 32 + lane;
          const bool up = ((p & k2) == 0);
          const bool lower = ((lane & j) == 0);
          const bool pb = better(pv, pi, v[s], ix[s]);
          const bool take = (pb == (lower == up));
          v[s] = take ? pv : v[s];
          ix[s] = take ? pi : ix[s];
        }
      }
    }
  }
}

// Keys-only descending bitonic sort of 32*S floats (position p = s*32 + lane).
template <int S>
__device__ __forceinline__ void warp_bitonic_sort_keys(float (&v)[S], int lane) {
  constexpr int NTOT = 32 * S;
#pragma unroll
  for (int k2 = 2; k2 <= NTOT; k2 <<= 1) {
#pragma unroll
    for (int j = k2 >> 1; j > 0; j >>= 1) {
      if (j >= 32) {
        const int js = j >> 5;
#pragma unroll
        for (int s = 0; s < S; ++s) {
          const int sp = s ^ js;
          if (sp > s) {
            const bool up = (((s * 32) & k2) == 0);
            const float hi = fmaxf(v[s], v[sp]);
            const float lo = fminf(v[s], v[sp]);
            v[s] = up ? hi : lo;
            v[sp] = up ? lo : hi;
          }
        }
      } else {
#pragma unroll
        for (int s = 0; s < S; ++s) {
          const float pv = __shfl_xor_sync(L3D_FULL_MASK, v[s], j);
          const int p = s * 32 + lane;
          const bool up = ((p & k2) == 0);
          const bool lower = ((lane & j) == 0);
          v[s] = (lower == up) ? fmaxf(v[s], pv) : fminf(v[s], pv);
        }
      }
    }
  }
}

// ---- second-generation selection network (v2) ----------------------------------------------
// A (key, index) pair is packed into ONE 64-bit composite whose unsigned order is the selection
// order: high word = order-preserving image of the fp32 key, low word = ~index (lower index ->
// larger composite).  All-zero is the sentinel (worse than any real pair).  One comparison per
// exchange instead of three, and a sorting network in which every exchange has the same
// direction rule ("the lower lane keeps the larger composite"): the classic flip + half-cleaner
// bitonic merger, so a stage is 2 SHFL + 2 ISETP + 1 PLOP3 + 2 SEL.
__device__ __forceinline__ uint32_t f32_order(float f) {
  const uint32_t u = __float_as_uint(f);
  return u ^ ((uint32_t)((int32_t)u >> 31) | 0x80000000u);
}
__device__ __forceinline__ float f32_unorder(uint32_t o) {
  const uint32_t u = (o & 0x80000000u) ? (o ^ 0x80000000u) : ~o;
  return __uint_as_float(u);
}
__device__ __forceinline__ unsigned long long pack_pair(float key, uint32_t idx) {
  // key + 0.0f folds -0.0 into +0.0 so that equal keys always produce equal high words
  return ((unsigned long long)f32_order(key + 0.0f) << 32) | (unsigned long long)(~idx);
}
__device__ __forceinline__ unsigned long long shfl_u64(unsigned long long v, int src) {
  const uint32_t lo = __shfl_sync(L3D_FULL_MASK, (uint32_t)v, src);
  const uint32_t hi = __shfl_sync(L3D_FULL_MASK, (uint32_t)(v >> 32), src);
  return ((unsigned long long)hi << 32) | lo;
}
__device__ __forceinline__ unsigned long long shfl_xor_u64(unsigned long long v, int m) {
  const uint32_t lo = __shfl_xor_sync(L3D_FULL_MASK, (uint32_t)v, m);
  const uint32_t hi = __shfl_xor_sync(L3D_FULL_MASK, (uint32_t)(v >> 32), m);
  return ((unsigned long long)hi << 32) | lo;
}
// exchange with lane ^ m; the lane whose `bit` of the lane id is clear keeps the larger composite
__device__ __forceinline__ unsigned long long cmpx_u64(unsigned long long c, int m, bool keep_big) {
  const unsigned long long o = shfl_xor_u64(c, m);
  return ((o > c) == keep_big) ? o : c;
}
// Sort 32 composites (one per lane) descending: lane 0 ends with the largest.
__device__ __forceinline__ unsigned long long warp_sort32_desc(unsigned long long c, int lane) {
#pragma unroll
  for (int k2 = 2; k2 <= 32; k2 <<= 1) {
    c = cmpx_u64(c, k2 - 1, (lane & (k2 >> 1)) == 0);          // flip
#pragma unroll
    for (int j = k2 >> 2; j > 0; j >>= 1) c = cmpx_u64(c, j, (lane & j) == 0);   // half-cleaners
  }
  return c;
}
// R independent 32-wide sorts interleaved stage by stage (ILP across rows).
template <int R>
__device__ __forceinline__ void warp_sort32_desc_x(unsigned long long (&c)[R], int lane) {
#pragma unroll
  for (int k2 = 2; k2 <= 32; k2 <<= 1) {
    const bool kb = (lane & (k2 >> 1)) == 0;
#pragma unroll
    for (int r = 0; r < R; ++r) c[r] = cmpx_u64(c[r], k2 - 1, kb);
#pragma unroll
    for (int j = k2 >> 2; j > 0; j >>= 1) {
      const bool kj = (lane & j) == 0;
#pragma unroll
      for (int r = 0; r < R; ++r) c[r] = cmpx_u64(c[r], j, kj);
    }
  }
}
// Largest 32 of 64 composites (two per lane), sorted descending into one register per lane.
__device__ __forceinline__ unsigned long long warp_top32_of64(unsigned long long a, unsigned long long b,
                                                                int lane) {
#pragma unroll
  for (int k2 = 2; k2 <= 32; k2 <<= 1) {
    const bool kb = (lane & (k2 >> 1)) == 0;
    a = cmpx_u64(a, k2 - 1, kb);
    b = cmpx_u64(b, k2 - 1, kb);
#pragma unroll
    for (int j = k2 >> 2; j > 0; j >>= 1) {
      const bool kj = (lane & j) == 0;
      a = cmpx_u64(a, j, kj);
      b = cmpx_u64(b, j, kj);
    }
  }
  const unsigned long long br = shfl_xor_u64(b, 31);   // b reversed: pairs a[i] with b[31-i]
  unsigned long long c = (br > a) ? br : a;             // bitonic sequence holding the best 32
#pragma unroll
  for (int j = 16; j > 0; j >>= 1) c = cmpx_u64(c, j, (lane & j) == 0);
  return c;
}
// Keys-only descending sort of 32 floats with the same uniform-direction network.
__device__ __forceinline__ float warp_sort32_keys_desc(float v, int lane) {
#pragma unroll
  for (int k2 = 2; k2 <= 32; k2 <<= 1) {
    {
      const float o = __shfl_xor_sync(L3D_FULL_MASK, v, k2 - 1);
      v = ((lane & (k2 >> 1)) == 0) ? fmaxf(v, o) : fminf(v, o);
    }
#pragma unroll
    for (int j = k2 >> 2; j > 0; j >>= 1) {
      const float o = __shfl_xor_sync(L3D_FULL_MASK, v, j);
      v = ((lane & j) == 0) ? fmaxf(v, o) : fminf(v, o);
    }
  }
  return v;
}

// R independent keys-only sorts, interleaved stage by stage (their shuffle latencies overlap)
template <int R>
__device__ __forceinline__ void warp_sort32_keys_desc_x(float (&v)[R], int lane) {
#pragma unroll
  for (int k2 = 2; k2 <= 32; k2 <<= 1) {
    const bool kb = (lane & (k2 >> 1)) == 0;
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const float o = __shfl_xor_sync(L3D_FULL_MASK, v[r], k2 - 1);
      v[r] = kb ? fmaxf(v[r], o) : fminf(v[r], o);
    }
#pragma unroll
    for (int j = k2 >> 2; j > 0; j >>= 1) {
      const bool kj = (lane & j) == 0;
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const float o = __shfl_xor_sync(L3D_FULL_MASK, v[r], j);
        v[r] = kj ? fmaxf(v[r], o) : fminf(v[r], o);
      }
    }
  }
}

__device__ __forceinline__ int warp_inclusive_scan(int x, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(L3D_FULL_MASK, x, o);
    if (lane >= o) x += y;
  }
  return x;
}

}  // namespace l3d
