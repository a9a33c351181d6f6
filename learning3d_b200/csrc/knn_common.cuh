// Shared pieces of the kNN kernels (knn.cu: warp-per-row-pair selection, knn_tpr.cu: thread-per-row selection).
#pragma once
#include "common.cuh"
#include "launch_count.h"

namespace l3d {

constexpr size_t KNN_SMEM_LIMIT = 227 * 1024;   // opt-in dynamic shared memory per CTA on sm_100

enum KnnMode {
  MODE_EXPANSION_NEG = 0,  // key = ((-|c|^2) + 2 q.c) - |q|^2              (largest = nearest)
  MODE_SQDIST_EXP = 1,     // key = -(((-2 q.c) + |q|^2) + |c|^2)
  MODE_DIRECT_RN = 2,      // key = -((dx*dx + dy*dy) + dz*dz), each op rounded
  MODE_DIRECT_FMA = 3      // key = -fma(dz,dz, fma(dx,dx, dy*dy))  (nvcc's contraction, see below)
};

struct KnnParams {
  const float* cand;   // [B,3,N] (CAND_BCN) or [B,N,3]
  const float* query;  // [B,M,3] or nullptr when SELF
  void* out_idx;       // [B,M,k] int64 / int32
  float* out_val;      // optional [B,M,k]
  float* feat_out;     // optional [B,6,N,k] graph feature (knn() on xyz only: SELF, [B,3,N] input)
  int B, N, M, k;
  int idx64;      // 1 -> int64 indices, 0 -> int32, 2 -> uint16 (host-buffer path: narrow on the PCIe wire)
  int val_xform;  // 0: key, 1: -key, 2: sqrt(-key)
  int use_tma;    // alignment preconditions for cp.async.bulk hold
  int force_slow;
  int full_sort;  // N <= KNN_SORT_MAX_N and k is a large fraction of N: sort the whole row
};

template <int MODE>
__device__ __forceinline__ float knn_key(const float4 q, const float4 c) {
  if (MODE == MODE_EXPANSION_NEG) {
    // torch.matmul K=3 accumulation: fma(z,z', fma(y,y', x*x'))  (model_common_utils.py:5)
    const float dot = fmaf(q.z, c.z, fmaf(q.y, c.y, __fmul_rn(q.x, c.x)));
    // pd = -xx - inner - xx^T, inner = -2*dot (exact): ((-|c|^2) + 2dot) - |q|^2   (:6-7)
    return __fsub_rn(fmaf(2.0f, dot, -c.w), q.w);
  } else if (MODE == MODE_SQDIST_EXP) {
    const float dot = fmaf(q.z, c.z, fmaf(q.y, c.y, __fmul_rn(q.x, c.x)));
    // dist = -2*matmul; dist += |src|^2; dist += |dst|^2   (pointconv_util.py:36-38)
    const float v = __fadd_rn(fmaf(-2.0f, dot, q.w), c.w);
    return -v;
  } else if (MODE == MODE_DIRECT_RN) {
    const float dx = __fsub_rn(c.x, q.x), dy = __fsub_rn(c.y, q.y), dz = __fsub_rn(c.z, q.z);
    const float v = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
    return -v;
  } else {
    const float dx = __fsub_rn(q.x, c.x), dy = __fsub_rn(q.y, c.y), dz = __fsub_rn(q.z, c.z);
    // nvcc (12.9, -O2, sm_100) compiles the reference's `dx*dx + dy*dy + dz*dz`
    // (interpolate_gpu.cu:38,104) to FMUL(dy,dy); FFMA(dx,dx,.); FFMA(dz,dz,.) — checked in the
    // SASS of the reference file itself (oracle/README.md).
    const float v = fmaf(dz, dz, fmaf(dx, dx, __fmul_rn(dy, dy)));
    return -v;
  }
}

template <int MODE>
__device__ __forceinline__ float4 knn_pack(float x, float y, float z) {
  float w = 0.0f;
  if (MODE == MODE_EXPANSION_NEG || MODE == MODE_SQDIST_EXP)
    w = __fadd_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)), __fmul_rn(z, z));  // sum(x**2)
  return make_float4(x, y, z, w);
}

template <int MODE>
__device__ __forceinline__ float4 knn_padding() {
  // a padded slot must evaluate to key = -inf for every finite query
  if (MODE == MODE_EXPANSION_NEG || MODE == MODE_SQDIST_EXP)
    return make_float4(0.f, 0.f, 0.f, INFINITY);
  return make_float4(INFINITY, INFINITY, INFINITY, 0.f);
}

__device__ __forceinline__ void knn_store_index(const KnnParams& p, long o, uint32_t ix) {
  if (p.idx64 == 1) reinterpret_cast<long long*>(p.out_idx)[o] = (long long)ix;
  else if (p.idx64 == 0) reinterpret_cast<int*>(p.out_idx)[o] = (int)ix;
  else reinterpret_cast<unsigned short*>(p.out_idx)[o] = (unsigned short)ix;
}

__device__ __forceinline__ float knn_val_xform(float key, int xform) {
  // 0 - key (not -key): a zero distance comes out as +0.0 like the reference's
  if (xform == 1) return 0.0f - key;
  if (xform == 2) return sqrtf(0.0f - key);
  return key;
}

// Exact but O(k*N) selection: k rounds of "best pair strictly after the previous one".
template <int MODE>
__device__ __noinline__ void knn_row_slow(const KnnParams& p, const float4* __restrict__ packed,
                                          const float4 q, long row, int lane) {
  float pv = INFINITY;
  uint32_t pi = 0;
  bool first = true;
  for (int r = 0; r < p.k; ++r) {
    float bv = -INFINITY;
    uint32_t bi = 0xffffffffu;
    for (int j = lane; j < p.N; j += 32) {
      const float d = knn_key<MODE>(q, packed[j]);
      const bool after = first || better(pv, pi, d, (uint32_t)j);
      if (after && better(d, (uint32_t)j, bv, bi)) { bv = d; bi = (uint32_t)j; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(L3D_FULL_MASK, bv, o);
      const uint32_t oi = __shfl_xor_sync(L3D_FULL_MASK, bi, o);
      if (better(ov, oi, bv, bi)) { bv = ov; bi = oi; }
    }
    if (lane == 0) {
      const long o = row * p.k + r;
      knn_store_index(p, o, bi);
      if (p.out_val) p.out_val[o] = knn_val_xform(bv, p.val_xform);
    }
    pv = bv; pi = bi; first = false;
  }
}

constexpr int KNN_TILE = 1024;   // candidates per tile = 32 lanes x 32 registers

// ---- v2 row routine ---------------------------------------------------------------------------
// Same algorithm as knn_row, re-engineered after the first ncu capture (profiles/r01): the
// count / compaction pass kept 32 predicates alive in a bit-packed register (~400 LOP3/ISETP/VIADD
// per row).  Here the survivors of a lane are a 32-bit mask built once (FSETP + predicated OR),
// counted with POPC, and written by a short loop over the set bits that RE-EVALUATES the key
// from shared memory (registers cannot be indexed dynamically; same inputs, same instructions ->
// the same bits).  Survivors are stored as 64-bit composites and sorted with the uniform-direction
// network of common.cuh.  KS = 1 keeps everything in one or two registers per lane.
__device__ __forceinline__ void knn_store_packed(const KnnParams& p, long row, int pos,
                                                 unsigned long long c) {
  if (pos < p.k) {
    const long o = row * p.k + pos;
    const uint32_t ix = ~(uint32_t)c;
    knn_store_index(p, o, ix);
    if (p.out_val) p.out_val[o] = knn_val_xform(f32_unorder((uint32_t)(c >> 32)), p.val_xform);
  }
}

template <int MODE>
__device__ __forceinline__ void knn_row_v2(const KnnParams& p, const float4* __restrict__ packed,
                                           unsigned long long* __restrict__ cbuf, const float4 q,
                                           long row, int ntiles, int lane) {
  constexpr int CAP = 64;
  const int k = p.k;            // k <= 24 on this path
  int base = 0;                 // composites carried over from earlier tiles (running top-k)
  float kth = -INFINITY;
  bool overflow = (p.force_slow != 0);
  unsigned long long best = 0ull;   // lane l holds the l-th best composite after each tile

  for (int t = 0; t < ntiles && !overflow; ++t) {
    float d[32];
    const float4* pt = packed + t * KNN_TILE + lane;
#pragma unroll
    for (int e = 0; e < 32; ++e) d[e] = knn_key<MODE>(q, pt[e * 32]);

    float m = d[0];
#pragma unroll
    for (int e = 1; e < 32; ++e) m = fmaxf(m, d[e]);
    // k-th largest lane maximum: at least k keys of the tile are >= t0
    const float t0 = __shfl_sync(L3D_FULL_MASK, warp_sort32_keys_desc(m, lane), k - 1);
    const float thr = fmaxf(t0, kth);

    uint32_t mask = 0u;
#pragma unroll
    for (int e = 0; e < 32; ++e) mask |= (d[e] >= thr) ? (1u << e) : 0u;
    const int cnt = __popc(mask);
    const int incl = warp_inclusive_scan(cnt, lane);
    const int total = __shfl_sync(L3D_FULL_MASK, incl, 31);
    if (base + total > CAP) { overflow = true; break; }

    if (base) {   // running top-k of the previous tiles goes first
      if (lane < base) cbuf[lane] = best;
    }
    int off = base + incl - cnt;
    while (mask) {
      const int e = __ffs(mask) - 1;
      mask &= mask - 1;
      const int j = t * KNN_TILE + e * 32 + lane;
      cbuf[off++] = pack_pair(knn_key<MODE>(q, packed[j]), (uint32_t)j);
    }
    __syncwarp();
    const int n_in = base + total;
    const unsigned long long a = (lane < n_in) ? cbuf[lane] : 0ull;
    if (n_in <= 32) {
      best = warp_sort32_desc(a, lane);
    } else {
      const unsigned long long b = (lane + 32 < n_in) ? cbuf[lane + 32] : 0ull;
      best = warp_top32_of64(a, b, lane);
    }
    __syncwarp();
    if (t + 1 < ntiles) {
      const uint32_t kw = __shfl_sync(L3D_FULL_MASK, (uint32_t)(best >> 32), k - 1);
      kth = f32_unorder(kw);
      base = k;
    }
  }

  if (overflow) knn_row_slow<MODE>(p, packed, q, row, lane);
  else knn_store_packed(p, row, lane, best);
}

// Launches a kNN kernel with programmatic dependent launch: the next launch on the stream may start filling SMs as
// this one's CTAs retire (the kernels run griddepcontrol.wait before they touch global memory).
inline int knn_launch_pdl(void (*kern)(KnnParams), long grid, int threads, size_t smem, cudaStream_t stream,
                          const KnnParams& p) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  const cudaError_t le = cudaLaunchKernelEx(&cfg, kern, p);
  if (le != cudaSuccess) return (int)le;
  count_launch();
  L3D_LAUNCH_CHECK();
  return L3D_OK;
}

// knn_tpr.cu: thread-per-row kernel for knn() on xyz clouds (k <= 24, N % 32 == 0, N <= 2048)
bool knn_tpr_eligible(const KnnParams& p);
int knn_tpr_launch(const KnnParams& p, cudaStream_t stream);
int knn_path_flag();   // l3d_debug_knn_path: 0 auto, 1 warp kernel only, 2 thread-per-row whenever eligible

}  // namespace l3d
