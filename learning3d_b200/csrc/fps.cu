// Farthest point sampling (sm_100a).
//
// Replaces furthest_point_sampling_kernel (utils/lib/src/sampling_gpu.cu:93-209, K10) and the three
// pure-torch loops farthest_point_sample (utils/model_common_utils.py:58-82,
// utils/pointconv_util.py:60-83, utils/ppfnet_util.py:71-93: `npoint` iterations of ~6 tiny kernels).
//
// FPS is inherently sequential (npoint dependent rounds), so it is latency bound: one CTA per batch
// item keeps every point and its running min-distance in REGISTERS for the whole run, and a round
// costs one distance update per register, one REDUX (__reduce_max_sync) warp arg-max on the distance
// bits plus a tie-key pass, ONE __syncthreads (double-buffered per-warp results) and a redundant
// per-warp final reduce — no global-memory traffic inside the loop at all: the coordinates of the newly
// selected point come from a shared-memory copy of the cloud (12 bytes, LDS broadcast).
//
// Selection semantics reproduced exactly (indices are bit-identical on tie-free AND tied inputs):
//   mode 0 (pointnet2 CUDA): d = nvcc-contracted fma form; per-thread strict '>' over k = tid, tid+bs, ...;
//           tree reduce keeps the LEFT (lower tid) entry on ties (sampling_gpu.cu:86-91,136-137):
//           the tree pairs tid with tid+stride for stride = bs/2 .. 1, so among equal distances the winner
//           is the smallest (bit-reversed (k mod bs) over log2 bs bits, then k), bs = the reference's
//           block size 2^floor(log2 n) <= 1024 (cuda_utils.h:10-14) — oracle/l3d_oracle_group.c simulates
//           the tree literally and the two agree on lattice clouds (tests/test_gpu_fuzz.py);
//   mode 1 (torch): d = (dx*dx + dy*dy) + dz*dz rounded; torch.max returns the first maximal index.
#include "common.cuh"
#include "../../include/l3d_b200.h"
#include "launch_count.h"

#include <cmath>

namespace l3d {

constexpr int FPS_THREADS = 512;
constexpr int FPS_WARPS = FPS_THREADS / 32;

struct FpsParams {
  const float* xyz;          // [B,N,3]
  float* temp;               // optional [B,N] in/out running min distance (pointnet2 `temp`)
  const long long* start;    // optional [B] start indices (torch random-start variants)
  void* out;                 // [B,M] int32 / int64
  int B, N, M;
  int mode;                  // 0: pointnet2 CUDA, 1: torch
  int idx64;
  int ref_bs;                // the reference kernel's block size (tie rule of mode 0)
  int ref_log2;              // log2(ref_bs)
};

__device__ __forceinline__ float fps_dist(int mode, float x, float y, float z, float cx, float cy,
                                          float cz) {
  const float dx = __fsub_rn(x, cx), dy = __fsub_rn(y, cy), dz = __fsub_rn(z, cz);
  if (mode == 0) return fmaf(dz, dz, fmaf(dx, dx, __fmul_rn(dy, dy)));           // sampling_gpu.cu:131
  return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));  // torch sum
}

// larger distance wins; equal distance -> smaller tie key wins
__device__ __forceinline__ bool fps_better(float av, uint32_t at, float bv, uint32_t bt) {
  return (av > bv) || (av == bv && at < bt);
}

template <int PPT>
__global__ void __launch_bounds__(FPS_THREADS) fps_kernel(const FpsParams p) {
  __shared__ uint2 s_r[2][FPS_WARPS];   // per-warp (max distance bits, ~tiekey), double-buffered
  // The cloud also lives in shared memory: every round starts by reading the coordinates of the point
  // selected by the previous one — a dependent access on the critical path of all N-1 rounds.  From
  // global memory (a line this SM never touched through that path: an L2 round trip) a round took ~990
  // cycles; an LDS broadcast is ~30.
  extern __shared__ float s_xyz[];

  const int b = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int N = p.N, M = p.M;
  const float* gxyz = p.xyz + (size_t)b * N * 3;
  for (int i = tid; i < 3 * N; i += FPS_THREADS) s_xyz[i] = gxyz[i];
  __syncthreads();
  const float* xyz = s_xyz;

  float px[PPT], py[PPT], pz[PPT], td[PPT];
  uint32_t tk[PPT];
#pragma unroll
  for (int i = 0; i < PPT; ++i) {
    const int k = tid + i * FPS_THREADS;
    if (k < N) {
      px[i] = xyz[k * 3]; py[i] = xyz[k * 3 + 1]; pz[i] = xyz[k * 3 + 2];
      td[i] = p.temp ? p.temp[(size_t)b * N + k] : 1e10f;
      // tie key: mode 1 orders by k.  Mode 0: the reference's smem tree (strides bs/2 .. 1, left
      // entry kept on ties) prefers the thread whose id is smallest when read BIT-REVERSED over
      // log2(bs) bits (stride 1 decides between even/odd tids last, i.e. bit 0 is most significant),
      // and inside a thread the smallest k: key = (bitrev(k mod bs), k / bs).
      if (p.mode == 0) {
        const uint32_t r = (p.ref_log2 == 0) ? 0u : (__brev((uint32_t)(k % p.ref_bs)) >> (32 - p.ref_log2));
        tk[i] = (r << 16) | (uint32_t)(k / p.ref_bs);
      } else {
        tk[i] = (uint32_t)k;
      }
    } else {
      px[i] = py[i] = pz[i] = 0.f;
      td[i] = 0.f;             // padding: smallest distance and the worst tie key -> never preferred
      tk[i] = 0xffffffffu;
    }
  }

  int old = p.start ? (int)p.start[b] : 0;
  if (tid == 0) {
    if (p.idx64) reinterpret_cast<long long*>(p.out)[(size_t)b * M] = old;
    else reinterpret_cast<int*>(p.out)[(size_t)b * M] = old;
  }

  for (int j = 1; j < M; ++j) {
    const float cx = xyz[old * 3], cy = xyz[old * 3 + 1], cz = xyz[old * 3 + 2];   // LDS broadcast
    // Distances are >= +0, so their bit patterns order like unsigned integers: the arg-max is two
    // hardware warp reductions (REDUX.MAX.U32) — first the distance bits, then ~tiekey among the
    // lanes that hold the maximum — instead of a 5-step shuffle butterfly over three values.
    uint32_t bv = 0u, bt = 0xffffffffu;
#pragma unroll
    for (int i = 0; i < PPT; ++i) {
      const int k = tid + i * FPS_THREADS;
      if (k < N) {
        const float d = fps_dist(p.mode, px[i], py[i], pz[i], cx, cy, cz);
        td[i] = fminf(d, td[i]);          // d2 = min(d, temp[k])  /  distance[mask] = dist[mask]
      }
      const uint32_t u = __float_as_uint(td[i]);
      if (u > bv || (u == bv && tk[i] < bt)) { bv = u; bt = tk[i]; }
    }
    uint32_t wv = __reduce_max_sync(L3D_FULL_MASK, bv);
    uint32_t wc = __reduce_max_sync(L3D_FULL_MASK, (bv == wv) ? ~bt : 0u);
    const int buf = j & 1;
    if (lane == 0) s_r[buf][warp] = make_uint2(wv, wc);
    __syncthreads();
    // every warp reduces the FPS_WARPS partial winners redundantly: no second barrier
    const uint2 e = (lane < FPS_WARPS) ? s_r[buf][lane] : make_uint2(0u, 0u);
    wv = __reduce_max_sync(L3D_FULL_MASK, e.x);
    wc = __reduce_max_sync(L3D_FULL_MASK, (e.x == wv) ? e.y : 0u);
    const uint32_t wtk = ~wc;
    if (p.mode == 0) {
      const uint32_t r = (p.ref_log2 == 0) ? 0u : (__brev(wtk >> 16) >> (32 - p.ref_log2));
      old = (int)((wtk & 0xffffu) * (uint32_t)p.ref_bs + r);
    } else {
      old = (int)wtk;
    }
    if (tid == 0) {
      if (p.idx64) reinterpret_cast<long long*>(p.out)[(size_t)b * M + j] = old;
      else reinterpret_cast<int*>(p.out)[(size_t)b * M + j] = old;
    }
  }

  if (p.temp) {
#pragma unroll
    for (int i = 0; i < PPT; ++i) {
      const int k = tid + i * FPS_THREADS;
      if (k < N) p.temp[(size_t)b * N + k] = td[i];
    }
  }
}

// Clouds beyond the register-resident kernel (N > 16 * FPS_THREADS = 8192; the reference kernel and the torch loops
// have no size limit): same rounds, same distance forms and tie keys, but the running minimum lives in the caller's
// `temp` array (or a stream-ordered scratch for the torch variants) and the coordinates are re-read through L1/L2
// every round.  Each thread owns the same elements k = tid, tid + 1024, ... in every round, so no two threads ever
// touch the same temp[k].
constexpr int FPS_BIG_THREADS = 1024;

__global__ void __launch_bounds__(FPS_BIG_THREADS) fps_stream_kernel(const FpsParams p, float* scratch) {
  __shared__ uint2 s_r[2][FPS_BIG_THREADS / 32];
  const int b = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int N = p.N, M = p.M;
  const float* xyz = p.xyz + (size_t)b * N * 3;
  float* temp = (p.temp ? p.temp : scratch) + (size_t)b * N;
  if (!p.temp)
    for (int k = tid; k < N; k += FPS_BIG_THREADS) temp[k] = 1e10f;   // own elements only: no barrier needed

  int old = p.start ? (int)p.start[b] : 0;
  if (tid == 0) {
    if (p.idx64) reinterpret_cast<long long*>(p.out)[(size_t)b * M] = old;
    else reinterpret_cast<int*>(p.out)[(size_t)b * M] = old;
  }
  for (int j = 1; j < M; ++j) {
    const float cx = __ldg(xyz + (size_t)old * 3), cy = __ldg(xyz + (size_t)old * 3 + 1), cz = __ldg(xyz + (size_t)old * 3 + 2);
    uint32_t bv = 0u, bt = 0xffffffffu;
    for (int k = tid; k < N; k += FPS_BIG_THREADS) {
      const float d = fps_dist(p.mode, __ldg(xyz + (size_t)k * 3), __ldg(xyz + (size_t)k * 3 + 1), __ldg(xyz + (size_t)k * 3 + 2),
                               cx, cy, cz);
      const float t = fminf(d, temp[k]);
      temp[k] = t;
      uint32_t tk = (uint32_t)k;
      if (p.mode == 0) {
        const uint32_t r = (p.ref_log2 == 0) ? 0u : (__brev((uint32_t)(k % p.ref_bs)) >> (32 - p.ref_log2));
        tk = (r << 16) | (uint32_t)(k / p.ref_bs);
      }
      const uint32_t u = __float_as_uint(t);
      if (u > bv || (u == bv && tk < bt)) { bv = u; bt = tk; }
    }
    uint32_t wv = __reduce_max_sync(L3D_FULL_MASK, bv);
    uint32_t wc = __reduce_max_sync(L3D_FULL_MASK, (bv == wv) ? ~bt : 0u);
    const int buf = j & 1;
    if (lane == 0) s_r[buf][warp] = make_uint2(wv, wc);
    __syncthreads();
    const uint2 e = s_r[buf][lane];                       // 32 warps: one entry per lane
    wv = __reduce_max_sync(L3D_FULL_MASK, e.x);
    wc = __reduce_max_sync(L3D_FULL_MASK, (e.x == wv) ? e.y : 0u);
    const uint32_t wtk = ~wc;
    if (p.mode == 0) {
      const uint32_t r = (p.ref_log2 == 0) ? 0u : (__brev(wtk >> 16) >> (32 - p.ref_log2));
      old = (int)((wtk & 0xffffu) * (uint32_t)p.ref_bs + r);
    } else {
      old = (int)wtk;
    }
    if (tid == 0) {
      if (p.idx64) reinterpret_cast<long long*>(p.out)[(size_t)b * M + j] = old;
      else reinterpret_cast<int*>(p.out)[(size_t)b * M + j] = old;
    }
  }
}

static int fps_launch(FpsParams p, cudaStream_t s) {
  if (!p.xyz || !p.out || p.B < 0 || p.N < 1 || p.M < 0) return L3D_ERR_INVALID;
  if (p.B == 0 || p.M == 0) return L3D_OK;   // `if (m <= 0) return;` (sampling_gpu.cu:99)
  // the reference's launch width: opt_n_threads(n) = max(min(1 << int(log(n)/log(2)), 1024), 1)
  const int pow_2 = (int)(std::log(static_cast<double>(p.N)) / std::log(2.0));
  int bs = 1 << pow_2;
  if (bs > 1024) bs = 1024;
  if (bs < 1) bs = 1;
  p.ref_bs = bs;
  p.ref_log2 = 0;
  while ((1 << p.ref_log2) < bs) ++p.ref_log2;
  if (p.N > 16 * FPS_THREADS) {
    if ((long)p.N > 65535L * p.ref_bs) return L3D_ERR_UNSUPPORTED;   // 16-bit per-thread element counter of the tie key
    float* scratch = nullptr;
    if (!p.temp) {
      cudaError_t e = cudaMallocAsync((void**)&scratch, (size_t)p.B * p.N * sizeof(float), s);
      if (e != cudaSuccess) return (int)e;
    }
    fps_stream_kernel<<<p.B, FPS_BIG_THREADS, 0, s>>>(p, scratch);
    count_launch();
    const cudaError_t le = cudaGetLastError();
    if (scratch) cudaFreeAsync(scratch, s);
    return le == cudaSuccess ? L3D_OK : (int)le;
  }
  const int ppt = (p.N + FPS_THREADS - 1) / FPS_THREADS;
  const size_t smem = (size_t)p.N * 3 * sizeof(float);   // <= 96 KB (N <= 8192)
  if (smem > 40 * 1024) {   // (static shared memory also counts against the 48 KB default)
    // opt in to > 48 KB of dynamic shared memory (only the two widest instantiations need it)
    int dev = 0;
    cudaGetDevice(&dev);
    cudaError_t e = raise_smem_once<fps_kernel<8>>(dev, 96 * 1024);
    if (e == cudaSuccess) e = raise_smem_once<fps_kernel<16>>(dev, 96 * 1024);
    if (e != cudaSuccess) return (int)e;
  }
  if (ppt <= 1) fps_kernel<1><<<p.B, FPS_THREADS, smem, s>>>(p);
  else if (ppt <= 2) fps_kernel<2><<<p.B, FPS_THREADS, smem, s>>>(p);
  else if (ppt <= 4) fps_kernel<4><<<p.B, FPS_THREADS, smem, s>>>(p);
  else if (ppt <= 8) fps_kernel<8><<<p.B, FPS_THREADS, smem, s>>>(p);
  else fps_kernel<16><<<p.B, FPS_THREADS, smem, s>>>(p);
  count_launch();
  L3D_LAUNCH_CHECK();
  return L3D_OK;
}

}  // namespace l3d

using namespace l3d;

extern "C" int l3d_pn2_furthest_point_sampling(int b, int n, int m, const float* dataset_dev,
                                               float* temp_dev, int32_t* idxs_dev, void* stream) {
  if (!temp_dev) return L3D_ERR_INVALID;
  FpsParams p{};
  p.xyz = dataset_dev; p.temp = temp_dev; p.start = nullptr; p.out = idxs_dev;
  p.B = b; p.N = n; p.M = m; p.mode = 0; p.idx64 = 0;
  return fps_launch(p, (cudaStream_t)stream);
}

extern "C" int l3d_farthest_point_sample(const float* xyz_dev, int B, int N, int npoint,
                                         const int64_t* start_dev, int64_t* centroids_dev,
                                         void* stream) {
  FpsParams p{};
  p.xyz = xyz_dev; p.temp = nullptr; p.start = (const long long*)start_dev; p.out = centroids_dev;
  p.B = B; p.N = N; p.M = npoint; p.mode = 1; p.idx64 = 1;
  return fps_launch(p, (cudaStream_t)stream);
}
