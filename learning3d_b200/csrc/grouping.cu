// Neighbourhood grouping family (sm_100a): ball query, group / gather (+grads), 3-NN interpolation,
// square_distance, index_points, compute_density.
//
// Replaces the pointnet2 CUDA ops of utils/lib/src/{ball_query,group_points,sampling,interpolate}_gpu.cu
// (K7, K8, K9, K13 of SURVEY.md §2.2) and the pure-torch grouping helpers of
// utils/model_common_utils.py, utils/pointconv_util.py and utils/ppfnet_util.py (a3, a6, a8, a9).
// All of these are HBM / L2-bandwidth bound gathers or short linear scans: one thread (or warp) per
// output row, coalesced 32-bit stores, index loaded once and reused across channels.
#include "common.cuh"
#include "../../include/l3d_b200.h"
#include "launch_count.h"

namespace l3d {

// ---- distances -------------------------------------------------------------------------
// pointnet2 CUDA kernels: `dx*dx + dy*dy + dz*dz` as nvcc contracts it (see knn.cu).
__device__ __forceinline__ float d2_pn2(float dx, float dy, float dz) {
  return fmaf(dz, dz, fmaf(dx, dx, __fmul_rn(dy, dy)));
}
// torch expansion form: square_distance(src, dst) = ((-2 * src.dst) + |src|^2) + |dst|^2 with the
// K=3 GEMM accumulation order (model_common_utils.py:35-37).
__device__ __forceinline__ float sumsq3(float x, float y, float z) {
  return __fadd_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)), __fmul_rn(z, z));
}
__device__ __forceinline__ float d2_expansion(float sx, float sy, float sz, float ss, float dx,
                                              float dy, float dz, float dd) {
  const float dot = fmaf(sz, dz, fmaf(sy, dy, __fmul_rn(sx, dx)));
  return __fadd_rn(fmaf(-2.0f, dot, ss), dd);
}

// ---- ball query ------------------------------------------------------------------------
// One warp per query.  32 candidates are tested per step; hits keep their index order through
// ballot/popc ranks, so "first nsample in ascending index order" needs no sort (the torch
// reference sorts a [B,S,N] int64 tensor: model_common_utils.py:123).
struct BallParams {
  const float* xyz;       // [B,N,3]
  const float* new_xyz;   // [B,S,3]
  const long long* itself;  // optional [B,S] (ppfnet_util variant)
  void* out_idx;          // [B,S,nsample] int32 / int64
  long long* out_cnt;     // optional [B,S]
  int B, N, S, nsample;
  float r2;
  int mode;   // 0: pointnet2 CUDA semantics (direct fma distance, d2 < r2, pad first, none -> 0)
              // 1: torch semantics (expansion distance, keep d2 <= r2, pad first, none -> N)
  int idx64;
};

__global__ void __launch_bounds__(256) ball_query_kernel(const BallParams p) {
  const int lane = threadIdx.x & 31;
  const long q = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (q >= (long)p.B * p.S) return;
  const int b = (int)(q / p.S);
  const float* xyz = p.xyz + (size_t)b * p.N * 3;
  const float qx = p.new_xyz[q * 3], qy = p.new_xyz[q * 3 + 1], qz = p.new_xyz[q * 3 + 2];
  const float qq = sumsq3(qx, qy, qz);
  const int self = p.itself ? (int)p.itself[q] : -1;
  const unsigned lt = (1u << lane) - 1u;

  int written = 0, first = -1;
  long long total = 0;
  for (int k0 = 0; k0 < p.N; k0 += 32) {
    const int k = k0 + lane;
    bool hit = false;
    if (k < p.N) {
      const float x = xyz[k * 3], y = xyz[k * 3 + 1], z = xyz[k * 3 + 2];
      if (p.mode == 0) {
        // (new_x - x)^2 + ... < radius^2          (ball_query_gpu.cu:33-34)
        hit = d2_pn2(__fsub_rn(qx, x), __fsub_rn(qy, y), __fsub_rn(qz, z)) < p.r2;
      } else {
        // group_idx[sqrdists > radius**2] = N    (model_common_utils.py:116)
        const float d = d2_expansion(qx, qy, qz, qq, x, y, z, sumsq3(x, y, z));
        hit = !(d > p.r2) && (k != self);
      }
    }
    const unsigned m = __ballot_sync(L3D_FULL_MASK, hit);
    if (m) {
      if (first < 0) first = k0 + __ffs(m) - 1;
      const int slot = written + __popc(m & lt);
      if (hit && slot < p.nsample) {
        const long o = q * p.nsample + slot;
        if (p.idx64) reinterpret_cast<long long*>(p.out_idx)[o] = k;
        else reinterpret_cast<int*>(p.out_idx)[o] = k;
      }
      const int c = __popc(m);
      written += c;
      total += c;
    }
    if (!p.out_cnt && written >= p.nsample) break;
  }
  if (written > p.nsample) written = p.nsample;
  // padding: first hit (pointnet2: ball_query_gpu.cu:36-40; torch: :124-126); with itself_indices
  // the query's own index (ppfnet_util.py:125-126); no hit at all: 0 (pre-zeroed idx,
  // pointnet2_utils.py:245) or N (model_common_utils.py:116 leaves N in place)
  int pad;
  if (p.itself) pad = self;
  else if (first >= 0) pad = first;
  else pad = (p.mode == 0) ? 0 : p.N;
  for (int s = written + lane; s < p.nsample; s += 32) {
    const long o = q * p.nsample + s;
    if (p.idx64) reinterpret_cast<long long*>(p.out_idx)[o] = pad;
    else reinterpret_cast<int*>(p.out_idx)[o] = pad;
  }
  if (p.out_cnt && lane == 0) p.out_cnt[q] = total;
}

// ---- group / gather ----------------------------------------------------------------------
// out[b,c,pos] = points[b,c,idx[b,pos]] for pos in [0, P) (P = npoints*nsample; gather: nsample=1).
// A thread owns one pos and a slab of GROUP_CPB channels: the index is loaded once, stores are
// coalesced along pos.  grid = (ceil(P/256), ceil(C/GROUP_CPB), B).
constexpr int GROUP_CPB = 16;

template <typename IdxT>
__global__ void __launch_bounds__(256) group_points_kernel(int c, int n, long P,
                                                           const float* __restrict__ points,
                                                           const IdxT* __restrict__ idx,
                                                           float* __restrict__ out) {
  const int b = blockIdx.z;
  const long pos = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (pos >= P) return;
  const int c0 = blockIdx.y * GROUP_CPB;
  const int c1 = min(c, c0 + GROUP_CPB);
  const long j = (long)idx[(size_t)b * P + pos];
  const float* src = points + ((size_t)b * c + c0) * n + j;
  float* dst = out + ((size_t)b * c + c0) * P + pos;
#pragma unroll 4
  for (int cc = c0; cc < c1; ++cc) {
    *dst = __ldg(src);
    src += n;
    dst += P;
  }
}

template <typename IdxT>
__global__ void __launch_bounds__(256) group_points_grad_kernel(int c, int n, long P,
                                                                const float* __restrict__ grad_out,
                                                                const IdxT* __restrict__ idx,
                                                                float* __restrict__ grad_points) {
  const int b = blockIdx.z;
  const long pos = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (pos >= P) return;
  const int c0 = blockIdx.y * GROUP_CPB;
  const int c1 = min(c, c0 + GROUP_CPB);
  const long j = (long)idx[(size_t)b * P + pos];
  const float* src = grad_out + ((size_t)b * c + c0) * P + pos;
  float* dst = grad_points + ((size_t)b * c + c0) * n + j;
  for (int cc = c0; cc < c1; ++cc) {
    atomicAdd(dst, *src);   // same scatter as group_points_gpu.cu:24 / sampling_gpu.cu:61
    src += P;
    dst += n;
  }
}

// ---- three_interpolate --------------------------------------------------------------------
// out[b,c,n] = w0*p[i0] + w1*p[i1] + w2*p[i2] as nvcc contracts it: fma(w2,p2, fma(w0,p0, w1*p1))
// (interpolate_gpu.cu:164; SASS of the reference file).
__global__ void __launch_bounds__(256) three_interpolate_kernel(int c, int m, int n,
                                                                const float* __restrict__ points,
                                                                const int* __restrict__ idx,
                                                                const float* __restrict__ weight,
                                                                float* __restrict__ out) {
  const int b = blockIdx.z;
  const int pt = blockIdx.x * blockDim.x + threadIdx.x;
  if (pt >= n) return;
  const int c0 = blockIdx.y * GROUP_CPB, c1 = min(c, c0 + GROUP_CPB);
  const int* ip = idx + ((size_t)b * n + pt) * 3;
  const float* wp = weight + ((size_t)b * n + pt) * 3;
  const int i0 = ip[0], i1 = ip[1], i2 = ip[2];
  const float w0 = wp[0], w1 = wp[1], w2 = wp[2];
  for (int cc = c0; cc < c1; ++cc) {
    const float* pp = points + ((size_t)b * c + cc) * m;
    out[((size_t)b * c + cc) * n + pt] =
        fmaf(w2, __ldg(pp + i2), fmaf(w0, __ldg(pp + i0), __fmul_rn(w1, __ldg(pp + i1))));
  }
}

__global__ void __launch_bounds__(256) three_interpolate_grad_kernel(
    int c, int n, int m, const float* __restrict__ grad_out, const int* __restrict__ idx,
    const float* __restrict__ weight, float* __restrict__ grad_points) {
  const int b = blockIdx.z;
  const int pt = blockIdx.x * blockDim.x + threadIdx.x;
  if (pt >= n) return;
  const int c0 = blockIdx.y * GROUP_CPB, c1 = min(c, c0 + GROUP_CPB);
  const int* ip = idx + ((size_t)b * n + pt) * 3;
  const float* wp = weight + ((size_t)b * n + pt) * 3;
  const int i0 = ip[0], i1 = ip[1], i2 = ip[2];
  const float w0 = wp[0], w1 = wp[1], w2 = wp[2];
  for (int cc = c0; cc < c1; ++cc) {
    const float g = grad_out[((size_t)b * c + cc) * n + pt];
    float* gp = grad_points + ((size_t)b * c + cc) * m;
    atomicAdd(gp + i0, __fmul_rn(g, w0));   // interpolate_gpu.cu:208-210
    atomicAdd(gp + i1, __fmul_rn(g, w1));
    atomicAdd(gp + i2, __fmul_rn(g, w2));
  }
}

// ---- square_distance (materialised; the API returns the matrix) ------------------------------
// out[b,i,j] = ((-2 src_i.dst_j) + |src_i|^2) + |dst_j|^2.  Write-bound: 4*N*M bytes per item.
__global__ void __launch_bounds__(256) square_distance_kernel(const float* __restrict__ src,
                                                              const float* __restrict__ dst, int N,
                                                              int M, float* __restrict__ out) {
  __shared__ float4 s_dst[256];
  const int b = blockIdx.z;
  const int j = blockIdx.x * 256 + threadIdx.x;
  {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (j < M) {
      const float* d = dst + ((size_t)b * M + j) * 3;
      v = make_float4(d[0], d[1], d[2], sumsq3(d[0], d[1], d[2]));
    }
    s_dst[threadIdx.x] = v;
  }
  __syncthreads();
  const float4 dj = s_dst[threadIdx.x];
  const int i0 = blockIdx.y * 64, i1 = min(N, i0 + 64);
  for (int i = i0; i < i1; ++i) {
    const float* s = src + ((size_t)b * N + i) * 3;   // warp-uniform -> broadcast load
    const float sx = __ldg(s), sy = __ldg(s + 1), sz = __ldg(s + 2);
    if (j < M)
      out[((size_t)b * N + i) * M + j] = d2_expansion(sx, sy, sz, sumsq3(sx, sy, sz), dj.x, dj.y, dj.z, dj.w);
  }
}

// ---- index_points: out[b, r, :] = points[b, idx[b, r], :] ------------------------------------
__global__ void __launch_bounds__(256) index_points_kernel(const float* __restrict__ points,
                                                           const long long* __restrict__ idx, int N,
                                                           long R, int C, float* __restrict__ out) {
  const int b = blockIdx.y;
  const long total = R * C;
  for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < total;
       t += (long)gridDim.x * blockDim.x) {
    const long r = t / C;
    const int c = (int)(t - r * C);
    const long j = idx[(size_t)b * R + r];
    // an index outside [0, N) (torch-mode ball query pads empty rows with N, model_common_utils.py:116) would
    // be a device-side assert in the reference's advanced indexing; here it reads nothing and yields NaN
    out[(size_t)b * total + t] = ((unsigned long)j < (unsigned long)N)
                                     ? __ldg(points + ((size_t)b * N + j) * C + c) : __int_as_float(0x7fc00000);
  }
}
__global__ void __launch_bounds__(256) index_points_grad_kernel(const float* __restrict__ grad_out,
                                                                const long long* __restrict__ idx,
                                                                int N, long R, int C,
                                                                float* __restrict__ grad_points) {
  const int b = blockIdx.y;
  const long total = R * C;
  for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < total;
       t += (long)gridDim.x * blockDim.x) {
    const long r = t / C;
    const int c = (int)(t - r * C);
    const long j = idx[(size_t)b * R + r];
    if ((unsigned long)j < (unsigned long)N)   // out-of-range rows received NaN in the forward; scatter nothing
      atomicAdd(grad_points + ((size_t)b * N + j) * C + c, grad_out[(size_t)b * total + t]);
  }
}

// ---- compute_density (pointconv_util.py:199-209) ----------------------------------------------
// density_i = mean_j exp(-d2_ij / (2 bw^2)) / (2.5 bw): a row reduction of the distance tile loop,
// never materialising the N x N matrix.  One warp per row, fixed summation order (deterministic).
__global__ void __launch_bounds__(256) density_kernel(const float* __restrict__ xyz, int B, int N,
                                                      float two_bw2, float norm,
                                                      float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const long row = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= (long)B * N) return;
  const int b = (int)(row / N);
  const float* base = xyz + (size_t)b * N * 3;
  const float sx = xyz[row * 3], sy = xyz[row * 3 + 1], sz = xyz[row * 3 + 2];
  const float ss = sumsq3(sx, sy, sz);
  float acc = 0.f;
  for (int j = lane; j < N; j += 32) {
    const float x = base[j * 3], y = base[j * 3 + 1], z = base[j * 3 + 2];
    const float d = d2_expansion(sx, sy, sz, ss, x, y, z, sumsq3(x, y, z));
    // torch: exp(-sqrdists / (2.0*bw*bw)) / (2.5*bw)
    acc += __fdiv_rn(expf(__fdiv_rn(-d, two_bw2)), norm);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(L3D_FULL_MASK, acc, o);
  if (lane == 0) out[row] = acc / (float)N;
}

static inline dim3 grid3(long x, long y, long z) { return dim3((unsigned)x, (unsigned)y, (unsigned)z); }

}  // namespace l3d

using namespace l3d;

static int ball_launch(BallParams p, cudaStream_t s) {
  if (!p.xyz || !p.new_xyz || !p.out_idx || p.B < 0 || p.N < 1 || p.S < 0 || p.nsample < 1)
    return L3D_ERR_INVALID;
  const long q = (long)p.B * p.S;
  if (q == 0) return L3D_OK;
  ball_query_kernel<<<(unsigned)((q + 7) / 8), 256, 0, s>>>(p);
  count_launch();
  L3D_LAUNCH_CHECK();
  return L3D_OK;
}

extern "C" int l3d_pn2_ball_query(int b, int n, int m, float radius, int nsample,
                                  const float* new_xyz_dev, const float* xyz_dev, int32_t* idx_dev,
                                  void* stream) {
  BallParams p{};
  p.xyz = xyz_dev; p.new_xyz = new_xyz_dev; p.out_idx = idx_dev;
  p.B = b; p.N = n; p.S = m; p.nsample = nsample;
  p.r2 = radius * radius;   // float radius2 = radius * radius;  (ball_query_gpu.cu:21)
  p.mode = 0; p.idx64 = 0;
  return ball_launch(p, (cudaStream_t)stream);
}

extern "C" int l3d_query_ball_point(const float* xyz_dev, const float* new_xyz_dev, int B, int N,
                                    int S, float radius2, int nsample,
                                    const int64_t* itself_indices_dev, int64_t* group_idx_dev,
                                    int64_t* cnt_dev, void* stream) {
  BallParams p{};
  p.xyz = xyz_dev; p.new_xyz = new_xyz_dev; p.out_idx = group_idx_dev;
  p.itself = (const long long*)itself_indices_dev; p.out_cnt = (long long*)cnt_dev;
  p.B = B; p.N = N; p.S = S; p.nsample = nsample; p.r2 = radius2; p.mode = 1; p.idx64 = 1;
  return ball_launch(p, (cudaStream_t)stream);
}

template <typename IdxT, bool GRAD>
static int group_launch(int b, int c, int n, long P, const float* in, const IdxT* idx, float* out,
                        cudaStream_t s) {
  if (!in || !idx || !out || b < 0 || c < 1 || n < 1 || P < 0 || b > 65535) return L3D_ERR_INVALID;
  if (b == 0 || P == 0) return L3D_OK;
  const dim3 grid = grid3((P + 255) / 256, (c + GROUP_CPB - 1) / GROUP_CPB, b);
  if (grid.y > 65535) return L3D_ERR_UNSUPPORTED;
  if (GRAD) group_points_grad_kernel<IdxT><<<grid, 256, 0, s>>>(c, n, P, in, idx, out);
  else group_points_kernel<IdxT><<<grid, 256, 0, s>>>(c, n, P, in, idx, out);
  count_launch();
  L3D_LAUNCH_CHECK();
  return L3D_OK;
}

extern "C" int l3d_pn2_group_points(int b, int c, int n, int npoints, int nsample,
                                    const float* points_dev, const int32_t* idx_dev, float* out_dev,
                                    void* stream) {
  return group_launch<int, false>(b, c, n, (long)npoints * nsample, points_dev, idx_dev, out_dev,
                                  (cudaStream_t)stream);
}
extern "C" int l3d_pn2_group_points_grad(int b, int c, int n, int npoints, int nsample,
                                         const float* grad_out_dev, const int32_t* idx_dev,
                                         float* grad_points_dev, void* stream) {
  return group_launch<int, true>(b, c, n, (long)npoints * nsample, grad_out_dev, idx_dev,
                                 grad_points_dev, (cudaStream_t)stream);
}
extern "C" int l3d_pn2_gather_points(int b, int c, int n, int npoints, const float* points_dev,
                                     const int32_t* idx_dev, float* out_dev, void* stream) {
  return group_launch<int, false>(b, c, n, (long)npoints, points_dev, idx_dev, out_dev,
                                  (cudaStream_t)stream);
}
extern "C" int l3d_pn2_gather_points_grad(int b, int c, int n, int npoints,
                                          const float* grad_out_dev, const int32_t* idx_dev,
                                          float* grad_points_dev, void* stream) {
  return group_launch<int, true>(b, c, n, (long)npoints, grad_out_dev, idx_dev, grad_points_dev,
                                 (cudaStream_t)stream);
}

extern "C" int l3d_pn2_three_interpolate(int b, int c, int m, int n, const float* points_dev,
                                         const int32_t* idx_dev, const float* weight_dev,
                                         float* out_dev, void* stream) {
  if (!points_dev || !idx_dev || !weight_dev || !out_dev || b < 0 || c < 1 || m < 1 || n < 0 || b > 65535)
    return L3D_ERR_INVALID;
  if (b == 0 || n == 0) return L3D_OK;
  const dim3 grid = grid3((n + 255) / 256, (c + GROUP_CPB - 1) / GROUP_CPB, b);
  three_interpolate_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(c, m, n, points_dev, idx_dev,
                                                                    weight_dev, out_dev);
  count_launch();
  L3D_LAUNCH_CHECK();
  return L3D_OK;
}
extern "C" int l3d_pn2_three_interpolate_grad(int b, int c, int n, int m, const float* grad_out_dev,
                                              const int32_t* idx_dev, const float* weight_dev,
                                              float* grad_points_dev, void* stream) {
  if (!grad_out_dev || !idx_dev || !weight_dev || !grad_points_dev || b < 0 || c < 1 || m < 1 ||
      n < 0 || b > 65535)
    return L3D_ERR_INVALID;
  if (b == 0 || n == 0) return L3D_OK;
  const dim3 grid = grid3((n + 255) / 256, (c + GROUP_CPB - 1) / GROUP_CPB, b);
  three_interpolate_grad_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(
      c, n, m, grad_out_dev, idx_dev, weight_dev, grad_points_dev);
  count_launch();
  L3D_LAUNCH_CHECK();
  return L3D_OK;
}

extern "C" int l3d_square_distance(const float* src_dev, const float* dst_dev, int B, int N, int M,
                                   float* out_dev, void* stream) {
  if (!src_dev || !dst_dev || !out_dev || B < 0 || N < 0 || M < 0 || B > 65535) return L3D_ERR_INVALID;
  if (B == 0 || N == 0 || M == 0) return L3D_OK;
  const dim3 grid = grid3((M + 255) / 256, (N + 63) / 64, B);
  if (grid.y > 65535) return L3D_ERR_UNSUPPORTED;
  square_distance_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(src_dev, dst_dev, N, M, out_dev);
  count_launch();
  L3D_LAUNCH_CHECK();
  return L3D_OK;
}

extern "C" int l3d_index_points(const float* points_dev, const int64_t* idx_dev, int B, int N,
                                int64_t R, int C, float* out_dev, void* stream) {
  if (!points_dev || !idx_dev || !out_dev || B < 0 || N < 1 || R < 0 || C < 1 || B > 65535)
    return L3D_ERR_INVALID;
  if (B == 0 || R == 0) return L3D_OK;
  long gx = (R * C + 255) / 256;
  if (gx > 148L * 32) gx = 148L * 32;
  index_points_kernel<<<grid3(gx, B, 1), 256, 0, (cudaStream_t)stream>>>(
      points_dev, (const long long*)idx_dev, N, R, C, out_dev);
  count_launch();
  L3D_LAUNCH_CHECK();
  return L3D_OK;
}
extern "C" int l3d_index_points_grad(const float* grad_out_dev, const int64_t* idx_dev, int B, int N,
                                     int64_t R, int C, float* grad_points_dev, void* stream) {
  if (!grad_out_dev || !idx_dev || !grad_points_dev || B < 0 || N < 1 || R < 0 || C < 1 || B > 65535)
    return L3D_ERR_INVALID;
  if (B == 0 || R == 0) return L3D_OK;
  long gx = (R * C + 255) / 256;
  if (gx > 148L * 32) gx = 148L * 32;
  index_points_grad_kernel<<<grid3(gx, B, 1), 256, 0, (cudaStream_t)stream>>>(
      grad_out_dev, (const long long*)idx_dev, N, R, C, grad_points_dev);
  count_launch();
  L3D_LAUNCH_CHECK();
  return L3D_OK;
}

// Staged variant (N <= DENS_MAX_N): the cloud of one batch item sits in shared memory as
// (x, y, z, |p|^2) — one conflict-free LDS.128 per candidate, shared by the DENS_R rows a warp owns — and the
// two true divisions and the libm exp of the per-pair expression are replaced by one multiply and
// ex2.approx (exp(-d/(2bw^2)) = 2^(d * c), c = -log2(e)/(2bw^2)); 1/(2.5 bw N) is applied once per row.
// Toleranced row (1e-5 relative, DESIGN.md §4): ~10 instructions per pair instead of ~50.
constexpr int DENS_R = 4;                 // rows per warp
constexpr int DENS_ROWS_PER_CTA = 8 * DENS_R * 2;
constexpr int DENS_MAX_N = 12288;         // 192 KB of float4
__global__ void __launch_bounds__(256) density_staged_kernel(const float* __restrict__ xyz, int B, int N,
                                                             float c_log2, float inv_norm_n,
                                                             float* __restrict__ out) {
  extern __shared__ float4 s_pts[];
  const int b = blockIdx.y;
  const float* base = xyz + (size_t)b * N * 3;
  for (int j = threadIdx.x; j < N; j += 256) {
    const float x = base[j * 3], y = base[j * 3 + 1], z = base[j * 3 + 2];
    s_pts[j] = make_float4(x, y, z, sumsq3(x, y, z));
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int row_end = min(N, (int)(blockIdx.x + 1) * DENS_ROWS_PER_CTA);
  for (int r0 = blockIdx.x * DENS_ROWS_PER_CTA + warp * DENS_R; r0 < row_end; r0 += 8 * DENS_R) {
    float4 q[DENS_R];
    float acc[DENS_R];
#pragma unroll
    for (int r = 0; r < DENS_R; ++r) { q[r] = s_pts[min(r0 + r, N - 1)]; acc[r] = 0.f; }
    for (int j = lane; j < N; j += 32) {
      const float4 cnd = s_pts[j];
#pragma unroll
      for (int r = 0; r < DENS_R; ++r) {
        const float d = d2_expansion(q[r].x, q[r].y, q[r].z, q[r].w, cnd.x, cnd.y, cnd.z, cnd.w);
        float e;
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(__fmul_rn(d, c_log2)));
        acc[r] = __fadd_rn(acc[r], e);
      }
    }
#pragma unroll
    for (int r = 0; r < DENS_R; ++r) {
      float a = acc[r];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(L3D_FULL_MASK, a, o);
      if (lane == 0 && r0 + r < row_end) out[(size_t)b * N + r0 + r] = __fmul_rn(a, inv_norm_n);
    }
  }
}

extern "C" int l3d_compute_density(const float* xyz_dev, int B, int N, float two_bw2, float norm,
                                   float* density_dev, void* stream) {
  if (!xyz_dev || !density_dev || B < 0 || N < 1) return L3D_ERR_INVALID;
  if (B == 0) return L3D_OK;
  if (N <= DENS_MAX_N && B <= 65535 && two_bw2 > 0.f && norm != 0.f) {
    const size_t smem = (size_t)N * sizeof(float4);
    if (smem > 40 * 1024) {
      int dev = 0;
      cudaGetDevice(&dev);
      const cudaError_t e = raise_smem_once<density_staged_kernel>(dev, DENS_MAX_N * sizeof(float4));
      if (e != cudaSuccess) return (int)e;
    }
    const float c_log2 = (float)(-1.4426950408889634 / (double)two_bw2);
    const float inv_norm_n = (float)(1.0 / ((double)norm * (double)N));
    dim3 grid((N + DENS_ROWS_PER_CTA - 1) / DENS_ROWS_PER_CTA, B);
    density_staged_kernel<<<grid, 256, smem, (cudaStream_t)stream>>>(xyz_dev, B, N, c_log2, inv_norm_n, density_dev);
    count_launch();
    L3D_LAUNCH_CHECK();
    return L3D_OK;
  }
  const long rows = (long)B * N;
  density_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, (cudaStream_t)stream>>>(xyz_dev, B, N, two_bw2,
                                                                                norm, density_dev);
  count_launch();
  L3D_LAUNCH_CHECK();
  return L3D_OK;
}
