// Approximate Earth Mover's Distance (approxmatch / matchcost / matchcostgrad), sm_100a.
//
// Replaces losses/cuda/emd_torch/pkg/include/cuda/emd.cuh (K3 :6-185, K4 :201-244, K5 :301-323,
// K6 :258-299) and pkg/src/cuda/emd.cu:8-70.
//
// The reference runs ONE 512-thread CTA per batch item (8 of 148 SMs at B=8) through 30 full
// N x M exp-sweeps and read-modify-writes the N x M `match` matrix in global memory on each of
// its 10 levels.  Here every sweep is a grid-wide "weighted row sweep"
//     S[r] = sum_c exp(level * |p_r - q_c|^2) * v[c]
// spread over all SMs (a warp owns 4 rows, columns staged in shared memory), and the three
// per-level sweeps are algebraically regrouped so that `match` is never touched inside the loop:
//   (1) ratioL[k] = remainL[k] / (1e-9 + S(level; v = remainR))                 emd.cuh:32-60
//   (2) sumr[l]   = remainR[l] * S^T(level; v = ratioL); ratioR/remainR update   emd.cuh:80-116
//   (3) suml[k]   = ratioL[k] * S(level; v = ratioR); remainL update             emd.cuh:135-168
// (3) of level j and (1) of level j+1 sweep the same rows over the same columns and are fused
// (two exponentials per pair, one pass).  The per-level (ratioL, ratioR) vectors are kept (10*(n+m)
// floats per item) and one final pass rebuilds match = sum_j exp(level_j d2) ratioL_j[k] ratioR_j[l]
// with coalesced stores (written once instead of 10 read-modify-writes) fused with the matchcost
// reduction.  20 sweep launches + 1 final launch; MUFU(ex2)-bound.
// fp32 throughout, ex2.approx like the reference's __expf; results agree with the sequential
// restatement to ~1e-6 relative (summation order differs), inside the 1e-5 contract.
#include "common.cuh"
#include "../../include/l3d_b200.h"
#include "launch_count.h"

#include <algorithm>

namespace l3d {

constexpr int EMD_THREADS = 256;
constexpr int EMD_WARPS = EMD_THREADS / 32;
constexpr int EMD_R = 4;                         // rows per warp (two packed-f32x2 row pairs)
constexpr int EMD_CSPLIT = 2;                    // warps sharing a row group, each sweeping every 2nd 32-column block
constexpr int EMD_RGROUPS = EMD_WARPS / EMD_CSPLIT;
constexpr int EMD_ROWS_PER_CTA = EMD_RGROUPS * EMD_R;
constexpr int EMD_CHUNK = 1024;                  // columns staged per chunk
constexpr int EMD_LEVELS = 10;                   // j = 7 .. -2 (emd.cuh:27)
constexpr float LOG2E = 1.4426950408889634f;

__host__ __device__ inline float emd_level(int it) {
  // level = -4^j for j = 7..-1, and 0 at j = -2   (emd.cuh:28-31)
  if (it == EMD_LEVELS - 1) return 0.f;
  float v = 1.f;
  const int j = 7 - it;
  if (j >= 0) { for (int i = 0; i < j; ++i) v *= 4.f; }
  else { for (int i = 0; i < -j; ++i) v *= 0.25f; }
  return -v;
}

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// __expf(level * d2) exactly as nvcc expands it in the reference kernels (emd.cuh:58,103,157; SASS of
// oracle/_ref/libemd_ref.so): FMUL level*d2, FMUL by fp32 log2(e), MUFU.EX2.  (Below 2^-126 the reference
// squares ex2(t/2) to keep denormals; those weights are < 1.2e-38 and flush to 0 here.)
__device__ __forceinline__ float emd_exp(float level, float d2) {
  return ex2_approx(__fmul_rn(__fmul_rn(level, d2), LOG2E));
}

__device__ __forceinline__ float emd_d2(float ax, float ay, float az, float bx, float by, float bz) {
  const float dx = bx - ax, dy = by - ay, dz = bz - az;
  return fmaf(dz, dz, fmaf(dx, dx, dy * dy));
}

enum { EMD_PH1 = 1, EMD_PH2 = 2, EMD_PH3_PH1 = 3 };

struct EmdSweepParams {
  const float* rows;    // [B,nr,3] row cloud
  const float* cols;    // [B,nc,3] column cloud
  int B, nr, nc;
  int phase;
  float lvlA, lvlB;     // level (-4^j) of sweep A (and B when fused)
  const float* vA;      // [B,nc] column weights of sweep A
  const float* vB;      // [B,nc] column weights of sweep B (fused only)
  // per-row state (all [B,nr])
  float* remain;        // remainL (ph1, ph3) or remainR (ph2)
  const float* ratio_in;   // ratioL of the finishing level (ph3)
  float* ratio_out;        // ratioL (ph1 / fused) or ratioR (ph2) of the level being computed
  float multi;             // initial remain value when `init` (multiL)
  int init;                // ph1 of the first level: remain = multi
};

// One weighted row sweep for the rows [row_begin, row_end) of batch item b, executed by one CTA: 4 row groups of 4
// rows, each shared by 2 warps that take alternate 32-column blocks (twice the warps per row = twice the latency
// hiding; their partial sums meet in shared memory).  The 4 rows of a warp are two packed-f32x2 pairs: every FADD /
// FMUL / FFMA below processes two rows (sm_100 FADD2 / FMUL2 / FFMA2, per-lane IEEE rounding = the scalar results).
// COHERENT: the column weights / row state were written by OTHER CTAs of the same launch (persistent kernel, after
// a per-item barrier), so they are read with ld.global.cg (L2) instead of through L1.
template <bool FUSED, bool COHERENT>
__device__ __forceinline__ void emd_sweep_rows(const EmdSweepParams& p, int b, int row_begin, int row_end,
                                               float4* s_col, float* s_vb, float (*s_part)[EMD_RGROUPS][2 * EMD_R]) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int rg = warp % EMD_RGROUPS, ch = warp / EMD_RGROUPS;
  const float* rows = p.rows + (size_t)b * p.nr * 3;
  const float* cols = p.cols + (size_t)b * p.nc * 3;
  auto ldv = [](const float* q) -> float { return COHERENT ? __ldcg(q) : *q; };
  const unsigned long long lvlA2 = f2_pack(p.lvlA, p.lvlA), lvlB2 = f2_pack(p.lvlB, p.lvlB), l2e2 = f2_pack(LOG2E, LOG2E);
  for (int base = row_begin; base < row_end; base += EMD_ROWS_PER_CTA) {
    const int r0 = base + rg * EMD_R;
    unsigned long long nrx[2], nry[2], nrz[2], sa[2], sb[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int ra = min(r0 + 2 * h, p.nr - 1), rb = min(r0 + 2 * h + 1, p.nr - 1);
      nrx[h] = f2_pack(-rows[ra * 3], -rows[rb * 3]);
      nry[h] = f2_pack(-rows[ra * 3 + 1], -rows[rb * 3 + 1]);
      nrz[h] = f2_pack(-rows[ra * 3 + 2], -rows[rb * 3 + 2]);
      sa[h] = 0ull; sb[h] = 0ull;
    }
    for (int c0 = 0; c0 < p.nc; c0 += EMD_CHUNK) {
      const int cn = min(EMD_CHUNK, p.nc - c0);
      __syncthreads();
      for (int c = tid; c < cn; c += EMD_THREADS) {
        const float* q = cols + (size_t)(c0 + c) * 3;
        s_col[c] = make_float4(q[0], q[1], q[2], ldv(p.vA + (size_t)b * p.nc + c0 + c));
        if (FUSED) s_vb[c] = ldv(p.vB + (size_t)b * p.nc + c0 + c);
      }
      __syncthreads();
      if (r0 < row_end) {
        for (int c = ch * 32 + lane; c < cn; c += 32 * EMD_CSPLIT) {
          const float4 q = s_col[c];
          const unsigned long long qx = f2_pack(q.x, q.x), qy = f2_pack(q.y, q.y), qz = f2_pack(q.z, q.z);
          const unsigned long long qw = f2_pack(q.w, q.w);
          unsigned long long vb2 = 0ull;
          if (FUSED) { const float vb = s_vb[c]; vb2 = f2_pack(vb, vb); }
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            // d2 = fma(dz, dz, fma(dx, dx, dy*dy)), d = column - row   (emd_d2, per lane)
            const unsigned long long dx = f2_add(qx, nrx[h]), dy = f2_add(qy, nry[h]), dz = f2_add(qz, nrz[h]);
            const unsigned long long d2 = f2_fma(dz, dz, f2_fma(dx, dx, f2_mul(dy, dy)));
            float t0, t1;
            f2_unpack(f2_mul(f2_mul(lvlA2, d2), l2e2), t0, t1);              // emd_exp: (level*d2)*log2e, then ex2
            sa[h] = f2_fma(f2_pack(ex2_approx(t0), ex2_approx(t1)), qw, sa[h]);
            if (FUSED) {
              f2_unpack(f2_mul(f2_mul(lvlB2, d2), l2e2), t0, t1);
              sb[h] = f2_fma(f2_pack(ex2_approx(t0), ex2_approx(t1)), vb2, sb[h]);
            }
          }
        }
      }
    }
    float fa[EMD_R], fb[EMD_R];
    f2_unpack(sa[0], fa[0], fa[1]); f2_unpack(sa[1], fa[2], fa[3]);
    f2_unpack(sb[0], fb[0], fb[1]); f2_unpack(sb[1], fb[2], fb[3]);
#pragma unroll
    for (int i = 0; i < EMD_R; ++i) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        fa[i] += __shfl_xor_sync(L3D_FULL_MASK, fa[i], o);
        if (FUSED) fb[i] += __shfl_xor_sync(L3D_FULL_MASK, fb[i], o);
      }
    }
    if (lane < EMD_R) {
      float S = fa[0], S2 = fb[0];
#pragma unroll
      for (int i = 1; i < EMD_R; ++i) if (lane == i) { S = fa[i]; S2 = fb[i]; }
      s_part[ch][rg][lane] = S;
      s_part[ch][rg][EMD_R + lane] = S2;
    }
    __syncthreads();
    if (ch == 0 && lane < EMD_R) {
      float S = s_part[0][rg][lane], S2 = s_part[0][rg][EMD_R + lane];
#pragma unroll
      for (int k = 1; k < EMD_CSPLIT; ++k) { S += s_part[k][rg][lane]; S2 += s_part[k][rg][EMD_R + lane]; }
      const int r = r0 + lane;
      if (r < row_end && r < p.nr) {
        const size_t o = (size_t)b * p.nr + r;
        if (p.phase == EMD_PH1) {
          const float rem = p.init ? p.multi : ldv(p.remain + o);
          if (p.init) p.remain[o] = rem;
          p.ratio_out[o] = rem / (1e-9f + S);                       // emd.cuh:40,60
        } else if (p.phase == EMD_PH2) {
          const float rem = ldv(p.remain + o);
          const float sumr = S * rem;                                 // emd.cuh:110
          const float consumption = fminf(rem / (sumr + 1e-9f), 1.0f);
          p.ratio_out[o] = consumption * rem;
          p.remain[o] = fmaxf(0.0f, rem - sumr);
        } else {
          // finish level j: remainL = max(0, remainL - ratioL_j * S_j)   (emd.cuh:157-168) ...
          const float rem = fmaxf(0.0f, ldv(p.remain + o) - ldv(p.ratio_in + o) * S);
          p.remain[o] = rem;
          // ... and start level j+1: ratioL_{j+1} = remainL / (1e-9 + S_{j+1})
          p.ratio_out[o] = rem / (1e-9f + S2);
        }
      }
    }
  }
}

template <bool FUSED>
__global__ void __launch_bounds__(EMD_THREADS) emd_sweep_kernel(const EmdSweepParams p) {
  __shared__ float4 s_col[EMD_CHUNK];
  __shared__ float s_vb[FUSED ? EMD_CHUNK : 1];
  __shared__ float s_part[EMD_CSPLIT][EMD_RGROUPS][2 * EMD_R];
  const int r0 = blockIdx.x * EMD_ROWS_PER_CTA;
  emd_sweep_rows<FUSED, false>(p, blockIdx.y, r0, min(r0 + EMD_ROWS_PER_CTA, p.nr), s_col, s_vb, s_part);
}

// ---- persistent forward: all 20 sweeps in ONE launch --------------------------------------------------------
// The sweeps of one batch item depend on each other only through the per-item vectors (remainL/R, ratioL/R), so
// the CTAs of an item synchronise among THEMSELVES (a monotonically increasing arrival counter per item in global
// memory, release/acquire at gpu scope) — no grid-wide barrier, items drift apart freely.  Every CTA of the grid
// must be co-resident (the host sizes the grid from the occupancy query).  Replaces the 20 sweep launches + the
// fill launch of the multi-launch path (kept below for batches too large to be co-resident).
struct EmdPersistParams {
  const float* xyz1; const float* xyz2;
  float* remainL; float* remainR;      // [B,n], [B,m]
  float* ratioL; float* ratioR;        // [LEVELS,B,n], [LEVELS,B,m]
  unsigned int* arrive;                // [B] zero-initialised arrival counters
  unsigned int* err;                   // zero-initialised error word (barrier time-out)
  int B, n, m, ctas_per_item;
  float multiL, multiR;
  float lvl[EMD_LEVELS];
};

// false = the other CTAs of the item never arrived (cannot happen under a cooperative launch; bounded so that
// a bug is an error word and NaN costs, never a hung GPU)
__device__ __forceinline__ bool emd_item_barrier(unsigned int* ctr, unsigned int target, unsigned int* err,
                                                 int* s_flag) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(ctr, 1u);
    unsigned int v = 0;
    unsigned long long spins = 0;
    do {
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(ctr) : "memory");
    } while (v < target && ++spins < (1ull << 26) && *(volatile unsigned int*)err == 0u);
    if (v < target) atomicExch(err, 1u);
    *s_flag = (v >= target) ? 1 : 0;
    __threadfence();
  }
  __syncthreads();
  return *s_flag != 0;
}

__global__ void __launch_bounds__(EMD_THREADS) emd_persistent_kernel(const EmdPersistParams q) {
  __shared__ float4 s_col[EMD_CHUNK];
  __shared__ float s_vb[EMD_CHUNK];
  __shared__ float s_part[EMD_CSPLIT][EMD_RGROUPS][2 * EMD_R];
  __shared__ int s_flag;
  const int C = q.ctas_per_item;
  const int b = blockIdx.x / C, cx = blockIdx.x - b * C;
  // contiguous row shares in both clouds, rounded up to whole warps' worth of rows
  auto share = [&](int nr, int& r0, int& r1) {
    const int per = ((nr + C - 1) / C + EMD_R - 1) / EMD_R * EMD_R;
    r0 = min(nr, cx * per); r1 = min(nr, r0 + per);
  };
  int l0, l1, r0, r1;
  share(q.n, l0, l1);
  share(q.m, r0, r1);
  unsigned int* ctr = q.arrive + b;
  unsigned int phase = 0;
  const size_t Bn = (size_t)q.B * q.n, Bm = (size_t)q.B * q.m;
  // remainR = multiR before anybody sweeps over it
  for (int r = r0 + (int)threadIdx.x; r < r1; r += EMD_THREADS) q.remainR[(size_t)b * q.m + r] = q.multiR;
  if (!emd_item_barrier(ctr, ++phase * C, q.err, &s_flag)) return;
  {
    EmdSweepParams p{};
    p.rows = q.xyz1; p.cols = q.xyz2; p.B = q.B; p.nr = q.n; p.nc = q.m; p.phase = EMD_PH1;
    p.lvlA = q.lvl[0]; p.vA = q.remainR; p.remain = q.remainL; p.ratio_out = q.ratioL; p.multi = q.multiL; p.init = 1;
    emd_sweep_rows<false, true>(p, b, l0, l1, s_col, s_vb, s_part);
  }
  if (!emd_item_barrier(ctr, ++phase * C, q.err, &s_flag)) return;
  for (int it = 0; it < EMD_LEVELS; ++it) {
    {
      EmdSweepParams p{};
      p.rows = q.xyz2; p.cols = q.xyz1; p.B = q.B; p.nr = q.m; p.nc = q.n; p.phase = EMD_PH2;
      p.lvlA = q.lvl[it]; p.vA = q.ratioL + (size_t)it * Bn; p.remain = q.remainR; p.ratio_out = q.ratioR + (size_t)it * Bm;
      emd_sweep_rows<false, true>(p, b, r0, r1, s_col, s_vb, s_part);
    }
    if (it + 1 == EMD_LEVELS) break;
    if (!emd_item_barrier(ctr, ++phase * C, q.err, &s_flag)) return;
    {
      EmdSweepParams p{};
      p.rows = q.xyz1; p.cols = q.xyz2; p.B = q.B; p.nr = q.n; p.nc = q.m; p.phase = EMD_PH3_PH1;
      p.lvlA = q.lvl[it]; p.vA = q.ratioR + (size_t)it * Bm; p.lvlB = q.lvl[it + 1]; p.vB = q.remainR;
      p.remain = q.remainL; p.ratio_in = q.ratioL + (size_t)it * Bn; p.ratio_out = q.ratioL + (size_t)(it + 1) * Bn;
      emd_sweep_rows<true, true>(p, b, l0, l1, s_col, s_vb, s_part);
    }
    if (!emd_item_barrier(ctr, ++phase * C, q.err, &s_flag)) return;
  }
}

// ---- cluster forward: one thread-block CLUSTER per batch item ------------------------------------------------------
// The sweeps of an item only talk to each other, so an item is given to one cluster of up to 16 CTAs (one GPC's worth
// of SMs; B = 8 fills the 8 GPCs of a B200): both clouds stay resident in every CTA's shared memory for the whole
// kernel (only the 4-byte column weights are refreshed per sweep), the CTAs split the rows, and the 20 phase
// boundaries are hardware cluster barriers (barrier.cluster, ~0.3 us) instead of global-memory counters.  Clusters
// are independent, so nothing has to be co-resident across items: no cooperative launch, any B.
constexpr int EMDC_THREADS = 512;
constexpr int EMDC_WARPS = EMDC_THREADS / 32;
constexpr int EMDC_RGROUPS = EMDC_WARPS / EMD_CSPLIT;          // 8 row groups of 4 rows per pass
constexpr int EMDC_ROWS = EMDC_RGROUPS * EMD_R;

struct EmdClusterSmem {
  float part[EMD_CSPLIT][EMDC_RGROUPS][2 * EMD_R];
};

__device__ __forceinline__ void emd_cluster_barrier() {
  __threadfence();
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// rows [row_begin, row_end) of the row cloud (resident, float4 xyz_) against ALL columns of the column cloud
// (resident, float4 xyz + current weight in .w); same arithmetic as emd_sweep_rows
template <bool FUSED>
__device__ __forceinline__ void emdc_sweep(const EmdSweepParams& p, int b, int row_begin, int row_end,
                                           const float4* __restrict__ s_rows, float4* __restrict__ s_cols,
                                           float* __restrict__ s_vb, EmdClusterSmem* sm) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int rg = warp % EMDC_RGROUPS, ch = warp / EMDC_RGROUPS;
  // refresh the column weights (written by other CTAs of the cluster in the previous phase: read through L2)
  for (int c = tid; c < p.nc; c += EMDC_THREADS) {
    s_cols[c].w = __ldcg(p.vA + (size_t)b * p.nc + c);
    if (FUSED) s_vb[c] = __ldcg(p.vB + (size_t)b * p.nc + c);
  }
  __syncthreads();
  const unsigned long long lvlA2 = f2_pack(p.lvlA, p.lvlA), lvlB2 = f2_pack(p.lvlB, p.lvlB), l2e2 = f2_pack(LOG2E, LOG2E);
  for (int base = row_begin; base < row_end; base += EMDC_ROWS) {
    const int r0 = base + rg * EMD_R;
    unsigned long long nrx[2], nry[2], nrz[2], sa[2], sb[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const float4 ra = s_rows[min(r0 + 2 * h, p.nr - 1)], rb = s_rows[min(r0 + 2 * h + 1, p.nr - 1)];
      nrx[h] = f2_pack(-ra.x, -rb.x); nry[h] = f2_pack(-ra.y, -rb.y); nrz[h] = f2_pack(-ra.z, -rb.z);
      sa[h] = 0ull; sb[h] = 0ull;
    }
    if (r0 < row_end) {
      for (int c = ch * 32 + lane; c < p.nc; c += 32 * EMD_CSPLIT) {
        const float4 q = s_cols[c];
        const unsigned long long qx = f2_pack(q.x, q.x), qy = f2_pack(q.y, q.y), qz = f2_pack(q.z, q.z);
        const unsigned long long qw = f2_pack(q.w, q.w);
        unsigned long long vb2 = 0ull;
        if (FUSED) { const float vb = s_vb[c]; vb2 = f2_pack(vb, vb); }
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const unsigned long long dx = f2_add(qx, nrx[h]), dy = f2_add(qy, nry[h]), dz = f2_add(qz, nrz[h]);
          const unsigned long long d2 = f2_fma(dz, dz, f2_fma(dx, dx, f2_mul(dy, dy)));
          float t0, t1;
          f2_unpack(f2_mul(f2_mul(lvlA2, d2), l2e2), t0, t1);
          sa[h] = f2_fma(f2_pack(ex2_approx(t0), ex2_approx(t1)), qw, sa[h]);
          if (FUSED) {
            f2_unpack(f2_mul(f2_mul(lvlB2, d2), l2e2), t0, t1);
            sb[h] = f2_fma(f2_pack(ex2_approx(t0), ex2_approx(t1)), vb2, sb[h]);
          }
        }
      }
    }
    float fa[EMD_R], fb[EMD_R];
    f2_unpack(sa[0], fa[0], fa[1]); f2_unpack(sa[1], fa[2], fa[3]);
    f2_unpack(sb[0], fb[0], fb[1]); f2_unpack(sb[1], fb[2], fb[3]);
#pragma unroll
    for (int i = 0; i < EMD_R; ++i) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        fa[i] += __shfl_xor_sync(L3D_FULL_MASK, fa[i], o);
        if (FUSED) fb[i] += __shfl_xor_sync(L3D_FULL_MASK, fb[i], o);
      }
    }
    __syncthreads();                       // the previous pass has consumed sm->part
    if (lane < EMD_R) {
      float S = fa[0], S2 = fb[0];
#pragma unroll
      for (int i = 1; i < EMD_R; ++i) if (lane == i) { S = fa[i]; S2 = fb[i]; }
      sm->part[ch][rg][lane] = S;
      sm->part[ch][rg][EMD_R + lane] = S2;
    }
    __syncthreads();
    if (ch == 0 && lane < EMD_R) {
      float S = sm->part[0][rg][lane], S2 = sm->part[0][rg][EMD_R + lane];
#pragma unroll
      for (int k = 1; k < EMD_CSPLIT; ++k) { S += sm->part[k][rg][lane]; S2 += sm->part[k][rg][EMD_R + lane]; }
      const int r = r0 + lane;
      if (r < row_end && r < p.nr) {
        const size_t o = (size_t)b * p.nr + r;
        if (p.phase == EMD_PH1) {
          const float rem = p.init ? p.multi : __ldcg(p.remain + o);
          if (p.init) p.remain[o] = rem;
          p.ratio_out[o] = rem / (1e-9f + S);
        } else if (p.phase == EMD_PH2) {
          const float rem = p.init ? p.multi : __ldcg(p.remain + o);
          const float sumr = S * rem;
          const float consumption = fminf(rem / (sumr + 1e-9f), 1.0f);
          p.ratio_out[o] = consumption * rem;
          p.remain[o] = fmaxf(0.0f, rem - sumr);
        } else {
          const float rem = fmaxf(0.0f, __ldcg(p.remain + o) - __ldcg(p.ratio_in + o) * S);
          p.remain[o] = rem;
          p.ratio_out[o] = rem / (1e-9f + S2);
        }
      }
    }
  }
}

__global__ void __launch_bounds__(EMDC_THREADS, 1) emd_cluster_kernel(const EmdPersistParams q) {
  extern __shared__ __align__(16) unsigned char emdc_raw[];
  float4* s_c1 = reinterpret_cast<float4*>(emdc_raw);                 // [n] cloud 1 (+ weight slot)
  float4* s_c2 = s_c1 + q.n;                                           // [m] cloud 2
  float* s_vb = reinterpret_cast<float*>(s_c2 + q.m);                  // [max(n, m)]
  EmdClusterSmem* sm = reinterpret_cast<EmdClusterSmem*>(s_vb + max(q.n, q.m));
  uint32_t NC, cx;
  asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(NC));
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(cx));
  const int b = blockIdx.x / NC;
  const float* x1 = q.xyz1 + (size_t)b * q.n * 3;
  const float* x2 = q.xyz2 + (size_t)b * q.m * 3;
  for (int i = threadIdx.x; i < q.n; i += EMDC_THREADS) s_c1[i] = make_float4(x1[i * 3], x1[i * 3 + 1], x1[i * 3 + 2], 0.f);
  for (int i = threadIdx.x; i < q.m; i += EMDC_THREADS) s_c2[i] = make_float4(x2[i * 3], x2[i * 3 + 1], x2[i * 3 + 2], 0.f);
  auto share = [&](int nr, int& a0, int& a1) {
    const int per = ((nr + (int)NC - 1) / (int)NC + EMD_R - 1) / EMD_R * EMD_R;
    a0 = min(nr, (int)cx * per); a1 = min(nr, a0 + per);
  };
  int l0, l1, r0, r1;
  share(q.n, l0, l1);
  share(q.m, r0, r1);
  const size_t Bn = (size_t)q.B * q.n, Bm = (size_t)q.B * q.m;
  for (int r = r0 + (int)threadIdx.x; r < r1; r += EMDC_THREADS) q.remainR[(size_t)b * q.m + r] = q.multiR;
  __syncthreads();
  emd_cluster_barrier();
  {
    EmdSweepParams p{};
    p.B = q.B; p.nr = q.n; p.nc = q.m; p.phase = EMD_PH1;
    p.lvlA = q.lvl[0]; p.vA = q.remainR; p.remain = q.remainL; p.ratio_out = q.ratioL; p.multi = q.multiL; p.init = 1;
    emdc_sweep<false>(p, b, l0, l1, s_c1, s_c2, s_vb, sm);
  }
  emd_cluster_barrier();
  for (int it = 0; it < EMD_LEVELS; ++it) {
    {
      EmdSweepParams p{};
      p.B = q.B; p.nr = q.m; p.nc = q.n; p.phase = EMD_PH2;
      p.lvlA = q.lvl[it]; p.vA = q.ratioL + (size_t)it * Bn; p.remain = q.remainR; p.ratio_out = q.ratioR + (size_t)it * Bm;
      emdc_sweep<false>(p, b, r0, r1, s_c2, s_c1, s_vb, sm);
    }
    if (it + 1 == EMD_LEVELS) break;
    emd_cluster_barrier();
    {
      EmdSweepParams p{};
      p.B = q.B; p.nr = q.n; p.nc = q.m; p.phase = EMD_PH3_PH1;
      p.lvlA = q.lvl[it]; p.vA = q.ratioR + (size_t)it * Bm; p.lvlB = q.lvl[it + 1]; p.vB = q.remainR;
      p.remain = q.remainL; p.ratio_in = q.ratioL + (size_t)it * Bn; p.ratio_out = q.ratioL + (size_t)(it + 1) * Bn;
      emdc_sweep<true>(p, b, l0, l1, s_c1, s_c2, s_vb, sm);
    }
    emd_cluster_barrier();
  }
}

static size_t emd_cluster_smem(int n, int m) {
  return ((size_t)n + m) * sizeof(float4) + (size_t)std::max(n, m) * sizeof(float) + sizeof(EmdClusterSmem) + 16;
}

// Final pass: match[b, l, k] (reference index l*n + k, emd.cuh:158) = sum_j exp(level_j d2)
// ratioL_j[k] ratioR_j[l]; cost[b] = sum match * |x1_k - x2_l|   (emd.cuh:201-244).
// One warp per l (row of match), lanes over k: coalesced stores.  Deterministic two-level cost sum.
struct EmdFinalParams {
  const float* xyz1; const float* xyz2;   // [B,n,3], [B,m,3]
  const float* ratioL;                    // [LEVELS,B,n]
  const float* ratioR;                    // [LEVELS,B,m]
  float* match;                           // optional [B,m*n]
  float* partial;                         // [B, gridDim.x]
  float* cost;                            // [B]
  unsigned int* ticket;                   // [B] self-resetting
  const unsigned int* err;                // optional: nonzero = the persistent sweeps timed out -> cost = NaN
  int B, n, m;
  float lvl[EMD_LEVELS];
};

constexpr int EMD_FK = 1024;                                  // k-tile of the final pass
constexpr size_t EMD_FINAL_SMEM = (size_t)(EMD_LEVELS + 4) * EMD_FK * sizeof(float);
__global__ void __launch_bounds__(EMD_THREADS) emd_final_kernel(const EmdFinalParams p) {
  // the 10 ratioL rows of the current k-tile and the (negated) row cloud are staged once per CTA and shared by its
  // 8 match rows; a lane handles the pair (k, k + 32) with packed f32x2 arithmetic
  extern __shared__ __align__(16) float fsm[];
  float(*s_rl)[EMD_FK] = reinterpret_cast<float(*)[EMD_FK]>(fsm);
  float4* s_nx1 = reinterpret_cast<float4*>(fsm + EMD_LEVELS * EMD_FK);
  __shared__ float red[EMD_WARPS];
  __shared__ bool is_last;
  const int b = blockIdx.y;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int l = blockIdx.x * EMD_WARPS + warp;
  const float* x1 = p.xyz1 + (size_t)b * p.n * 3;
  const unsigned long long l2e2 = f2_pack(LOG2E, LOG2E);
  float acc = 0.f;
  float qx = 0.f, qy = 0.f, qz = 0.f;
  float rr[EMD_LEVELS];
#pragma unroll
  for (int j = 0; j < EMD_LEVELS; ++j) rr[j] = 0.f;
  if (l < p.m) {
    const float* q = p.xyz2 + ((size_t)b * p.m + l) * 3;
    qx = q[0]; qy = q[1]; qz = q[2];
#pragma unroll
    for (int j = 0; j < EMD_LEVELS; ++j) rr[j] = p.ratioR[((size_t)j * p.B + b) * p.m + l];
  }
  const unsigned long long qx2 = f2_pack(qx, qx), qy2 = f2_pack(qy, qy), qz2 = f2_pack(qz, qz);
  for (int k0 = 0; k0 < p.n; k0 += EMD_FK) {
    const int kn = min(EMD_FK, p.n - k0);
    __syncthreads();
    for (int i = tid; i < kn; i += EMD_THREADS) {
      const float* a = x1 + (size_t)(k0 + i) * 3;
      s_nx1[i] = make_float4(-a[0], -a[1], -a[2], 0.f);
#pragma unroll
      for (int j = 0; j < EMD_LEVELS; ++j) s_rl[j][i] = p.ratioL[((size_t)j * p.B + b) * p.n + k0 + i];
    }
    __syncthreads();
    if (l < p.m) {
      for (int kk = lane; kk < kn; kk += 64) {
        const bool v1 = kk + 32 < kn;
        const int k1 = v1 ? kk + 32 : kk;
        const float4 a0 = s_nx1[kk], a1 = s_nx1[k1];
        const unsigned long long dx = f2_add(qx2, f2_pack(a0.x, a1.x)), dy = f2_add(qy2, f2_pack(a0.y, a1.y)),
                                 dz = f2_add(qz2, f2_pack(a0.z, a1.z));
        const unsigned long long d2 = f2_fma(dz, dz, f2_fma(dx, dx, f2_mul(dy, dy)));
        unsigned long long mt = 0ull;
#pragma unroll
        for (int j = 0; j < EMD_LEVELS; ++j) {
          const unsigned long long rl = f2_pack(s_rl[j][kk], s_rl[j][k1]);
          const unsigned long long rj = f2_pack(rr[j], rr[j]);
          if (j == EMD_LEVELS - 1) {
            mt = f2_add(mt, f2_mul(rl, rj));                                // level 0: exp(0) = 1
          } else {
            float t0, t1;
            f2_unpack(f2_mul(f2_mul(f2_pack(p.lvl[j], p.lvl[j]), d2), l2e2), t0, t1);
            mt = f2_add(mt, f2_mul(f2_mul(f2_pack(ex2_approx(t0), ex2_approx(t1)), rl), rj));   // match += w (emd.cuh:157-158)
          }
        }
        float m0, m1, e0, e1;
        f2_unpack(mt, m0, m1);
        f2_unpack(d2, e0, e1);
        float* mrow = p.match ? p.match + (size_t)b * p.n * p.m + (size_t)l * p.n + k0 : nullptr;
        if (mrow) mrow[kk] = m0;
        acc = fmaf(sqrtf(e0), m0, acc);                                     // emd.cuh:225-226
        if (v1) {
          if (mrow) mrow[kk + 32] = m1;
          acc = fmaf(sqrtf(e1), m1, acc);
        }
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(L3D_FULL_MASK, acc, o);
  if (lane == 0) red[warp] = acc;
  __syncthreads();
  if (tid == 0) {
    float s = 0.f;
    for (int w = 0; w < EMD_WARPS; ++w) s += red[w];
    p.partial[(size_t)b * gridDim.x + blockIdx.x] = s;
    __threadfence();
    is_last = (atomicAdd(p.ticket + b, 1u) == gridDim.x - 1);
  }
  __syncthreads();
  if (is_last) {
    __threadfence();
    float a = 0.f;
    for (unsigned i = tid; i < gridDim.x; i += EMD_THREADS) a += __ldcg(p.partial + (size_t)b * gridDim.x + i);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(L3D_FULL_MASK, a, o);
    if (lane == 0) red[warp] = a;
    __syncthreads();
    if (tid == 0) {
      float s = 0.f;
      for (int w = 0; w < EMD_WARPS; ++w) s += red[w];
      p.cost[b] = (p.err && *p.err) ? __int_as_float(0x7fc00000) : s;
      p.ticket[b] = 0u;
    }
  }
}

// ---- gradients (match held constant) -------------------------------------------------------
// grad2[l] = sum_k match[l,k] (x2_l - x1_k) / max(|.|, 1e-10)   (emd.cuh:258-299): warp per l.
__global__ void __launch_bounds__(EMD_THREADS) emd_grad2_kernel(const float* __restrict__ xyz1,
                                                                const float* __restrict__ xyz2,
                                                                const float* __restrict__ match,
                                                                int n, int m, float* __restrict__ grad2) {
  const int b = blockIdx.y;
  const int lane = threadIdx.x & 31;
  const int l = blockIdx.x * EMD_WARPS + (threadIdx.x >> 5);
  if (l >= m) return;
  const float* x1 = xyz1 + (size_t)b * n * 3;
  const float* q = xyz2 + ((size_t)b * m + l) * 3;
  const float* mrow = match + (size_t)b * n * m + (size_t)l * n;
  const float qx = q[0], qy = q[1], qz = q[2];
  float gx = 0.f, gy = 0.f, gz = 0.f;
  for (int k = lane; k < n; k += 32) {
    const float dx = qx - x1[k * 3], dy = qy - x1[k * 3 + 1], dz = qz - x1[k * 3 + 2];
    const float d = mrow[k] * rsqrtf(fmaxf(fmaf(dz, dz, fmaf(dx, dx, dy * dy)), 1e-20f));
    gx = fmaf(dx, d, gx); gy = fmaf(dy, d, gy); gz = fmaf(dz, d, gz);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    gx += __shfl_xor_sync(L3D_FULL_MASK, gx, o);
    gy += __shfl_xor_sync(L3D_FULL_MASK, gy, o);
    gz += __shfl_xor_sync(L3D_FULL_MASK, gz, o);
  }
  if (lane == 0) {
    float* g = grad2 + ((size_t)b * m + l) * 3;
    g[0] = gx; g[1] = gy; g[2] = gz;
  }
}

// grad1[k] = sum_l match[l,k] (x1_k - x2_l) / max(|.|, 1e-10)   (emd.cuh:301-323): thread per k,
// coalesced along k, rows l split in `slices` (grid.y) whose partial sums are combined in a fixed
// order by emd_grad1_reduce_kernel (deterministic).
__global__ void __launch_bounds__(EMD_THREADS) emd_grad1_partial_kernel(
    const float* __restrict__ xyz1, const float* __restrict__ xyz2, const float* __restrict__ match,
    int n, int m, int slices, float* __restrict__ partial /*[B,slices,n,3]*/) {
  const int b = blockIdx.z, sl = blockIdx.y;
  const int k = blockIdx.x * EMD_THREADS + threadIdx.x;
  const int l0 = (int)((long)m * sl / slices), l1 = (int)((long)m * (sl + 1) / slices);
  if (k >= n) return;
  const float* p1 = xyz1 + ((size_t)b * n + k) * 3;
  const float px = p1[0], py = p1[1], pz = p1[2];
  const float* x2 = xyz2 + (size_t)b * m * 3;
  const float* mb = match + (size_t)b * n * m;
  float gx = 0.f, gy = 0.f, gz = 0.f;
  for (int l = l0; l < l1; ++l) {
    const float dx = px - __ldg(x2 + l * 3), dy = py - __ldg(x2 + l * 3 + 1), dz = pz - __ldg(x2 + l * 3 + 2);
    const float d = mb[(size_t)l * n + k] * rsqrtf(fmaxf(fmaf(dz, dz, fmaf(dx, dx, dy * dy)), 1e-20f));
    gx = fmaf(dx, d, gx); gy = fmaf(dy, d, gy); gz = fmaf(dz, d, gz);
  }
  float* o = partial + (((size_t)b * slices + sl) * n + k) * 3;
  o[0] = gx; o[1] = gy; o[2] = gz;
}
__global__ void __launch_bounds__(256) emd_grad1_reduce_kernel(const float* __restrict__ partial, int B,
                                                               int n, int slices, float* __restrict__ grad1) {
  const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long)B * n * 3) return;
  const int b = (int)(t / ((long)n * 3));
  const long r = t - (long)b * n * 3;
  float s = 0.f;
  for (int sl = 0; sl < slices; ++sl) s += partial[((size_t)b * slices + sl) * n * 3 + r];
  grad1[t] = s;
}

__global__ void emd_fill_kernel(float* dst, long n, float v, unsigned int* ticket, int B) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = v;
  if (i < B) ticket[i] = 0u;
}

static int emd_slices(int B, int n, int m) {
  int s = 1;
  const long ctas = (long)B * ((n + EMD_THREADS - 1) / EMD_THREADS);
  while (s < 32 && ctas * s < 296 && m / (s * 2) >= 16) s *= 2;
  return s;
}

}  // namespace l3d

using namespace l3d;

static thread_local int g_emd_force_multilaunch = 0;   // per host thread: a test toggling it cannot affect launches of other threads
// Testing hook: 0 = default (cooperative persistent launch), 1 = multi-launch (21 kernels), 2 = cooperative,
// 3 / 4 = one cluster of 16 / 8 CTAs per item (hardware cluster barriers, clouds resident in shared memory).
extern "C" void l3d_debug_emd_force_multilaunch(int mode) { g_emd_force_multilaunch = (mode >= 0 && mode <= 4) ? mode : 0; }

// workspace layout (floats): remainL[B,n] remainR[B,m] ratioL[LEVELS,B,n] ratioR[LEVELS,B,m]
//                            partial[B*gx] | ticket[B] arrive[B] err[1] (uint)
static size_t emd_fwd_ws_floats(int B, int n, int m) {
  const size_t gx = (size_t)(m + EMD_WARPS - 1) / EMD_WARPS;
  return (size_t)B * n + (size_t)B * m + (size_t)B * EMD_LEVELS * ((size_t)n + m) + (size_t)B * gx + 2 * (size_t)B + 1;
}
extern "C" size_t l3d_emd_forward_ws_bytes(int B, int n, int m) {
  if (B < 1 || n < 1 || m < 1) return 0;
  return sizeof(float) * emd_fwd_ws_floats(B, n, m);
}
extern "C" size_t l3d_emd_backward_ws_bytes(int B, int n, int m) {
  if (B < 1 || n < 1 || m < 1) return 0;
  return sizeof(float) * (size_t)B * emd_slices(B, n, m) * n * 3;
}

extern "C" int l3d_emd_forward(const float* xyz1_dev, const float* xyz2_dev, int B, int n, int m,
                               float* cost_dev, float* match_dev, void* ws_dev, void* stream) {
  if (!xyz1_dev || !xyz2_dev || !cost_dev || !ws_dev || B < 0 || n < 1 || m < 1 || B > 65535)
    return L3D_ERR_INVALID;
  if (B == 0) return L3D_OK;
  cudaStream_t s = (cudaStream_t)stream;
  float* ws = reinterpret_cast<float*>(ws_dev);
  float* remainL = ws;
  float* remainR = remainL + (size_t)B * n;
  float* ratioL = remainR + (size_t)B * m;
  float* ratioR = ratioL + (size_t)B * EMD_LEVELS * n;
  const unsigned gx_final = (unsigned)((m + EMD_WARPS - 1) / EMD_WARPS);
  float* partial = ratioR + (size_t)B * EMD_LEVELS * m;
  unsigned int* ticket = reinterpret_cast<unsigned int*>(partial + (size_t)B * gx_final);

  // multiL / multiR with the reference's INTEGER division (emd.cuh:10-16)
  const float multiL = (n >= m) ? 1.f : (float)(m / n);
  const float multiR = (n >= m) ? (float)(n / m) : 1.f;
  unsigned int* arrive = ticket + B;
  unsigned int* errw = arrive + B;
  EmdFinalParams fp{};
  for (int it = 0; it < EMD_LEVELS; ++it) fp.lvl[it] = emd_level(it);

  // ---- cluster path: one cluster of 16 (else 8) CTAs per item, hardware cluster barriers ------------------------
  bool clustered = false;
  // mode 0 (default) = cooperative persistent launch; 3 / 4 = cluster kernel with 16 / 8 CTAs per item (measured
  // slower at C5: 8 clusters of 16 one-CTA-per-SM blocks do not all fit at once, profiles/r02)
  if ((g_emd_force_multilaunch == 3 || g_emd_force_multilaunch == 4) && emd_cluster_smem(n, m) <= 200 * 1024) {
    static thread_local int c_dev = -1, c_nc = 0, c_mode = -1;
    if (c_mode != g_emd_force_multilaunch) { c_dev = -1; c_mode = g_emd_force_multilaunch; }
    int dev = 0;
    cudaGetDevice(&dev);
    const size_t smem = emd_cluster_smem(n, m);
    if (dev != c_dev) {
      c_nc = 0;
      cudaFuncSetAttribute(emd_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
      cudaFuncSetAttribute(emd_cluster_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
      for (int nc = (g_emd_force_multilaunch == 3 ? 16 : 8); nc >= 8 && !c_nc; nc >>= 1) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(nc); cfg.blockDim = dim3(EMDC_THREADS); cfg.dynamicSmemBytes = 200 * 1024;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = nc; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        int ncl = 0;
        if (cudaOccupancyMaxActiveClusters(&ncl, emd_cluster_kernel, &cfg) == cudaSuccess && ncl >= 1) c_nc = nc;
      }
      (void)cudaGetLastError();
      c_dev = dev;
    }
    if (c_nc > 0) {
      cudaError_t me = cudaMemsetAsync(ticket, 0, (2 * (size_t)B + 1) * sizeof(unsigned int), s);
      if (me != cudaSuccess) return (int)me;
      EmdPersistParams q{};
      q.xyz1 = xyz1_dev; q.xyz2 = xyz2_dev; q.remainL = remainL; q.remainR = remainR; q.ratioL = ratioL; q.ratioR = ratioR;
      q.arrive = arrive; q.err = errw; q.B = B; q.n = n; q.m = m; q.ctas_per_item = c_nc;
      q.multiL = multiL; q.multiR = multiR;
      for (int it = 0; it < EMD_LEVELS; ++it) q.lvl[it] = fp.lvl[it];
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3((unsigned)(B * c_nc)); cfg.blockDim = dim3(EMDC_THREADS); cfg.dynamicSmemBytes = smem;
      cfg.stream = s;
      cudaLaunchAttribute at[1];
      at[0].id = cudaLaunchAttributeClusterDimension;
      at[0].val.clusterDim.x = c_nc; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
      cfg.attrs = at; cfg.numAttrs = 1;
      if (cudaLaunchKernelEx(&cfg, emd_cluster_kernel, q) == cudaSuccess) {
        count_launch();
        clustered = true;
      } else {
        (void)cudaGetLastError();
      }
    }
  }

  // ---- persistent path: one cooperative launch runs all 20 sweeps (per-item barriers) ---------------------
  bool persistent = !clustered && g_emd_force_multilaunch != 1;
  int ctas_per_item = 0;
  if (persistent) {
    static thread_local int c_dev = -1, c_cap = 0;
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev != c_dev) {
      int occ = 0, coop = 0;
      cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev);
      const int sms = sm_count(dev);
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, emd_persistent_kernel, EMD_THREADS, 0) != cudaSuccess) occ = 0;
      if (occ > 4) occ = 4;                 // 32 warps/SM: while one item's CTAs sit in a barrier the others sweep
      c_cap = coop ? sms * occ : 0;
      c_dev = dev;
    }
    const int want = (std::max(n, m) + EMD_R - 1) / EMD_R;      // at least one warp's worth of rows per CTA
    ctas_per_item = c_cap / B;
    if (ctas_per_item > want) ctas_per_item = want;
    persistent = ctas_per_item >= 1;
  }
  if (persistent) {
    cudaError_t me = cudaMemsetAsync(ticket, 0, (2 * (size_t)B + 1) * sizeof(unsigned int), s);
    if (me != cudaSuccess) return (int)me;
    EmdPersistParams q{};
    q.xyz1 = xyz1_dev; q.xyz2 = xyz2_dev; q.remainL = remainL; q.remainR = remainR; q.ratioL = ratioL; q.ratioR = ratioR;
    q.arrive = arrive; q.err = errw; q.B = B; q.n = n; q.m = m; q.ctas_per_item = ctas_per_item;
    q.multiL = multiL; q.multiR = multiR;
    for (int it = 0; it < EMD_LEVELS; ++it) q.lvl[it] = fp.lvl[it];
    void* args[] = {&q};
    cudaError_t le = cudaLaunchCooperativeKernel((const void*)emd_persistent_kernel, dim3((unsigned)(B * ctas_per_item)),
                                                 dim3(EMD_THREADS), args, 0, s);
    if (le == cudaSuccess) {
      count_launch();
      fp.err = errw;
    } else {
      (void)cudaGetLastError();            // e.g. cudaErrorCooperativeLaunchTooLarge under MPS: take the multi-launch path
      persistent = false;
    }
  }
  if (!persistent && !clustered) {
  {
    // remainR = multiR (emd.cuh:24-25) and zero the arrival tickets
    const long tot = (long)B * m;
    emd_fill_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, s>>>(remainR, tot, multiR, ticket, B);
    count_launch();
    L3D_LAUNCH_CHECK();
  }
  const dim3 gridL((n + EMD_ROWS_PER_CTA - 1) / EMD_ROWS_PER_CTA, B);
  const dim3 gridR((m + EMD_ROWS_PER_CTA - 1) / EMD_ROWS_PER_CTA, B);
  for (int it = 0; it < EMD_LEVELS; ++it) {
    if (it == 0) {
      EmdSweepParams p{};
      p.rows = xyz1_dev; p.cols = xyz2_dev; p.B = B; p.nr = n; p.nc = m; p.phase = EMD_PH1;
      p.lvlA = fp.lvl[0]; p.vA = remainR; p.remain = remainL; p.ratio_out = ratioL;  // level 0 slot
      p.multi = multiL; p.init = 1;
      emd_sweep_kernel<false><<<gridL, EMD_THREADS, 0, s>>>(p);
      count_launch();
      L3D_LAUNCH_CHECK();
    }
    {
      EmdSweepParams p{};
      p.rows = xyz2_dev; p.cols = xyz1_dev; p.B = B; p.nr = m; p.nc = n; p.phase = EMD_PH2;
      p.lvlA = fp.lvl[it]; p.vA = ratioL + (size_t)it * B * n; p.remain = remainR;
      p.ratio_out = ratioR + (size_t)it * B * m;
      emd_sweep_kernel<false><<<gridR, EMD_THREADS, 0, s>>>(p);
      count_launch();
      L3D_LAUNCH_CHECK();
    }
    if (it + 1 < EMD_LEVELS) {
      EmdSweepParams p{};
      p.rows = xyz1_dev; p.cols = xyz2_dev; p.B = B; p.nr = n; p.nc = m; p.phase = EMD_PH3_PH1;
      p.lvlA = fp.lvl[it]; p.vA = ratioR + (size_t)it * B * m;
      p.lvlB = fp.lvl[it + 1]; p.vB = remainR;
      p.remain = remainL; p.ratio_in = ratioL + (size_t)it * B * n;
      p.ratio_out = ratioL + (size_t)(it + 1) * B * n;
      emd_sweep_kernel<true><<<gridL, EMD_THREADS, 0, s>>>(p);
      count_launch();
      L3D_LAUNCH_CHECK();
    }
  }
  }
  fp.xyz1 = xyz1_dev; fp.xyz2 = xyz2_dev; fp.ratioL = ratioL; fp.ratioR = ratioR;
  fp.match = match_dev; fp.partial = partial; fp.cost = cost_dev; fp.ticket = ticket;
  fp.B = B; fp.n = n; fp.m = m;
  {
    int dev = 0;
    cudaGetDevice(&dev);
    const cudaError_t e = raise_smem_once<emd_final_kernel>(dev, EMD_FINAL_SMEM);
    if (e != cudaSuccess) return (int)e;
  }
  emd_final_kernel<<<dim3(gx_final, B), EMD_THREADS, EMD_FINAL_SMEM, s>>>(fp);
  count_launch();
  L3D_LAUNCH_CHECK();
  return L3D_OK;
}

extern "C" int l3d_emd_backward(const float* xyz1_dev, const float* xyz2_dev, const float* match_dev,
                                int B, int n, int m, float* grad1_dev, float* grad2_dev, void* ws_dev,
                                void* stream) {
  if (!xyz1_dev || !xyz2_dev || !match_dev || !grad1_dev || !grad2_dev || !ws_dev || B < 0 || n < 1 ||
      m < 1 || B > 65535)
    return L3D_ERR_INVALID;
  if (B == 0) return L3D_OK;
  cudaStream_t s = (cudaStream_t)stream;
  emd_grad2_kernel<<<dim3((m + EMD_WARPS - 1) / EMD_WARPS, B), EMD_THREADS, 0, s>>>(
      xyz1_dev, xyz2_dev, match_dev, n, m, grad2_dev);
  count_launch();
  L3D_LAUNCH_CHECK();
  const int slices = emd_slices(B, n, m);
  float* partial = reinterpret_cast<float*>(ws_dev);
  emd_grad1_partial_kernel<<<dim3((n + EMD_THREADS - 1) / EMD_THREADS, slices, B), EMD_THREADS, 0, s>>>(
      xyz1_dev, xyz2_dev, match_dev, n, m, slices, partial);
  count_launch();
  L3D_LAUNCH_CHECK();
  const long tot = (long)B * n * 3;
  emd_grad1_reduce_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, s>>>(partial, B, n, slices, grad1_dev);
  count_launch();
  L3D_LAUNCH_CHECK();
  return L3D_OK;
}
