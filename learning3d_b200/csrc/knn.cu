// Fused pairwise-distance + top-k selection (sm_100a).
//
// Replaces, without ever materialising the B x M x N distance matrix:
//   knn()                       utils/model_common_utils.py:3-9      (MODE_EXPANSION_NEG)
//   pointconv_util.knn_point()  utils/pointconv_util.py:107-118      (MODE_SQDIST_EXP)
//   knn_point()                 utils/model_common_utils.py:84-100   (MODE_DIRECT_RN)
//   pointnet2 knn / three_nn    utils/lib/src/interpolate_gpu.cu:9-57,81-124 (MODE_DIRECT_FMA)
//
// Design (see DESIGN.md §3.1):
//   1. the candidate cloud of batch item b is bulk-copied (cp.async.bulk + mbarrier) into
//      shared memory once per CTA and repacked to float4 (x, y, z, |p|^2);
//   2. a warp owns KNN_R = 2 query rows at a time (k <= 24: knn_rows_v2) and each lane evaluates
//      32 candidates per 1024-candidate tile into registers, the candidate float4 shared by both rows;
//   3. the per-lane maxima are sorted across the warp: the k-th largest lane maximum T0 is a proven
//      lower bound of the k-th best key, so only keys >= T0 (about 1.5 k of them, found from the sign
//      bit of key - T0) survive; they are re-evaluated from shared memory into 64-bit composites
//      (order-preserving key bits << 32 | ~index), one or two per lane;
//   4. a flip + half-cleaner shuffle network sorts the composites (key desc, index asc) and the first
//      k are written with one coalesced store per row.
//   Larger k uses the generic knn_row<MODE,KS> (KS survivors per lane in shared memory); clouds with
//   N <= 256 and k*8 >= N sort the whole row in registers (knn_row_sort).  A row whose survivors
//   overflow (duplicate points, adversarial ties) is redone by an exact k-round arg-max scan
//   (knn_row_slow), so the result is always the full (key, index) order.
#include "common.cuh"
#include "knn_common.cuh"
#include "../../include/l3d_b200.h"
#include "launch_count.h"

#include <math.h>

namespace l3d {


constexpr int KNN_THREADS = 256;  // 128 (4 CTAs/SM) and 512 were slower (profiles/r01)
constexpr int KNN_WARPS = KNN_THREADS / 32;
constexpr int KNN_CHUNK = 1024;  // points per bulk-copy staging chunk
// Selection variants that were measured and dropped (profiles/r01, DESIGN.md §7): rank-by-counting
// against the shared-memory survivor list (40.9 us), an FMNMX key/value network with tie fallback
// (37.2 us) — both slower than the 64-bit composite network below (36.1 us at C2).
// Register budget: left to ptxas' own heuristic (127 registers at R = 2, 2 CTAs/SM), which measured
// fastest; forcing min-blocks 1..5 (48..167 registers) was 10-35 % slower (profiles/r01).
// Also measured and removed (the code is in git history before the change that removed it): a grid
// rounded to a multiple of B so that no CTA stages two clouds (34.7 vs 33.4 us), and a two-pass
// packed path that re-evaluates the keys for the survivor mask instead of holding 32 per row in
// registers (36.9 to 41.0 us against 34.9 us).
// 32-row units below which knn() stays on the warp-per-row-pair kernel (measured tie at 512:
// profiles/r02/knn_paths_time.txt)
constexpr int KNN_TPR_MIN_UNITS = 512;
constexpr int TPR_K_MAX = 24;
constexpr int KNN_R = 2;  // query rows per warp on the k <= 24 path (tuned in profiles/r01)
constexpr int KNN_SORT_MAX_N = 256;  // clouds this small may be sorted whole (8 keys per lane)

// Pair layout of a candidate tile for the packed path (expansion-mode k <= 24: two candidates per FFMA2):
// lane l's candidates e and e+1 (e even) of tile t, i.e. points j = t*1024 + e*32 + l and j + 32, sit side
// by side so that one LDS.128 feeds two FFMA2 operands:
//   pair_xy[t*512 + (e/2)*32 + l] = (x_e, x_e+1, y_e, y_e+1),  pair_zw[..] = (z_e, z_e+1, -|c_e|^2, -|c_e+1|^2)
template <int MODE, int KS>
struct KnnPairs { static constexpr bool value = MODE == MODE_EXPANSION_NEG && KS == 1; };


template <int S>
__device__ __forceinline__ void knn_store(const KnnParams& p, long row, int lane,
                                          const float (&v)[S], const uint32_t (&ix)[S]) {
#pragma unroll
  for (int s = 0; s < S; ++s) {
    const int pos = s * 32 + lane;
    if (pos < p.k) {
      const long o = row * p.k + pos;
      knn_store_index(p, o, ix[s]);
      if (p.out_val) p.out_val[o] = knn_val_xform(v[s], p.val_xform);
    }
  }
}

// Whole-row bitonic sort for small clouds (N <= 256): every candidate is a register slot.
template <int MODE>
__device__ __forceinline__ void knn_row_sort(const KnnParams& p, const float4* __restrict__ packed,
                                             const float4 q, long row, int lane) {
  constexpr int S = KNN_SORT_MAX_N / 32;
  float v[S];
  uint32_t ix[S];
#pragma unroll
  for (int s = 0; s < S; ++s) {
    const int j = s * 32 + lane;
    v[s] = (j < p.N) ? knn_key<MODE>(q, packed[j]) : -INFINITY;
    ix[s] = (j < p.N) ? (uint32_t)j : 0xffffffffu;
  }
  warp_bitonic_sort<S>(v, ix, lane);
  knn_store<S>(p, row, lane, v, ix);
}

// One query row, one warp.  KS = number of lane-group maxima per lane, in {1,2,4}.
template <int MODE, int KS>
__device__ __forceinline__ void knn_row(const KnnParams& p, const float4* __restrict__ packed,
                                        uint2* __restrict__ cbuf, const float4 q, long row,
                                        int ntiles, int lane) {
  constexpr int CAP = 64 * KS;   // survivors buffer (entries) per warp
  constexpr int GE = 32 / KS;    // registers per lane group
  const int k = p.k;

  int base = 0;            // entries carried over from earlier tiles (the running top-k)
  float kth = -INFINITY;   // key of the running k-th best
  bool overflow = (p.force_slow != 0);

  float rv[2 * KS];
  uint32_t ri[2 * KS];

  for (int t = 0; t < ntiles && !overflow; ++t) {
    float d[32];
    const float4* pt = packed + t * KNN_TILE + lane;
#pragma unroll
    for (int e = 0; e < 32; ++e) d[e] = knn_key<MODE>(q, pt[e * 32]);

    // k-th largest of the 32*KS lane-group maxima: at least k keys are >= T0
    float gm[KS];
#pragma unroll
    for (int g = 0; g < KS; ++g) {
      float m = d[g * GE];
#pragma unroll
      for (int e = 1; e < GE; ++e) m = fmaxf(m, d[g * GE + e]);
      gm[g] = m;
    }
    warp_bitonic_sort_keys<KS>(gm, lane);
    float t0 = gm[0];
#pragma unroll
    for (int g = 1; g < KS; ++g)
      if (((k - 1) >> 5) == g) t0 = gm[g];
    t0 = __shfl_sync(L3D_FULL_MASK, t0, (k - 1) & 31);
    const float thr = fmaxf(t0, kth);

    int cnt = 0;
#pragma unroll
    for (int e = 0; e < 32; ++e) cnt += (d[e] >= thr) ? 1 : 0;
    const int incl = warp_inclusive_scan(cnt, lane);
    const int total = __shfl_sync(L3D_FULL_MASK, incl, 31);
    if (base + total > CAP) { overflow = true; break; }

    int off = base + incl - cnt;
#pragma unroll
    for (int e = 0; e < 32; ++e) {
      if (d[e] >= thr) {
        cbuf[off] = make_uint2(__float_as_uint(d[e]), (uint32_t)(t * KNN_TILE + e * 32 + lane));
        ++off;
      }
    }
    __syncwarp();

    const int n_in = base + total;
    if (n_in <= 32 * KS) {
      float v[KS];
      uint32_t ix[KS];
#pragma unroll
      for (int s = 0; s < KS; ++s) {
        const int pos = s * 32 + lane;
        const uint2 c = cbuf[pos];   // buffer has CAP >= 32*KS entries: always in bounds
        const bool ok = pos < n_in;
        v[s] = ok ? __uint_as_float(c.x) : -INFINITY;
        ix[s] = ok ? c.y : 0xffffffffu;
      }
      warp_bitonic_sort<KS>(v, ix, lane);
#pragma unroll
      for (int s = 0; s < KS; ++s) { rv[s] = v[s]; ri[s] = ix[s]; }
    } else {
#pragma unroll
      for (int s = 0; s < 2 * KS; ++s) {
        const int pos = s * 32 + lane;
        const uint2 c = cbuf[pos];
        const bool ok = pos < n_in;
        rv[s] = ok ? __uint_as_float(c.x) : -INFINITY;
        ri[s] = ok ? c.y : 0xffffffffu;
      }
      warp_bitonic_sort<2 * KS>(rv, ri, lane);
    }
    __syncwarp();

    if (t + 1 < ntiles) {
      // carry the sorted top-k into the next tile as the first k buffer entries
      float kv = rv[0];
#pragma unroll
      for (int s = 0; s < KS; ++s) {
        const int pos = s * 32 + lane;
        if (pos < k) cbuf[pos] = make_uint2(__float_as_uint(rv[s]), ri[s]);
        if (((k - 1) >> 5) == s) kv = rv[s];
      }
      kth = __shfl_sync(L3D_FULL_MASK, kv, (k - 1) & 31);
      base = k;
      __syncwarp();
    }
  }

  if (overflow) {
    knn_row_slow<MODE>(p, packed, q, row, lane);
  } else {
    float v[KS];
    uint32_t ix[KS];
#pragma unroll
    for (int s = 0; s < KS; ++s) { v[s] = rv[s]; ix[s] = ri[s]; }
    knn_store<KS>(p, row, lane, v, ix);
  }
}

// R consecutive rows per warp: every candidate float4 is loaded from shared memory ONCE and used
// for R queries.  The second ncu capture showed the shared-memory/shuffle (MIO) pipe at 74 % with
// 128 of ~220 wavefronts per row being candidate loads: R = 2 halves them and doubles the ILP of
// the (shuffle-latency-bound) sorting networks.
template <int MODE, int R, bool PAIRS = false>
__device__ __forceinline__ void knn_rows_v2(const KnnParams& p, const float4* __restrict__ packed,
                                            unsigned long long* __restrict__ cbuf, const float4 (&q)[R],
                                            long row0, int ntiles, int lane,
                                            const ulonglong2* __restrict__ pair_xy = nullptr,
                                            const ulonglong2* __restrict__ pair_zw = nullptr) {
  constexpr int CAP = 64;
  const int k = p.k;
  int base[R];
  float kth[R];
  bool ovf[R];
  unsigned long long best[R];
#pragma unroll
  for (int r = 0; r < R; ++r) { base[r] = 0; kth[r] = -INFINITY; ovf[r] = (p.force_slow != 0); best[r] = 0ull; }

  for (int t = 0; t < ntiles; ++t) {
    // DEFER: the register copy of an expansion key leaves out the final "- |q|^2".  s -> RN(s - |q|^2)
    // is monotone, the registers only feed the threshold and the survivor mask (survivors are
    // re-evaluated with the full formula below), so the selection stays exact as long as the s-space
    // threshold is lowered to cover every s that can round to the k-th key (thr computation below).
    constexpr bool DEFER = MODE == MODE_EXPANSION_NEG;
    uint32_t mask[R];
    int cnt[R], incl[R], total[R];
    // the s-space threshold of a row from its sorted lane maxima (mx: lane l holds the l-th largest maximum)
    auto row_threshold = [&](int r, float mxr) -> float {
      float thr = __shfl_sync(L3D_FULL_MASK, mxr, k - 1);
      if (DEFER) {
        // kb: the exact key every survivor must reach (k-th lane maximum in key space, or the running
        // k-th best).  K(s) >= kb implies s >= kb + |q|^2 - ulp(kb)/2, so rounding that bound DOWN
        // (twice, with |kb| 2^-23 >= ulp/2 as the margin) keeps every such s; it admits at most the
        // few s within ~2 ulp below, which the exact re-evaluation sorts out.
        const float kb = fmaxf(__fsub_rn(thr, q[r].w), kth[r]);
        thr = __fadd_rd(__fadd_rd(kb, q[r].w), -__fmul_rn(fmaxf(fabsf(kb), 1e-30f), 1.1920929e-7f));
      } else {
        thr = fmaxf(thr, kth[r]);
      }
      return thr;
    };
    float d[R][32];
    if constexpr (PAIRS) {
      // two candidates per instruction: s = fma(2, fma(qz,cz, fma(qy,cy, qx*cx)), -|c|^2), same op order per lane
      const ulonglong2* pxy = pair_xy + t * (KNN_TILE / 2) + lane;
      const ulonglong2* pzw = pair_zw + t * (KNN_TILE / 2) + lane;
      unsigned long long qx2[R], qy2[R], qz2[R];
#pragma unroll
      for (int r = 0; r < R; ++r) { qx2[r] = f2_pack(q[r].x, q[r].x); qy2[r] = f2_pack(q[r].y, q[r].y); qz2[r] = f2_pack(q[r].z, q[r].z); }
      const unsigned long long two2 = f2_pack(2.0f, 2.0f);
#pragma unroll
      for (int pe = 0; pe < 16; ++pe) {
        const ulonglong2 a = pxy[pe * 32], bz = pzw[pe * 32];
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const unsigned long long dot = f2_fma(qz2[r], bz.x, f2_fma(qy2[r], a.y, f2_mul(qx2[r], a.x)));
          f2_unpack(f2_fma(two2, dot, bz.y), d[r][2 * pe], d[r][2 * pe + 1]);
        }
      }
    } else {
      const float4* pt = packed + t * KNN_TILE + lane;
#pragma unroll
      for (int e = 0; e < 32; ++e) {
        const float4 c = pt[e * 32];
#pragma unroll
        for (int r = 0; r < R; ++r) {
          if (DEFER) d[r][e] = fmaf(2.0f, fmaf(q[r].z, c.z, fmaf(q[r].y, c.y, __fmul_rn(q[r].x, c.x))), -c.w);
          else d[r][e] = knn_key<MODE>(q[r], c);
        }
      }
    }
    float mx[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      float m = d[r][0];
#pragma unroll
      for (int e = 1; e < 32; ++e) m = fmaxf(m, d[r][e]);
      mx[r] = m;
    }
    warp_sort32_keys_desc_x<R>(mx, lane);
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const float thr = row_threshold(r, mx[r]);
      // survivor mask: bit e = (d[e] >= thr).  d - thr is +0 on equality, so the survivors are the
      // differences with a clear sign bit; one FADD (FMA pipe) + one funnel shift (ALU pipe) per key
      // instead of FSETP + predicated OR (two ALU-pipe instructions; the ALU pipe is the busier one).
      uint32_t neg = 0u;
      if constexpr (PAIRS) {
        const unsigned long long nthr = f2_pack(-thr, -thr);
#pragma unroll
        for (int pe = 15; pe >= 0; --pe) {
          float s0, s1;
          f2_unpack(f2_add(f2_pack(d[r][2 * pe], d[r][2 * pe + 1]), nthr), s0, s1);
          neg = __funnelshift_l(__float_as_uint(s1), neg, 1);
          neg = __funnelshift_l(__float_as_uint(s0), neg, 1);
        }
      } else {
#pragma unroll
        for (int e = 31; e >= 0; --e)
          neg = __funnelshift_l(__float_as_uint(__fsub_rn(d[r][e], thr)), neg, 1);
      }
      const uint32_t mk = ~neg;
      mask[r] = mk;
      cnt[r] = __popc(mk);
    }
#pragma unroll
    for (int r = 0; r < R; ++r) incl[r] = warp_inclusive_scan(cnt[r], lane);
#pragma unroll
    for (int r = 0; r < R; ++r) {
      total[r] = __shfl_sync(L3D_FULL_MASK, incl[r], 31);
      if (base[r] + total[r] > CAP) ovf[r] = true;
    }
#pragma unroll
    for (int r = 0; r < R; ++r) {
      if (ovf[r]) continue;
      unsigned long long* cb = cbuf + r * CAP;
      if (base[r] && lane < base[r]) cb[lane] = best[r];
      int off = base[r] + incl[r] - cnt[r];
      uint32_t mk = mask[r];
      while (mk) {
        const int e = __ffs(mk) - 1;
        mk &= mk - 1;
        const int j = t * KNN_TILE + e * 32 + lane;
        cb[off++] = pack_pair(knn_key<MODE>(q[r], packed[j]), (uint32_t)j);
      }
    }
    __syncwarp();
    // first 32 survivors of every row: one straight-line network over all R rows (the exchanges of
    // different rows are independent, so their shuffle latencies overlap)
    unsigned long long a[R];
    int n_in[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      n_in[r] = base[r] + total[r];
      a[r] = (lane < n_in[r]) ? cbuf[r * CAP + lane] : 0ull;
    }
    warp_sort32_desc_x<R>(a, lane);
#pragma unroll
    for (int r = 0; r < R; ++r) {
      if (n_in[r] > 32 && !ovf[r]) {
        // survivors 32..63: sort them too, pair a[i] with b[31-i], keep the better 32, clean up
        unsigned long long b = (lane + 32 < n_in[r]) ? cbuf[r * CAP + lane + 32] : 0ull;
        b = shfl_xor_u64(warp_sort32_desc(b, lane), 31);
        unsigned long long c = (b > a[r]) ? b : a[r];
#pragma unroll
        for (int j = 16; j > 0; j >>= 1) c = cmpx_u64(c, j, (lane & j) == 0);
        a[r] = c;
      }
      best[r] = a[r];
      if (t + 1 < ntiles) {
        kth[r] = f32_unorder(__shfl_sync(L3D_FULL_MASK, (uint32_t)(best[r] >> 32), k - 1));
        base[r] = k;
      }
    }
    __syncwarp();
  }
#pragma unroll
  for (int r = 0; r < R; ++r) {
    if (ovf[r]) knn_row_slow<MODE>(p, packed, q[r], row0 + r, lane);
    else knn_store_packed(p, row0 + r, lane, best[r]);
  }
}

// Dynamic shared memory layout (bytes):
//   [0,16)                       mbarrier
//   [16, 16 + 12*KNN_CHUNK)      raw staging chunk (3 * KNN_CHUNK floats)
//   [.., + 16*NPAD)              packed candidates (float4), NPAD = N rounded up to KNN_TILE
//   [.., + 16*NPAD)              pair layout of the same candidates (packed-f32x2 path only, KnnPairs<>)
//   [.., + KNN_WARPS*CAP*8)      per-warp survivor buffers
// survivor-buffer entries per warp: KS = 1 runs KNN_R rows per warp, 64 entries each
#define KNN_CBUF(KS) ((KS) == 1 ? 64 * KNN_R : 64 * (KS))
__host__ __device__ inline size_t knn_smem_bytes(int N, int KS, bool pairs) {
  const size_t npad = (size_t)((N + KNN_TILE - 1) / KNN_TILE) * KNN_TILE;
  return 16 + 12 * (size_t)KNN_CHUNK + 16 * npad * (pairs ? 2 : 1) + (size_t)KNN_WARPS * KNN_CBUF(KS) * 8;
}

template <int MODE, int KS, bool SELF, bool CAND_BCN, bool FEAT = false, bool PAIRS = false>
__global__ void __launch_bounds__(KNN_THREADS) knn_kernel(const KnnParams p) {
  extern __shared__ __align__(128) unsigned char smem[];
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem);
  float* stage = reinterpret_cast<float*>(smem + 16);
  float4* packed = reinterpret_cast<float4*>(smem + 16 + 12 * KNN_CHUNK);
  const int N = p.N, M = p.M;
  const int ntiles = (N + KNN_TILE - 1) / KNN_TILE;
  const int npad = ntiles * KNN_TILE;
  static_assert(!PAIRS || KnnPairs<MODE, KS>::value, "the packed path exists for the k <= 24 expansion mode only");
  ulonglong2* pair_xy = reinterpret_cast<ulonglong2*>(packed + npad);          // npad/2 entries each
  ulonglong2* pair_zw = pair_xy + npad / 2;
  uint2* cbuf_all = reinterpret_cast<uint2*>(packed + (PAIRS ? 2 : 1) * npad);

  const int tid = threadIdx.x;
  const int lane = tid & 31, warp = tid >> 5;
  uint2* cbuf = cbuf_all + warp * KNN_CBUF(KS);

  if (tid == 0) {
    mbar_init(bar, 1);
    fence_mbar_init();
  }
  __syncthreads();
  uint32_t parity = 0;
  // programmatic dependent launch: let the next launch on the stream start filling SMs as our CTAs
  // retire, and do not touch global memory before the previous launch has fully completed
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");

  const long rows_total = (long)p.B * M;
  const long r0 = rows_total * blockIdx.x / gridDim.x;
  const long r1 = rows_total * (blockIdx.x + 1) / gridDim.x;

  for (long seg = r0; seg < r1;) {
    const int b = (int)(seg / M);
    const long seg_end = min(r1, (long)(b + 1) * M);

    // ---- stage candidate cloud b: bulk copy -> repack to (x,y,z,|p|^2) ---------------
    const float* src = p.cand + (size_t)b * 3 * N;
    for (int j0 = 0; j0 < N; j0 += KNN_CHUNK) {
      const int cnt = min(KNN_CHUNK, N - j0);
      if (p.use_tma) {
        if (tid == 0) {
          mbar_arrive_expect_tx(bar, (uint32_t)cnt * 12u);
          if (CAND_BCN) {
            bulk_g2s(stage, src + j0, (uint32_t)cnt * 4u, bar);
            bulk_g2s(stage + KNN_CHUNK, src + N + j0, (uint32_t)cnt * 4u, bar);
            bulk_g2s(stage + 2 * KNN_CHUNK, src + 2 * (size_t)N + j0, (uint32_t)cnt * 4u, bar);
          } else {
            bulk_g2s(stage, src + (size_t)j0 * 3, (uint32_t)cnt * 12u, bar);
          }
        }
        mbar_wait(bar, parity);
        parity ^= 1u;
      } else {
        if (CAND_BCN) {
          for (int i = tid; i < cnt; i += KNN_THREADS) {
            stage[i] = src[j0 + i];
            stage[KNN_CHUNK + i] = src[N + j0 + i];
            stage[2 * KNN_CHUNK + i] = src[2 * (size_t)N + j0 + i];
          }
        } else {
          for (int i = tid; i < cnt * 3; i += KNN_THREADS) stage[i] = src[(size_t)j0 * 3 + i];
        }
        __syncthreads();
      }
      for (int i = tid; i < cnt; i += KNN_THREADS) {
        float x, y, z;
        if (CAND_BCN) { x = stage[i]; y = stage[KNN_CHUNK + i]; z = stage[2 * KNN_CHUNK + i]; }
        else { x = stage[3 * i]; y = stage[3 * i + 1]; z = stage[3 * i + 2]; }
        packed[j0 + i] = knn_pack<MODE>(x, y, z);
      }
      __syncthreads();  // staging chunk may be overwritten; packed[] visible
    }
    for (int i = N + tid; i < npad; i += KNN_THREADS) packed[i] = knn_padding<MODE>();
    __syncthreads();
    if (PAIRS && !(p.full_sort && !p.force_slow)) {
      // pair layout for the packed-f32x2 distance loop: thread = (tile, pair, lane); two conflict-free
      // LDS.128 in, two STS.128 out
      for (int i = tid; i < npad / 2; i += KNN_THREADS) {
        const int t = i >> 9, pe = (i >> 5) & 15, l = i & 31;
        const float4 c0 = packed[t * KNN_TILE + (2 * pe) * 32 + l], c1 = packed[t * KNN_TILE + (2 * pe + 1) * 32 + l];
        pair_xy[i] = make_ulonglong2(f2_pack(c0.x, c1.x), f2_pack(c0.y, c1.y));
        pair_zw[i] = make_ulonglong2(f2_pack(c0.z, c1.z), f2_pack(-c0.w, -c1.w));
      }
      __syncthreads();
    }

    // ---- rows of this segment, one warp each ---------------------------------------
    auto load_query = [&](long row) -> float4 {
      if (SELF) return packed[(int)(row - (long)b * M)];
      const float* qp = p.query + row * 3;
      return knn_pack<MODE>(qp[0], qp[1], qp[2]);
    };
    // get_graph_feature() fused into knn() (SURVEY.md §8d "a1+a2"): the neighbours' coordinates are still
    // in shared memory when a row's indices are final, so cat(x[nbr], x[centre]) — [B,6,N,k] — is written
    // here and the separate gather launch (and its re-read of 5.2 MB of indices) disappears.  The row's own
    // warp re-reads the k indices it has just stored (L1) after a __syncwarp, so every selection path
    // (network / whole-row sort / exact scan) is covered by one helper.
    auto emit_feature = [&](long row) {
      if (!(FEAT && SELF)) return;   // compile-time: the plain knn() kernel carries none of this
      __syncwarp();
      const int n = (int)(row - (long)b * M);
      const float4 ctr = packed[n];
      const size_t cs = (size_t)N * p.k;
      for (int pos = lane; pos < p.k; pos += 32) {
        const long o = row * p.k + pos;
        const int j = p.idx64 ? (int)reinterpret_cast<const volatile long long*>(p.out_idx)[o]
                              : reinterpret_cast<const volatile int*>(p.out_idx)[o];
        const float4 c = packed[j];
        float* f = p.feat_out + ((size_t)b * 6 * N + n) * p.k + pos;
        f[0] = c.x; f[cs] = c.y; f[2 * cs] = c.z;
        f[3 * cs] = ctr.x; f[4 * cs] = ctr.y; f[5 * cs] = ctr.z;
      }
    };
    if (KS == 1 && !(p.full_sort && !p.force_slow)) {
      // KNN_R consecutive rows per warp; a ragged tail falls back to one row at a time
      unsigned long long* cb = reinterpret_cast<unsigned long long*>(cbuf);
      long row = seg + (long)warp * KNN_R;
      for (; row + KNN_R <= seg_end; row += (long)KNN_WARPS * KNN_R) {
        float4 q[KNN_R];
#pragma unroll
        for (int r = 0; r < KNN_R; ++r) q[r] = load_query(row + r);
        knn_rows_v2<MODE, KNN_R, PAIRS>(p, packed, cb, q, row, ntiles, lane, pair_xy, pair_zw);
#pragma unroll
        for (int r = 0; r < KNN_R; ++r) emit_feature(row + r);
      }
      for (; row < seg_end; ++row) {
        const float4 q1[1] = {load_query(row)};
        knn_rows_v2<MODE, 1>(p, packed, cb, q1, row, ntiles, lane);
        emit_feature(row);
      }
    } else {
      for (long row = seg + warp; row < seg_end; row += KNN_WARPS) {
        const float4 q = load_query(row);
        if (KS == 1) knn_row_sort<MODE>(p, packed, q, row, lane);
        else knn_row<MODE, KS>(p, packed, cbuf, q, row, ntiles, lane);
        emit_feature(row);
      }
    }
    seg = seg_end;
    __syncthreads();  // all warps done with packed[] before the next cloud is staged
  }
}

// ---- clouds beyond the shared-memory-resident path (N > L3D_KNN_MAX_N): streaming selection -------------------------
// The reference's knn() is torch.matmul + topk and has no size limit (model_common_utils.py:3-9); the resident kernel
// above keeps the whole candidate cloud in shared memory.  Here the cloud is streamed through a 32 KB tile, one query
// row per warp, and every warp keeps its running top-k as a sorted list of 64-bit composites (same key arithmetic,
// same (key desc, index asc) order as every other path).  Candidates arrive in index order, so a candidate enters the
// list only when its composite beats the current k-th entry; the expected number of insertions per row is
// ~k (1 + ln(N / k)), against N key evaluations.
constexpr int KNN_STREAM_TILE = 2048;
constexpr int KNN_STREAM_WARPS = 8;
constexpr int KNN_STREAM_MAX_K = 2048;

__host__ __device__ inline size_t knn_stream_smem_bytes(int k) {
  return (size_t)KNN_STREAM_TILE * 16 + (size_t)KNN_STREAM_WARPS * (size_t)((k + 31) & ~31) * 8;
}

template <int MODE, bool SELF, bool CAND_BCN>
__global__ void __launch_bounds__(KNN_STREAM_WARPS * 32) knn_stream_kernel(const KnnParams p) {
  extern __shared__ __align__(128) unsigned char smem[];
  float4* tile = reinterpret_cast<float4*>(smem);
  const int N = p.N, M = p.M, k = p.k;
  const int kpad = (k + 31) & ~31;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  unsigned long long* list = reinterpret_cast<unsigned long long*>(tile + KNN_STREAM_TILE) + (size_t)warp * kpad;

  const int row_blocks = (M + KNN_STREAM_WARPS - 1) / KNN_STREAM_WARPS;
  const int b = (int)(blockIdx.x / row_blocks);
  const int m = (int)(blockIdx.x % row_blocks) * KNN_STREAM_WARPS + warp;
  const bool live = m < M;
  const long row = (long)b * M + m;
  const float* src = p.cand + (size_t)b * 3 * N;

  float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
  if (live) {
    if (SELF) {
      q = CAND_BCN ? knn_pack<MODE>(src[m], src[(size_t)N + m], src[2 * (size_t)N + m])
                   : knn_pack<MODE>(src[3 * (size_t)m], src[3 * (size_t)m + 1], src[3 * (size_t)m + 2]);
    } else {
      const float* qp = p.query + row * 3;
      q = knn_pack<MODE>(qp[0], qp[1], qp[2]);
    }
  }
  for (int i = lane; i < kpad; i += 32) list[i] = 0ull;     // below every real composite
  __syncwarp();
  unsigned long long kth = 0ull;

  for (int t0 = 0; t0 < N; t0 += KNN_STREAM_TILE) {
    const int cnt = min(KNN_STREAM_TILE, N - t0);
    __syncthreads();                                          // the previous tile has been consumed
    for (int i = tid; i < cnt; i += KNN_STREAM_WARPS * 32) {
      const size_t j = (size_t)t0 + i;
      tile[i] = CAND_BCN ? knn_pack<MODE>(src[j], src[(size_t)N + j], src[2 * (size_t)N + j])
                         : knn_pack<MODE>(src[3 * j], src[3 * j + 1], src[3 * j + 2]);
    }
    __syncthreads();
    if (!live) continue;
    for (int j0 = 0; j0 < cnt; j0 += 32) {
      const int j = j0 + lane;
      const unsigned long long c = (j < cnt) ? pack_pair(knn_key<MODE>(q, tile[j]), (uint32_t)(t0 + j)) : 0ull;
      unsigned todo = __ballot_sync(L3D_FULL_MASK, c > kth);
      while (todo) {
        const int from = __ffs(todo) - 1;                     // lowest index first: equal keys keep their index order
        todo &= todo - 1;
        const unsigned long long cc = shfl_u64(c, from);
        if (cc <= kth) continue;                              // the threshold rose since the ballot
        int pos = 0;                                          // entries strictly better than cc
        for (int base = 0; base < k; base += 32) {
          const unsigned long long e = (base + lane < k) ? list[base + lane] : 0ull;
          const int n = __popc(__ballot_sync(L3D_FULL_MASK, e > cc));
          pos += n;
          if (n < 32) break;
        }
        for (int hi = k - 1; hi > pos; hi -= 32) {            // shift [pos, k-2] one slot down the list, top chunk first
          const int i = hi - lane;
          const unsigned long long v = (i > pos) ? list[i - 1] : 0ull;
          __syncwarp();
          if (i > pos) list[i] = v;
          __syncwarp();
        }
        if (lane == 0) list[pos] = cc;
        __syncwarp();
        kth = list[k - 1];
      }
    }
  }
  if (!live) return;
  __syncwarp();
  for (int pos = lane; pos < k; pos += 32) knn_store_packed(p, row, pos, list[pos]);
}

// ---- host side -----------------------------------------------------------------------
static thread_local int g_force_slow = 0;   // testing hooks are per host thread
int knn_force_slow_flag() { return g_force_slow; }   // knn_matrix.cu shares the testing hook

template <int MODE, int KS, bool SELF, bool CAND_BCN, bool FEAT = false, bool PAIRS = false>
static int knn_launch_t(KnnParams p, cudaStream_t stream) {
  if constexpr (!PAIRS && KnnPairs<MODE, KS>::value) {
    // packed-f32x2 variant whenever its second copy of the cloud fits in shared memory (N <= 6144)
    if (knn_smem_bytes(p.N, KS, true) <= KNN_SMEM_LIMIT)
      return knn_launch_t<MODE, KS, SELF, CAND_BCN, FEAT, true>(p, stream);
  }
  constexpr auto kern = knn_kernel<MODE, KS, SELF, CAND_BCN, FEAT, PAIRS>;
  const size_t smem = knn_smem_bytes(p.N, KS, PAIRS);
  if (smem > KNN_SMEM_LIMIT) return L3D_ERR_UNSUPPORTED;
  int dev = 0;
  cudaGetDevice(&dev);
  // raised to the architectural maximum, whatever N this call needs
  const cudaError_t ae = raise_smem_once<kern>(dev, KNN_SMEM_LIMIT);
  if (ae != cudaSuccess) return (int)ae;
  // the occupancy query is a host-side driver call (~3 us): cache it per (thread, device, smem size)
  static thread_local int c_dev = -1, c_occ = 0;
  static thread_local size_t c_smem = 0;
  if (dev != c_dev || smem != c_smem) {
    int o = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, kern, KNN_THREADS, smem);
    if (e != cudaSuccess) return (int)e;
    c_dev = dev; c_smem = smem; c_occ = o;
  }
  int occ = c_occ;
  if (occ < 1) return L3D_ERR_UNSUPPORTED;
  if (occ > 4) occ = 4;
  const long rows = (long)p.B * p.M;
  long grid = (long)sm_count(dev) * occ;       // persistent-style: every CTA resident at once
  const long max_useful = (rows + KNN_WARPS - 1) / KNN_WARPS;
  if (grid > max_useful) grid = max_useful;
  if (grid < 1) grid = 1;
  return knn_launch_pdl(kern, grid, KNN_THREADS, smem, stream, p);
}

extern "C" int l3d_graph_feature(const float* x_dev, const int64_t* idx_dev, int B, int C, int N, int k,
                                 float* out_dev, void* stream);

template <int MODE, bool SELF, bool CAND_BCN>
static int knn_stream_launch(KnnParams p, cudaStream_t stream) {
  if (p.k > KNN_STREAM_MAX_K) return L3D_ERR_UNSUPPORTED;
  if (p.idx64 == 2 && p.N > 65536) return L3D_ERR_UNSUPPORTED;          // 16-bit wire format of the host path
  constexpr auto kern = knn_stream_kernel<MODE, SELF, CAND_BCN>;
  const size_t smem = knn_stream_smem_bytes(p.k);
  if (smem > 48 * 1024) {
    // raised to the largest size this path can ask for
    int dev = 0;
    cudaGetDevice(&dev);
    const cudaError_t e = raise_smem_once<kern>(dev, knn_stream_smem_bytes(KNN_STREAM_MAX_K));
    if (e != cudaSuccess) return (int)e;
  }
  const long row_blocks = ((long)p.M + KNN_STREAM_WARPS - 1) / KNN_STREAM_WARPS;
  const long grid = (long)p.B * row_blocks;
  if (grid > 0x7fffffffL) return L3D_ERR_UNSUPPORTED;
  kern<<<(unsigned)grid, KNN_STREAM_WARPS * 32, smem, stream>>>(p);
  count_launch();
  L3D_LAUNCH_CHECK();
  if (p.feat_out)   // get_graph_feature on the finished indices (the fused variant needs the cloud resident on chip)
    return l3d_graph_feature(p.cand, (const int64_t*)p.out_idx, p.B, 3, p.N, p.k, p.feat_out, (void*)stream);
  return L3D_OK;
}

template <int MODE, bool SELF, bool CAND_BCN>
static int knn_launch(KnnParams p, cudaStream_t stream) {
  if (p.B < 0 || p.N < 1 || p.M < 0 || p.k < 1 || p.k > p.N) return L3D_ERR_INVALID;
  if ((long)p.B * p.M == 0) return L3D_OK;   // empty batch: nothing to do (its pointers may be null)
  if (!p.cand || !p.out_idx || (!SELF && !p.query)) return L3D_ERR_INVALID;
  if (p.N > L3D_KNN_MAX_N) return knn_stream_launch<MODE, SELF, CAND_BCN>(p, stream);   // streamed, any N
  // k > 128 (the reference's pointnet2 knn allows 200, torch.topk any k): beyond the survivor buffers of the
  // threshold scheme -> every row takes the exact k-round arg-max scan (O(k N) per row, same ordering rule)
  p.force_slow = (g_force_slow || p.k > 128) ? 1 : 0;
  p.use_tma = ((reinterpret_cast<uintptr_t>(p.cand) & 15u) == 0 && (p.N & 3) == 0) ? 1 : 0;
  // Heavy selections out of a small cloud (FlowNet3D's flow embedding: k = 64 of N = 256) sort the
  // whole row instead of thresholding it.
  if (p.N <= KNN_SORT_MAX_N && p.k * 8 >= p.N) p.full_sort = 1;
  if constexpr (SELF && CAND_BCN && MODE == MODE_EXPANSION_NEG) {
    // knn() on xyz with enough rows to give every SM sub-partition a warp of 32 rows: thread-per-row kernel
    // (knn_tpr.cu, bit-identical results); smaller batches keep the warp-per-row-pair kernel below
    if (!p.full_sort && !(p.k > TPR_K_MAX) && knn_path_flag() != 1 && knn_tpr_eligible(p) &&
        (knn_path_flag() == 2 || (long)p.B * (p.N / 32) >= KNN_TPR_MIN_UNITS))
      return knn_tpr_launch(p, stream);
  }
  if (SELF && CAND_BCN && MODE == MODE_EXPANSION_NEG && p.feat_out) {   // fused get_graph_feature variant
    if (p.full_sort || p.k <= 24) return knn_launch_t<MODE, 1, SELF, CAND_BCN, SELF && CAND_BCN>(p, stream);
    if (p.k <= 48) return knn_launch_t<MODE, 2, SELF, CAND_BCN, SELF && CAND_BCN>(p, stream);
    return knn_launch_t<MODE, 4, SELF, CAND_BCN, SELF && CAND_BCN>(p, stream);
  }
  if (p.full_sort) return knn_launch_t<MODE, 1, SELF, CAND_BCN>(p, stream);
  // KS sets the number of lane groups (32*KS) whose maxima bound the k-th best key; the expected
  // number of survivors stays below the 64*KS-entry buffer while k <= ~0.75 * 32 * KS
  // (N = 1024: k = 24 -> 43, k = 48 -> 85, k = 100 -> ~170 survivors).  Larger k / N ratios still
  // work (exact slow path) but lose the fast path.
  if (p.k <= 24) return knn_launch_t<MODE, 1, SELF, CAND_BCN>(p, stream);
  if (p.k <= 48) return knn_launch_t<MODE, 2, SELF, CAND_BCN>(p, stream);
  return knn_launch_t<MODE, 4, SELF, CAND_BCN>(p, stream);
}

}  // namespace l3d

using namespace l3d;

extern "C" void l3d_debug_force_slow_path(int on) { l3d::g_force_slow = on ? 1 : 0; }

extern "C" int l3d_knn_expansion(const float* x_dev, int B, int N, int k, int64_t* idx_dev,
                                 float* val_dev, void* stream) {
  KnnParams p{};
  p.cand = x_dev; p.query = nullptr; p.out_idx = idx_dev; p.out_val = val_dev;
  p.B = B; p.N = N; p.M = N; p.k = k; p.idx64 = 1; p.val_xform = 0;
  return knn_launch<MODE_EXPANSION_NEG, true, true>(p, (cudaStream_t)stream);
}

// knn() with 16-bit indices (N <= 65536 always holds: N <= L3D_KNN_MAX_N): the device half of
// l3d_knn_expansion_host, which moves 2 instead of 8 bytes per index over PCIe and widens on the host.
namespace l3d {
int knn_expansion_u16(const float* x_dev, int B, int N, int k, unsigned short* idx_dev, cudaStream_t stream) {
  KnnParams p{};
  p.cand = x_dev; p.query = nullptr; p.out_idx = idx_dev; p.out_val = nullptr;
  p.B = B; p.N = N; p.M = N; p.k = k; p.idx64 = 2; p.val_xform = 0;
  return knn_launch<MODE_EXPANSION_NEG, true, true>(p, stream);
}
}  // namespace l3d

extern "C" int l3d_knn_graph_feature(const float* x_dev, int B, int N, int k, int64_t* idx_dev,
                                     float* feat_dev, void* stream) {
  if (!feat_dev) return L3D_ERR_INVALID;
  KnnParams p{};
  p.cand = x_dev; p.query = nullptr; p.out_idx = idx_dev; p.out_val = nullptr; p.feat_out = feat_dev;
  p.B = B; p.N = N; p.M = N; p.k = k; p.idx64 = 1; p.val_xform = 0;
  return knn_launch<MODE_EXPANSION_NEG, true, true>(p, (cudaStream_t)stream);
}

extern "C" int l3d_knn_point(const float* data_dev, const float* query_dev, int B, int N, int M,
                             int k, float* val_dev, int64_t* idx_dev, void* stream) {
  KnnParams p{};
  p.cand = data_dev; p.query = query_dev; p.out_idx = idx_dev; p.out_val = val_dev;
  p.B = B; p.N = N; p.M = M; p.k = k; p.idx64 = 1; p.val_xform = 2;
  return knn_launch<MODE_DIRECT_RN, false, false>(p, (cudaStream_t)stream);
}

extern "C" int l3d_knn_sqdist(const float* xyz_dev, const float* new_xyz_dev, int B, int N, int S,
                              int nsample, int64_t* idx_dev, void* stream) {
  KnnParams p{};
  p.cand = xyz_dev; p.query = new_xyz_dev; p.out_idx = idx_dev; p.out_val = nullptr;
  p.B = B; p.N = N; p.M = S; p.k = nsample; p.idx64 = 1; p.val_xform = 1;
  return knn_launch<MODE_SQDIST_EXP, false, false>(p, (cudaStream_t)stream);
}

extern "C" int l3d_pn2_knn(int b, int n, int m, int k, const float* unknown_dev,
                           const float* known_dev, float* dist2_dev, int32_t* idx_dev,
                           void* stream) {
  KnnParams p{};
  p.cand = known_dev; p.query = unknown_dev; p.out_idx = idx_dev; p.out_val = dist2_dev;
  p.B = b; p.N = m; p.M = n; p.k = k; p.idx64 = 0; p.val_xform = 1;
  return knn_launch<MODE_DIRECT_FMA, false, false>(p, (cudaStream_t)stream);
}

extern "C" int l3d_pn2_three_nn(int b, int n, int m, const float* unknown_dev,
                                const float* known_dev, float* dist2_dev, int32_t* idx_dev,
                                void* stream) {
  return l3d_pn2_knn(b, n, m, 3, unknown_dev, known_dev, dist2_dev, idx_dev, stream);
}
