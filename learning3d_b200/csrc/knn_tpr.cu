// Thread-per-row fused pairwise-distance + top-k (sm_100a): knn() on xyz clouds, k <= 24, large batches.
//
// Replaces knn() utils/model_common_utils.py:3-9 (same keys, same (key desc, index asc) order as knn.cu —
// bit-identical results, the test-suite compares the two kernels against each other and against the oracle).
//
// Why a second kernel (DESIGN.md §3.1, "round 2, second half"): knn.cu gives a warp two query rows and spreads
// the candidates over the lanes, so every step of the selection (lane-maximum sort, survivor scan, final sort)
// is a chain of warp shuffles: ~64 SHFL + 65 ISETP + 48 SEL per row, issue slots 53 % busy, and neither fewer
// arithmetic instructions (packed fp32) nor more resident warps moved the clock.  Here a THREAD owns a query
// row and a warp owns 32 consecutive rows of one cloud:
//   * every candidate operand is a shared-memory BROADCAST, two candidates per packed FFMA2 as before;
//   * the selection never leaves the thread's registers — no shuffles, no scans, no per-warp buffers:
//       pass 1: the maxima of 64 candidate groups (one FMNMX3 per candidate pair);
//       threshold: the k-th largest group maximum through an in-register network (2 x merge-exchange sort-32,
//         max-merge, pruned bitonic merge; FMNMX only) — at least k keys reach it and on average 23.5 do
//         (never more than 32 in 99.96 % of uniformly random rows);
//       pass 2: the same packed chain with -thr/2 folded into its first product (threshold lowered by a proven
//         error bound), the sign of the result shifted into a 32-bit survivor mask per 32 candidates, the few set
//         bits appended to a per-row list of 16-bit indices by branch-free steps;
//       final: the <= 32 survivors are re-evaluated with the full key formula (one gathered LDS.128 each),
//         packed into 62-bit (key, ~index) composites that compare as positive doubles (DSETP, reg_sort.cuh) and
//         sorted by a 191-exchange network; every thread stores its k indices with 128-bit stores.
//   * rows whose list exceeds 32 entries sort a second block of 32 and merge (whole warp, rare); a full list
//     (duplicate points, adversarial ties) hands the row to the warp-cooperative knn_row_v2 of knn_common.cuh
//     (itself backed by the exact k-round scan).
// Two kernels: knn_tpr_kernel (a warp = 32 rows over the whole candidate range; clouds with N % 64 != 0) and
// knn_duo_kernel (two warps = 64 rows, each warp one candidate half for all 64 rows, so that every operand load
// feeds two rows — the default; see its header below and profiles/micro/pipes.cu for the measurements behind it).
// The price is parallelism: a row is a thread, so B*N/32 warps exist in total (1024 at C2 = 6.9 per SM) and
// the kernel is one wave; the launcher therefore only takes this path when there are enough rows
// (knn.cu: knn_launch, KNN_TPR_MIN_UNITS), smaller batches stay on the warp-per-row-pair kernel.
// C2 (B=32, N=1024, k=20) on a B200: 33.1 us (knn.cu) -> 25.9 us (profiles/r02/knn_paths_time.txt).
#include "knn_common.cuh"
#include "reg_sort.cuh"
#include "../../include/l3d_b200.h"
#include "launch_count.h"

#include <math.h>

namespace l3d {

constexpr int TPR_G = 64;       // candidate groups per row (threshold = k-th largest group maximum)
constexpr int TPR_CAP = 64;     // survivor-list entries per row (uint16 indices)
__host__ __device__ inline int tpr_slots(int N) { return N <= 1024 ? 2 : 1; }   // clouds resident per CTA round
constexpr int TPR_MIN_N = 128, TPR_MAX_N = 2048, TPR_MAX_K = 24;
constexpr int TPR_THREADS = 256;

// shared memory per resident cloud: pair_xy + pair_zw (8 B per candidate each, npad entries) + float4 (x,y,z,|p|^2)
// padded to whole KNN_TILEs (the warp-cooperative overflow routine of knn_common.cuh reads whole tiles)
__host__ __device__ inline int tpr_npad(int N) { return (N + 127) & ~127; }
__host__ __device__ inline int tpr_ntile(int N) { return ((N + KNN_TILE - 1) / KNN_TILE) * KNN_TILE; }
__host__ __device__ inline size_t tpr_cloud_bytes(int N) { return (size_t)tpr_npad(N) * 16 + (size_t)tpr_ntile(N) * 16; }
// per-row index lists (+ the entry dead stores land on once a list is full) and group maxima, [..][threads]
constexpr size_t TPR_LIST_BYTES = (size_t)(TPR_CAP + 1) * TPR_THREADS * 2;
constexpr size_t TPR_GMAX_BYTES = (size_t)TPR_G * TPR_THREADS * 4;
__host__ __device__ inline size_t tpr_smem_bytes(int N) {
  return tpr_slots(N) * tpr_cloud_bytes(N) + TPR_LIST_BYTES + TPR_GMAX_BYTES + (size_t)(TPR_THREADS / 32) * 64 * 8 + 16;
}

// One query row per thread, a warp owns 32 consecutive rows of one cloud.  The micro-benchmark
// (profiles/micro/pipes.cu) puts a broadcast LDS.128 at 2 SM-cycles per warp instruction whatever the number of
// distinct addresses, so the 2 x 1024 operand loads of a row out-weigh its 2 x 2048 FFMA2 (2 scheduler-cycles each,
// four schedulers) two to one; knn_duo_kernel below halves them.
// PPG: candidate pairs per group when known at compile time (8 <=> N = 1024), 0 = run-time.
// KT:  k when known at compile time (20, DGCNN / DCP), 0 = run-time k <= 24.
template <int PPG, int KT, bool FEAT>
__global__ void __launch_bounds__(TPR_THREADS, 1) knn_tpr_kernel(const KnnParams p) {
  // one row per thread.  The loops over the thread's rows are kept: written as scalar code the kernel compiles to
  // different SASS (one to two more registers), so the row index r below is always 0.
  constexpr int R = 1;
  constexpr int MODE = MODE_EXPANSION_NEG;
  constexpr int THREADS = TPR_THREADS, WARPS = THREADS / 32;
  extern __shared__ __align__(128) unsigned char smem[];
  const int N = p.N, k = KT ? KT : p.k;
  const int npad = tpr_npad(N), ntile = tpr_ntile(N);
  const int ppg = PPG ? PPG : npad / (2 * TPR_G);
  const int nwords = npad / 32;
  const int upc = N / (32 * R);                 // warp units (32 R consecutive rows) per cloud
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  unsigned char* tail = smem + tpr_slots(N) * tpr_cloud_bytes(N);
  unsigned short* list = reinterpret_cast<unsigned short*>(tail) + tid;           // [R][TPR_CAP + 1][THREADS]
  float* gmax = reinterpret_cast<float*>(tail + TPR_LIST_BYTES) + tid;         // [R][TPR_G][THREADS]
  unsigned long long* cbuf = reinterpret_cast<unsigned long long*>(tail + TPR_LIST_BYTES + TPR_GMAX_BYTES) + warp * 64;
  int* wmax = reinterpret_cast<int*>(tail + TPR_LIST_BYTES + TPR_GMAX_BYTES + (size_t)WARPS * 64 * 8);   // [2]
  constexpr int LIST_ROW = (TPR_CAP + 1) * THREADS;     // list entries per row index r
  constexpr int GMAX_ROW = TPR_G * THREADS;

  // programmatic dependent launch, as in knn.cu: the next launch may start filling SMs as our CTAs retire,
  // and nothing touches global memory before the previous launch has completed
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");

  const long units = (long)p.B * upc;
  long u0 = units * blockIdx.x / gridDim.x;
  const long u1 = units * (blockIdx.x + 1) / gridDim.x;

  while (u0 < u1) {
    const int b0 = (int)(u0 / upc);
    const long round_end = min(u1, (long)(b0 + tpr_slots(N)) * upc);
    const int nb = (int)((round_end - 1) / upc) - b0 + 1;

    // ---- stage the clouds of this round: pair layout for the packed loops + float4 for the gathers -----
    if (tid < 2) wmax[tid] = 0;
    __syncthreads();
    for (int i = tid; i < nb * (ntile / 2); i += THREADS) {
      const int s = i / (ntile / 2), pi = i - s * (ntile / 2);
      unsigned char* base = smem + (size_t)s * tpr_cloud_bytes(N);
      ulonglong2* pxy = reinterpret_cast<ulonglong2*>(base);
      ulonglong2* pzw = pxy + npad / 2;
      float4* packed = reinterpret_cast<float4*>(pzw + npad / 2);
      const float* src = p.cand + (size_t)(b0 + s) * 3 * N;
      float4 c0 = knn_padding<MODE>(), c1 = knn_padding<MODE>();
      if (2 * pi < N) {   // N is even: a pair is either real or padding
        const float2 x = *reinterpret_cast<const float2*>(src + 2 * pi);
        const float2 y = *reinterpret_cast<const float2*>(src + N + 2 * pi);
        const float2 z = *reinterpret_cast<const float2*>(src + 2 * (size_t)N + 2 * pi);
        c0 = knn_pack<MODE>(x.x, y.x, z.x);
        c1 = knn_pack<MODE>(x.y, y.y, z.y);
        atomicMax(&wmax[s], __float_as_int(fmaxf(c0.w, c1.w)));      // |c|^2 >= 0: integer order == float order
      }
      packed[2 * pi] = c0;
      packed[2 * pi + 1] = c1;
      if (2 * pi < npad) {
        pxy[pi] = make_ulonglong2(f2_pack(c0.x, c1.x), f2_pack(c0.y, c1.y));
        pzw[pi] = make_ulonglong2(f2_pack(c0.z, c1.z), f2_pack(-c0.w, -c1.w));
      }
    }
    __syncthreads();

    for (long u = u0 + warp; u < round_end; u += WARPS) {
      const int b = (int)(u / upc);
      const int m0 = (int)(u - (long)b * upc) * 32 * R;          // first query point of the unit
      const long row0 = (long)b * N + m0;                        // thread's rows: row0 + r * 32 + lane
      unsigned char* base = smem + (size_t)(b - b0) * tpr_cloud_bytes(N);
      const ulonglong2* pxy = reinterpret_cast<const ulonglong2*>(base);
      const ulonglong2* pzw = pxy + npad / 2;
      const float4* packed = reinterpret_cast<const float4*>(pzw + npad / 2);
      float4 q[R];
#pragma unroll
      for (int r = 0; r < R; ++r) q[r] = packed[m0 + r * 32 + lane];
      unsigned slow_mask = p.force_slow ? (1u << R) - 1u : 0u;    // bit r: row r of this thread takes the exactness net

      if (!p.force_slow) {
        unsigned long long qx2[R], qy2[R], qz2[R];
#pragma unroll
        for (int r = 0; r < R; ++r) { qx2[r] = f2_pack(q[r].x, q[r].x); qy2[r] = f2_pack(q[r].y, q[r].y); qz2[r] = f2_pack(q[r].z, q[r].z); }
        const unsigned long long two2 = f2_pack(2.0f, 2.0f);
        // s (or s - thr when `fused`) of eight candidate pairs for one row, stage by stage: 16 independent fma chains
        auto eval8 = [&](const ulonglong2 (&cx)[8], const ulonglong2 (&cz)[8], unsigned long long (&t)[8],
                         unsigned long long x2, unsigned long long y2, unsigned long long z2, bool fused, unsigned long long h2v) {
#pragma unroll
          for (int i = 0; i < 8; ++i) t[i] = fused ? f2_fma(x2, cx[i].x, h2v) : f2_mul(x2, cx[i].x);
#pragma unroll
          for (int i = 0; i < 8; ++i) t[i] = f2_fma(y2, cx[i].y, t[i]);
#pragma unroll
          for (int i = 0; i < 8; ++i) t[i] = f2_fma(z2, cz[i].x, t[i]);
#pragma unroll
          for (int i = 0; i < 8; ++i) t[i] = f2_fma(two2, t[i], cz[i].y);
        };
        auto load8 = [&](int o, ulonglong2 (&cx)[8], ulonglong2 (&cz)[8]) {      // candidate pairs 8 o .. 8 o + 7
#pragma unroll
          for (int i = 0; i < 8; ++i) { cx[i] = pxy[o * 8 + i]; cz[i] = pzw[o * 8 + i]; }
        };
        auto max16 = [&](const unsigned long long (&t)[8]) -> float {
          float s0, s1, ma = -INFINITY, mb = -INFINITY;
#pragma unroll
          for (int i = 0; i < 8; i += 2) {
            f2_unpack(t[i], s0, s1);     ma = fmaxf(fmaxf(ma, s0), s1);
            f2_unpack(t[i + 1], s0, s1); mb = fmaxf(fmaxf(mb, s0), s1);
          }
          return fmaxf(ma, mb);
        };
        // ---- pass 1: group maxima of s = 2 q.c - |c|^2 (the key without its final "- |q|^2": monotone) ----
        if constexpr (PPG == 8) {
          // N = 1024: a group is eight pairs.  Software-pipelined by hand: the operands of group g + 1 are loaded
          // before group g is evaluated (ptxas does not overlap the trips of this loop by itself)
          ulonglong2 ax[8], az[8], bx[8], bz[8];
          load8(0, ax, az);
#pragma unroll 1
          for (int g = 0; g < TPR_G; g += 2) {
            unsigned long long t[8];
            load8(g + 1, bx, bz);
#pragma unroll
            for (int r = 0; r < R; ++r) {
              eval8(ax, az, t, qx2[r], qy2[r], qz2[r], false, 0ull);
              gmax[r * GMAX_ROW + g * THREADS] = max16(t);
            }
            load8(min(g + 2, TPR_G - 1), ax, az);
#pragma unroll
            for (int r = 0; r < R; ++r) {
              eval8(bx, bz, t, qx2[r], qy2[r], qz2[r], false, 0ull);
              gmax[r * GMAX_ROW + (g + 1) * THREADS] = max16(t);
            }
          }
        } else {
#pragma unroll 1
          for (int g = 0; g < TPR_G; ++g) {
            const ulonglong2* gxy = pxy + g * ppg;
            const ulonglong2* gzw = pzw + g * ppg;
            float mx[R];
#pragma unroll
            for (int r = 0; r < R; ++r) mx[r] = -INFINITY;
#pragma unroll 4
            for (int i = 0; i < ppg; ++i) {
              const ulonglong2 cx = gxy[i], cz = gzw[i];
#pragma unroll
              for (int r = 0; r < R; ++r) {
                const unsigned long long dot = f2_fma(qz2[r], cz.x, f2_fma(qy2[r], cx.y, f2_mul(qx2[r], cx.x)));
                float s0, s1;
                f2_unpack(f2_fma(two2, dot, cz.y), s0, s1);
                mx[r] = fmaxf(fmaxf(mx[r], s0), s1);
              }
            }
#pragma unroll
            for (int r = 0; r < R; ++r) gmax[r * GMAX_ROW + g * THREADS] = mx[r];
          }
        }
        // ---- threshold per row: k-th largest of the 64 group maxima ----------------------------------------
        float thr_r[R];
#pragma unroll 1
        for (int r = 0; r < R; ++r) {
          float t0;
          {
            float ga[32], gb[32];
            const float* gm = gmax + r * GMAX_ROW;
#pragma unroll
            for (int i = 0; i < 32; ++i) { ga[i] = gm[i * THREADS]; gb[i] = gm[(32 + i) * THREADS]; }
            reg_sort_desc<32>(ga, cex_f32);
            reg_sort_desc<32>(gb, cex_f32);
#pragma unroll
            for (int i = 0; i < 32; ++i) ga[i] = fmaxf(ga[i], gb[31 - i]);    // the 32 largest of the 64, bitonic
            reg_merge_desc<32>(ga, cex_f32);
            if (KT) {
              t0 = ga[KT ? KT - 1 : 0];
            } else {
              t0 = ga[0];
#pragma unroll
              for (int i = 1; i < TPR_MAX_K; ++i) t0 = (i == k - 1) ? ga[i] : t0;
            }
          }
          const float qw = q[r].w;
          // s-space threshold (knn.cu row_threshold, DEFER): keeps every s whose key can reach the k-th group
          // maximum's key kb, admits at most the few s within ~2 ulp below it
          const float kb = __fsub_rn(t0, qw);
          float thr = __fadd_rd(__fadd_rd(kb, qw), -__fmul_rn(fmaxf(fabsf(kb), 1e-30f), 1.1920929e-7f));
          // Pass 2 evaluates d = 2 (q.c - thr/2) - |c|^2 in ONE fma chain (the first product becomes an fma with the
          // addend -thr/2), i.e. s - thr with different roundings: |d - (s - thr)| <= 7 eps (|q|^2 + 2 max|c|^2 + |thr|),
          // eps = 2^-24 (three fma roundings of magnitude <= |q||c| + |thr|/2 <= (|q|^2 + |c|^2 + |thr|)/2, doubled, on
          // either side, plus the final roundings).  Lowering thr by 20 eps (|q|^2 + max|c|^2 + |thr|) keeps every
          // candidate with s >= thr on the non-negative side; the handful it admits besides are sorted out exactly below.
          {
            const float wm = __int_as_float(wmax[b - b0]);
            const float delta = __fmul_ru(1.2e-6f, __fadd_ru(__fadd_ru(qw, wm), fabsf(thr)));
            thr = __fadd_rd(thr, -delta);
          }
          thr_r[r] = thr;
        }
        unsigned long long hv[R];     // (-thr/2, -thr/2), added inside the pass-2 fma chain
#pragma unroll
        for (int r = 0; r < R; ++r) {
          hv[r] = f2_pack(-0.5f * thr_r[r], -0.5f * thr_r[r]);
        }

        // ---- pass 2: survivor mask per 32 candidates, set bits appended to the row's index list ----------
        // The list is written through a running shared-memory address: every step stores its candidate index at the
        // next free entry and only a step that really had a set bit advances the address (a dead step's store is
        // overwritten by the next live one), so the steps carry no branches; the address saturates at entry TPR_CAP.
        uint32_t lbase[R], laddr[R];
#pragma unroll
        for (int r = 0; r < R; ++r) { lbase[r] = smem_u32(list + r * LIST_ROW); laddr[r] = lbase[r]; }
        auto take_lowest = [&](uint32_t& mk, uint32_t& la, uint32_t lend, int wbase) {
          const uint32_t low = mk & (0u - mk);
          uint32_t e;
          asm("bfind.u32 %0, %1;" : "=r"(e) : "r"(low));                      // FLO of the isolated bit
          asm volatile("st.shared.u16 [%0], %1;" ::"r"(la), "h"((unsigned short)(wbase + (int)e)) : "memory");
          la = min(la + (low ? (uint32_t)(THREADS * 2) : 0u), lend);
          mk ^= low;
        };
        // sign bits of the sixteen d = s - thr of eight pairs (set = below the threshold): bit 2 i = pair i's first
        auto signs8 = [&](const unsigned long long (&t)[8]) -> uint32_t {
          uint32_t n0 = 0u, n1 = 0u;            // two chains of eight funnel shifts
#pragma unroll
          for (int i = 3; i >= 0; --i) {
            float d0, d1;
            f2_unpack(t[i], d0, d1);
            n0 = __funnelshift_l(__float_as_uint(d1), n0, 1);
            n0 = __funnelshift_l(__float_as_uint(d0), n0, 1);
            f2_unpack(t[4 + i], d0, d1);
            n1 = __funnelshift_l(__float_as_uint(d1), n1, 1);
            n1 = __funnelshift_l(__float_as_uint(d0), n1, 1);
          }
          return n0 + (n1 << 8);
        };
        {
          uint32_t mk_prev[R];     // the mask of word w - 1 is unpacked while word w is evaluated (independent work)
#pragma unroll
          for (int r = 0; r < R; ++r) mk_prev[r] = 0u;
          const int noct = npad / 16;             // octets of candidate pairs; a mask word = two octets
          ulonglong2 ax[8], az[8], bx[8], bz[8];
          load8(0, ax, az);
          load8(1, bx, bz);
#pragma unroll 1
          for (int w = 0; w < nwords; ++w) {
            unsigned long long t[8];
            uint32_t lo16[R], hi16[R];
#pragma unroll
            for (int r = 0; r < R; ++r) {
              eval8(ax, az, t, qx2[r], qy2[r], qz2[r], true, hv[r]);
              lo16[r] = signs8(t);
            }
            load8(min(2 * w + 2, noct - 1), ax, az);
#pragma unroll
            for (int r = 0; r < R; ++r) {
              eval8(bx, bz, t, qx2[r], qy2[r], qz2[r], true, hv[r]);
              hi16[r] = signs8(t);
            }
            load8(min(2 * w + 3, noct - 1), bx, bz);
#pragma unroll
            for (int r = 0; r < R; ++r) {
              const uint32_t lend = lbase[r] + TPR_CAP * THREADS * 2;
              // a word holds 0.7 survivors on average: three branch-free steps, then a rarely entered loop
              take_lowest(mk_prev[r], laddr[r], lend, (w - 1) * 32);
              take_lowest(mk_prev[r], laddr[r], lend, (w - 1) * 32);
              take_lowest(mk_prev[r], laddr[r], lend, (w - 1) * 32);
              while (mk_prev[r]) take_lowest(mk_prev[r], laddr[r], lend, (w - 1) * 32);
              mk_prev[r] = ~(lo16[r] + (hi16[r] << 16));
            }
          }
#pragma unroll
          for (int r = 0; r < R; ++r)
            while (mk_prev[r]) take_lowest(mk_prev[r], laddr[r], lbase[r] + TPR_CAP * THREADS * 2, (nwords - 1) * 32);
        }

        // ---- final, one row at a time: composites of the first 32 survivors, in-register sort, store ------------
#pragma unroll 1
        for (int r = 0; r < R; ++r) {
          const float4 qr = q[r];
          const int cnt = (int)((laddr[r] - lbase[r]) / (THREADS * 2));
          const bool slow = cnt >= TPR_CAP;     // the saturated address means "TPR_CAP or more": exactness net below
          if (slow) slow_mask |= 1u << r;
          const unsigned short* lr = list + r * LIST_ROW;
          const long row = row0 + r * 32 + lane;
          unsigned long long a[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const bool ok = i < cnt;
            const uint32_t j = ok ? (uint32_t)lr[i * THREADS] : 0u;
            const unsigned long long c = tpr_composite(knn_key<MODE>(qr, packed[j]), j);
            a[i] = ok ? c : 0ull;
          }
          reg_sort_desc<32>(a, tpr_cex);
          if (__any_sync(L3D_FULL_MASK, cnt > 32)) {
            // survivors 32..63 of the rows that have them: sort, keep the better 32 of the union, clean up
            unsigned long long bq[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              const bool ok = (32 + i < cnt) && !slow;
              const uint32_t j = ok ? (uint32_t)lr[(32 + i) * THREADS] : 0u;
              const unsigned long long c = tpr_composite(knn_key<MODE>(qr, packed[j]), j);
              bq[i] = ok ? c : 0ull;
            }
            reg_sort_desc<32>(bq, tpr_cex);
#pragma unroll
            for (int i = 0; i < 32; ++i) a[i] = (bq[31 - i] > a[i]) ? bq[31 - i] : a[i];
            reg_merge_desc<32>(a, tpr_cex);
          }
          // the k best (rank order): 128-bit stores when the row is 16-byte aligned
          if (!slow) {
            if (p.idx64 == 1) {
              long long* o = reinterpret_cast<long long*>(p.out_idx) + row * k;
              if ((k & 1) == 0) {
#pragma unroll
                for (int pos = 0; pos < TPR_MAX_K; pos += 2)
                  if (pos < k)
                    *reinterpret_cast<longlong2*>(o + pos) =
                        make_longlong2((long long)tpr_comp_index(a[pos]), (long long)tpr_comp_index(a[pos + 1]));
              } else {
#pragma unroll
                for (int pos = 0; pos < TPR_MAX_K; ++pos)
                  if (pos < k) o[pos] = (long long)tpr_comp_index(a[pos]);
              }
            } else {
#pragma unroll
              for (int pos = 0; pos < TPR_MAX_K; ++pos)
                if (pos < k) knn_store_index(p, row * k + pos, tpr_comp_index(a[pos]));
            }
            if (p.out_val) {
#pragma unroll
              for (int pos = 0; pos < TPR_MAX_K; ++pos)
                if (pos < k) p.out_val[row * k + pos] = knn_val_xform(tpr_comp_key(a[pos]), p.val_xform);
            }
          }
        }
      }

      // ---- exactness net: rows with 64 or more survivors (duplicate points, clouds far from the origin whose keys
      // collapse onto a few fp32 values) are redone by the warp-cooperative routine of knn.cu (lane-maximum
      // threshold, shuffle networks; itself backed by the exact k-round scan); the testing hook goes there too ----
#pragma unroll 1
      for (int r = 0; r < R; ++r) {
        unsigned todo = __ballot_sync(L3D_FULL_MASK, (slow_mask >> r) & 1u);
        const float4 qr = q[r];
        while (todo) {
          const int from = __ffs(todo) - 1;
          todo &= todo - 1;
          float4 qs;
          qs.x = __shfl_sync(L3D_FULL_MASK, qr.x, from); qs.y = __shfl_sync(L3D_FULL_MASK, qr.y, from);
          qs.z = __shfl_sync(L3D_FULL_MASK, qr.z, from); qs.w = __shfl_sync(L3D_FULL_MASK, qr.w, from);
          knn_row_v2<MODE>(p, packed, cbuf, qs, row0 + r * 32 + from, ntile / KNN_TILE, lane);
          __syncwarp();
        }
      }

      if (FEAT) {
        // get_graph_feature() fused (model_common_utils.py:132-155): cat(x[nbr], x[centre]) for the 32 R rows of this
        // warp; their 32 R k (index, position) entries are one contiguous run per channel -> coalesced stores
        __syncwarp();
        const long e0 = row0 * k;                                  // first entry of the warp's rows
        const size_t cs = (size_t)N * k;
        float* f = p.feat_out + (size_t)b * 6 * cs + (size_t)m0 * k;
        for (int e = lane; e < 32 * R * k; e += 32) {
          const int j = (int)reinterpret_cast<const volatile long long*>(p.out_idx)[e0 + e];
          const float4 c = packed[j];
          const float4 ctr = packed[m0 + e / k];
          f[e] = c.x; f[cs + e] = c.y; f[2 * cs + e] = c.z;
          f[3 * cs + e] = ctr.x; f[4 * cs + e] = ctr.y; f[5 * cs + e] = ctr.z;
        }
      }
    }
    u0 = round_end;
    __syncthreads();   // every warp is done with the resident clouds before the next round overwrites them
  }
}

// ---- "duo" kernel: two warps share 64 rows ---------------------------------------------------------------------
// The same selection as knn_tpr_kernel, re-cut after the pipe micro-benchmarks (profiles/micro/pipes.cu): with one
// row per thread the operand loads of the two passes (2 x 1024 broadcast LDS.128 per warp, 2 SM-cycles each) bound the
// kernel; two rows per thread halve them but leave one warp per scheduler, which cannot keep the pipes busy alone.
// Here a DUO of warps owns 64 consecutive rows: in the two candidate passes warp h evaluates candidate HALF h for all
// 64 rows (two rows per thread: every operand load feeds two rows), in the threshold and final phases thread (h, lane)
// owns row 32 h + lane.  The halves meet in shared memory (group maxima, thresholds, two index sub-lists per row),
// the phases are separated by a 64-thread named barrier.  Rows per SM, warps per SM and fma work are unchanged;
// shared-memory operand traffic halves.
constexpr int DUO_THREADS = 256, DUO_PER_CTA = DUO_THREADS / 64;
constexpr int DUO_LCAP = 32;                 // entries per (row, candidate half) sub-list that count as "not full"
constexpr int DUO_LROWS = DUO_LCAP + 4;      // + the entries the three unclamped steps of a word may touch
constexpr size_t DUO_GMAX_BYTES = (size_t)TPR_G * 64 * 4;
constexpr size_t DUO_LIST_BYTES = (size_t)2 * DUO_LROWS * 64 * 2;
constexpr size_t DUO_BYTES = DUO_GMAX_BYTES + DUO_LIST_BYTES + 64 * 4 + 2 * 64 * 4;     // + thr[64] + cnt[2][64]
__host__ __device__ inline size_t duo_smem_bytes(int N) {
  return tpr_slots(N) * tpr_cloud_bytes(N) + DUO_PER_CTA * DUO_BYTES + (size_t)(DUO_THREADS / 32) * 64 * 8 + 16;
}
__device__ __forceinline__ void duo_sync(int duo) { asm volatile("bar.sync %0, 64;" ::"r"(1 + duo) : "memory"); }

template <int PPG, int KT, bool FEAT>
__global__ void __launch_bounds__(DUO_THREADS, 1) knn_duo_kernel(const KnnParams p) {
  constexpr int MODE = MODE_EXPANSION_NEG;
  constexpr int THREADS = DUO_THREADS;
  extern __shared__ __align__(128) unsigned char smem[];
  const int N = p.N, k = KT ? KT : p.k;
  const int npad = tpr_npad(N), ntile = tpr_ntile(N);
  const int ppg = PPG ? PPG : npad / (2 * TPR_G);
  const int nwords = npad / 32;
  const int upc = N / 64;                       // duo units (64 consecutive rows) per cloud
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, duo = warp >> 1, h = warp & 1;

  unsigned char* tail = smem + tpr_slots(N) * tpr_cloud_bytes(N);
  unsigned char* dbase = tail + (size_t)duo * DUO_BYTES;
  float* gmax_d = reinterpret_cast<float*>(dbase);                                           // [TPR_G][64]
  unsigned short* list_d = reinterpret_cast<unsigned short*>(dbase + DUO_GMAX_BYTES);         // [2][DUO_LROWS][64]
  float* thr_d = reinterpret_cast<float*>(dbase + DUO_GMAX_BYTES + DUO_LIST_BYTES);           // [64]
  int* cnt_d = reinterpret_cast<int*>(thr_d + 64);                                            // [2][64]
  unsigned long long* cbuf = reinterpret_cast<unsigned long long*>(tail + DUO_PER_CTA * DUO_BYTES) + warp * 64;
  int* wmax = reinterpret_cast<int*>(tail + DUO_PER_CTA * DUO_BYTES + (size_t)(THREADS / 32) * 64 * 8);

  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");

  const long units = (long)p.B * upc;
  long u0 = units * blockIdx.x / gridDim.x;
  const long u1 = units * (blockIdx.x + 1) / gridDim.x;

  while (u0 < u1) {
    const int b0 = (int)(u0 / upc);
    const long round_end = min(u1, (long)(b0 + tpr_slots(N)) * upc);
    const int nb = (int)((round_end - 1) / upc) - b0 + 1;

    // ---- stage the clouds of this round: pair layout for the packed loops + float4 for the gathers --------------
    // Four candidate pairs per thread and trip, all twelve global loads issued before the first use (indices
    // clamped instead of predicated): the loop used to pay one L2 round trip per trip (~3 of the 26.6 us per launch).
    if (tid < 2) wmax[tid] = 0;
    __syncthreads();
    {
      const int half = ntile / 2;                     // candidate pairs per resident cloud, tile padding included
      const int total = nb * half;                    // nb <= 2
      for (int i0 = tid; i0 < total; i0 += 4 * THREADS) {
        float2 X[4], Y[4], Z[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int i = min(i0 + u * THREADS, total - 1);
          const int sc = (i >= half) ? 1 : 0, pi = min(i - sc * half, N / 2 - 1);
          const float* src = p.cand + (size_t)(b0 + sc) * 3 * N;
          X[u] = *reinterpret_cast<const float2*>(src + 2 * pi);
          Y[u] = *reinterpret_cast<const float2*>(src + N + 2 * pi);
          Z[u] = *reinterpret_cast<const float2*>(src + 2 * (size_t)N + 2 * pi);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int i = i0 + u * THREADS;
          if (i < total) {
            const int sc = (i >= half) ? 1 : 0, pi = i - sc * half;
            unsigned char* base = smem + (size_t)sc * tpr_cloud_bytes(N);
            ulonglong2* pxy = reinterpret_cast<ulonglong2*>(base);
            ulonglong2* pzw = pxy + npad / 2;
            float4* packed = reinterpret_cast<float4*>(pzw + npad / 2);
            float4 c0 = knn_padding<MODE>(), c1 = knn_padding<MODE>();
            if (2 * pi < N) {   // N is even: a pair is either real or padding
              c0 = knn_pack<MODE>(X[u].x, Y[u].x, Z[u].x);
              c1 = knn_pack<MODE>(X[u].y, Y[u].y, Z[u].y);
              atomicMax(&wmax[sc], __float_as_int(fmaxf(c0.w, c1.w)));      // |c|^2 >= 0: integer order == float order
            }
            packed[2 * pi] = c0;
            packed[2 * pi + 1] = c1;
            if (2 * pi < npad) {
              pxy[pi] = make_ulonglong2(f2_pack(c0.x, c1.x), f2_pack(c0.y, c1.y));
              pzw[pi] = make_ulonglong2(f2_pack(c0.z, c1.z), f2_pack(-c0.w, -c1.w));
            }
          }
        }
      }
    }
    __syncthreads();

    for (long u = u0 + duo; u < round_end; u += DUO_PER_CTA) {
      const int b = (int)(u / upc);
      const int m0 = (int)(u - (long)b * upc) * 64;              // first query point of the duo's 64 rows
      const long row0 = (long)b * N + m0;
      unsigned char* base = smem + (size_t)(b - b0) * tpr_cloud_bytes(N);
      const ulonglong2* pxy = reinterpret_cast<const ulonglong2*>(base);
      const ulonglong2* pzw = pxy + npad / 2;
      const float4* packed = reinterpret_cast<const float4*>(pzw + npad / 2);
      float4 q[2];
      q[0] = packed[m0 + lane];
      q[1] = packed[m0 + 32 + lane];
      const int rho = 32 * h + lane;                             // the row this thread owns outside the passes
      const float4 qo = h ? q[1] : q[0];
      const long row = row0 + rho;
      bool slow = (p.force_slow != 0);

      if (!p.force_slow) {
        unsigned long long qx2[2], qy2[2], qz2[2];
#pragma unroll
        for (int r = 0; r < 2; ++r) { qx2[r] = f2_pack(q[r].x, q[r].x); qy2[r] = f2_pack(q[r].y, q[r].y); qz2[r] = f2_pack(q[r].z, q[r].z); }
        const unsigned long long two2 = f2_pack(2.0f, 2.0f);
        // ---- pass 1: maxima of this warp's 32 candidate groups, two rows per thread --------------------------
#pragma unroll 1   // one group per trip (2 per trip: profiles/r02/knn_tpr_variants.txt)
        for (int gi = 0; gi < TPR_G / 2; ++gi) {
          const int g = h * (TPR_G / 2) + gi;
          const ulonglong2* gxy = pxy + g * ppg;
          const ulonglong2* gzw = pzw + g * ppg;
          float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll 8
          for (int i = 0; i < ppg; ++i) {
            const ulonglong2 cx = gxy[i], cz = gzw[i];
#pragma unroll
            for (int r = 0; r < 2; ++r) {
              const unsigned long long dot = f2_fma(qz2[r], cz.x, f2_fma(qy2[r], cx.y, f2_mul(qx2[r], cx.x)));
              float s0, s1;
              f2_unpack(f2_fma(two2, dot, cz.y), s0, s1);
              mx[r] = fmaxf(fmaxf(mx[r], s0), s1);
            }
          }
          gmax_d[g * 64 + lane] = mx[0];
          gmax_d[g * 64 + 32 + lane] = mx[1];
        }
        duo_sync(duo);
        // ---- threshold of row rho: k-th largest of its 64 group maxima ------------------------------------------
        {
          float t0;
          float ga[32], gb[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) { ga[i] = gmax_d[i * 64 + rho]; gb[i] = gmax_d[(32 + i) * 64 + rho]; }
          reg_sort_desc<32>(ga, cex_f32);
          reg_sort_desc<32>(gb, cex_f32);
#pragma unroll
          for (int i = 0; i < 32; ++i) ga[i] = fmaxf(ga[i], gb[31 - i]);
          reg_merge_desc<32>(ga, cex_f32);
          if (KT) {
            t0 = ga[KT ? KT - 1 : 0];
          } else {
            t0 = ga[0];
#pragma unroll
            for (int i = 1; i < TPR_MAX_K; ++i) t0 = (i == k - 1) ? ga[i] : t0;
          }
          // s-space threshold with the DEFER margin and the fused-evaluation margin (see knn_tpr_kernel)
          const float kb = __fsub_rn(t0, qo.w);
          float thr = __fadd_rd(__fadd_rd(kb, qo.w), -__fmul_rn(fmaxf(fabsf(kb), 1e-30f), 1.1920929e-7f));
          const float wm = __int_as_float(wmax[b - b0]);
          const float delta = __fmul_ru(1.2e-6f, __fadd_ru(__fadd_ru(qo.w, wm), fabsf(thr)));
          thr_d[rho] = __fadd_rd(thr, -delta);
        }
        duo_sync(duo);
        // ---- pass 2: this warp's candidate half again, d = s - thr inside the fma chain, sign masks, index lists --
        {
          unsigned long long hv[2];
#pragma unroll
          for (int r = 0; r < 2; ++r) { const float t = thr_d[r * 32 + lane]; hv[r] = f2_pack(-0.5f * t, -0.5f * t); }
          uint32_t lbase[2], laddr[2], mk_prev[2];
#pragma unroll
          for (int r = 0; r < 2; ++r) {
            lbase[r] = smem_u32(list_d + (h * DUO_LROWS) * 64 + r * 32 + lane);
            laddr[r] = lbase[r];
            mk_prev[r] = 0u;
          }
          auto take_lowest = [&](uint32_t& mk, uint32_t& la, int wbase) {
            const uint32_t low = mk & (0u - mk);
            uint32_t e;
            asm("bfind.u32 %0, %1;" : "=r"(e) : "r"(low));
            asm volatile("st.shared.u16 [%0], %1;" ::"r"(la), "h"((unsigned short)(wbase + (int)e)) : "memory");
            la += low ? 128u : 0u;       // a dead step's store is overwritten by the next live one
            mk ^= low;
          };
          const int w_begin = h * (nwords / 2), w_end = w_begin + nwords / 2;
#pragma unroll 1   // one mask word per trip (2 per trip: profiles/r02/knn_tpr_variants.txt)
          for (int w = w_begin; w < w_end; ++w) {
            uint32_t m16[2][2];
#pragma unroll
            for (int o = 0; o < 2; ++o) {
              ulonglong2 cx[8], cz[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) { cx[i] = pxy[(2 * w + o) * 8 + i]; cz[i] = pzw[(2 * w + o) * 8 + i]; }
#pragma unroll
              for (int r = 0; r < 2; ++r) {
                unsigned long long t[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) t[i] = f2_fma(qx2[r], cx[i].x, hv[r]);
#pragma unroll
                for (int i = 0; i < 8; ++i) t[i] = f2_fma(qy2[r], cx[i].y, t[i]);
#pragma unroll
                for (int i = 0; i < 8; ++i) t[i] = f2_fma(qz2[r], cz[i].x, t[i]);
#pragma unroll
                for (int i = 0; i < 8; ++i) t[i] = f2_fma(two2, t[i], cz[i].y);
                uint32_t n0 = 0u, n1 = 0u;
#pragma unroll
                for (int i = 3; i >= 0; --i) {
                  float d0, d1;
                  f2_unpack(t[i], d0, d1);
                  n0 = __funnelshift_l(__float_as_uint(d1), n0, 1);
                  n0 = __funnelshift_l(__float_as_uint(d0), n0, 1);
                  f2_unpack(t[4 + i], d0, d1);
                  n1 = __funnelshift_l(__float_as_uint(d1), n1, 1);
                  n1 = __funnelshift_l(__float_as_uint(d0), n1, 1);
                }
                m16[r][o] = n0 + (n1 << 8);
              }
            }
#pragma unroll
            for (int r = 0; r < 2; ++r) {
              const uint32_t lend = lbase[r] + DUO_LCAP * 128;
              take_lowest(mk_prev[r], laddr[r], (w - 1) * 32);
              take_lowest(mk_prev[r], laddr[r], (w - 1) * 32);
              take_lowest(mk_prev[r], laddr[r], (w - 1) * 32);
              while (mk_prev[r]) { take_lowest(mk_prev[r], laddr[r], (w - 1) * 32); laddr[r] = min(laddr[r], lend); }
              laddr[r] = min(laddr[r], lend);
              mk_prev[r] = ~(m16[r][0] + (m16[r][1] << 16));
            }
          }
#pragma unroll
          for (int r = 0; r < 2; ++r) {
            const uint32_t lend = lbase[r] + DUO_LCAP * 128;
            while (mk_prev[r]) { take_lowest(mk_prev[r], laddr[r], (w_end - 1) * 32); laddr[r] = min(laddr[r], lend); }
            cnt_d[h * 64 + r * 32 + lane] = (int)((laddr[r] - lbase[r]) / 128u);
          }
        }
        duo_sync(duo);
        // ---- final for row rho: the two sub-lists back to back, composites, in-register sort, store -------------
        {
          const int c0 = cnt_d[rho], c1 = cnt_d[64 + rho];
          const int cnt = c0 + c1;
          slow = (c0 >= DUO_LCAP) || (c1 >= DUO_LCAP);       // a saturated sub-list: exactness net below
          const unsigned short* lr = list_d + rho;
          auto entry = [&](int i) -> uint32_t {               // i-th survivor of the row (i < cnt)
            const int e = (i < c0) ? i : (DUO_LROWS + i - c0);
            return (uint32_t)lr[e * 64];
          };
          unsigned long long a[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const bool ok = i < cnt;
            const uint32_t j = ok ? entry(i) : 0u;
            const unsigned long long c = tpr_composite(knn_key<MODE>(qo, packed[j]), j);
            a[i] = ok ? c : 0ull;
          }
          reg_sort_desc<32>(a, tpr_cex);
          if (__any_sync(L3D_FULL_MASK, cnt > 32)) {
            unsigned long long bq[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              const bool ok = (32 + i < cnt) && !slow;
              const uint32_t j = ok ? entry(32 + i) : 0u;
              const unsigned long long c = tpr_composite(knn_key<MODE>(qo, packed[j]), j);
              bq[i] = ok ? c : 0ull;
            }
            reg_sort_desc<32>(bq, tpr_cex);
#pragma unroll
            for (int i = 0; i < 32; ++i) a[i] = (bq[31 - i] > a[i]) ? bq[31 - i] : a[i];
            reg_merge_desc<32>(a, tpr_cex);
          }
          // ---- output: the warp's 32 rows are one contiguous block of 32 k indices.  Every thread drops its k
          // indices as uint16 into a shared-memory image of that block (the duo's group-maximum array is free by
          // now), then the warp writes the block with fully coalesced 128-bit stores; a row bound for the exactness
          // net leaves garbage there, which that routine overwrites afterwards (same warp, program order).
          unsigned short* ob = reinterpret_cast<unsigned short*>(gmax_d) + h * 1024;
          if (!slow) {
#pragma unroll
            for (int pos = 0; pos < TPR_MAX_K; ++pos)
              if (pos < k) ob[lane * k + pos] = (unsigned short)tpr_comp_index(a[pos]);
          }
          __syncwarp();
          const long blk = (row0 + 32 * h) * k;                      // first entry of the warp's block
          if (p.idx64 == 1) {
            long long* o = reinterpret_cast<long long*>(p.out_idx) + blk;
            for (int e2 = lane; e2 < 16 * k; e2 += 32) {             // pairs of indices
              const uint32_t w2 = *reinterpret_cast<const uint32_t*>(ob + 2 * e2);
              *reinterpret_cast<longlong2*>(o + 2 * e2) = make_longlong2((long long)(w2 & 0xffffu), (long long)(w2 >> 16));
            }
          } else if (p.idx64 == 2 && ((reinterpret_cast<uintptr_t>(p.out_idx) + (size_t)blk * 2) & 15u) == 0) {
            uint4* o = reinterpret_cast<uint4*>(reinterpret_cast<unsigned short*>(p.out_idx) + blk);
            for (int e8 = lane; e8 < 4 * k; e8 += 32) o[e8] = *reinterpret_cast<const uint4*>(ob + 8 * e8);
          } else if (!slow) {
#pragma unroll
            for (int pos = 0; pos < TPR_MAX_K; ++pos)
              if (pos < k) knn_store_index(p, row * k + pos, tpr_comp_index(a[pos]));
          }
          if (p.out_val && !slow) {
#pragma unroll
            for (int pos = 0; pos < TPR_MAX_K; ++pos)
              if (pos < k) p.out_val[row * k + pos] = knn_val_xform(tpr_comp_key(a[pos]), p.val_xform);
          }
        }
      }

      // ---- exactness net (see knn_tpr_kernel): this warp's 32 rows ------------------------------------------------
      unsigned todo = __ballot_sync(L3D_FULL_MASK, slow);
      while (todo) {
        const int from = __ffs(todo) - 1;
        todo &= todo - 1;
        float4 qs;
        qs.x = __shfl_sync(L3D_FULL_MASK, qo.x, from); qs.y = __shfl_sync(L3D_FULL_MASK, qo.y, from);
        qs.z = __shfl_sync(L3D_FULL_MASK, qo.z, from); qs.w = __shfl_sync(L3D_FULL_MASK, qo.w, from);
        knn_row_v2<MODE>(p, packed, cbuf, qs, row0 + 32 * h + from, ntile / KNN_TILE, lane);
        __syncwarp();
      }

      if (FEAT) {
        // get_graph_feature() fused: cat(x[nbr], x[centre]) for this warp's 32 rows, coalesced per channel.  The
        // indices come from the shared-memory image of the output block; a warp with a row that went through the
        // exactness net (or the testing hook) re-reads what was stored.
        __syncwarp();
        const long e0 = (row0 + 32 * h) * k;
        const size_t cs = (size_t)N * k;
        const int n0 = m0 + 32 * h;
        float* f = p.feat_out + (size_t)b * 6 * cs + (size_t)n0 * k;
        const bool from_smem = !__any_sync(L3D_FULL_MASK, slow);
        const unsigned short* ob = reinterpret_cast<const unsigned short*>(gmax_d) + h * 1024;
        for (int e = lane; e < 32 * k; e += 32) {
          const int j = from_smem ? (int)ob[e] : (int)reinterpret_cast<const volatile long long*>(p.out_idx)[e0 + e];
          const float4 c = packed[j];
          const float4 ctr = packed[n0 + e / k];
          f[e] = c.x; f[cs + e] = c.y; f[2 * cs + e] = c.z;
          f[3 * cs + e] = ctr.x; f[4 * cs + e] = ctr.y; f[5 * cs + e] = ctr.z;
        }
      }
      duo_sync(duo);    // the duo's shared arrays are reused by its next unit
    }
    u0 = round_end;
    __syncthreads();
  }
}

static thread_local int g_knn_path = 0;   // 0 auto, 1 warp-per-row-pair kernel only, 2 thread-per-row whenever eligible
int knn_path_flag() { return g_knn_path; }

// shapes the thread-per-row kernel takes at all (the launcher in knn.cu adds the "enough rows" rule)
bool knn_tpr_eligible(const KnnParams& p) {
  if (p.N % 32 != 0 || p.N < TPR_MIN_N || p.N > TPR_MAX_N || p.k > TPR_MAX_K || p.k < 1) return false;
  if (p.M != p.N || p.query != nullptr) return false;
  if ((reinterpret_cast<uintptr_t>(p.cand) & 7u) != 0) return false;       // float2 staging loads
  if (p.idx64 == 1 && (reinterpret_cast<uintptr_t>(p.out_idx) & 15u) != 0) return false;
  if (p.feat_out && p.idx64 != 1) return false;
  return tpr_smem_bytes(p.N) <= KNN_SMEM_LIMIT;
}

// One CTA per SM, every CTA resident at once; a unit is `unit_rows` consecutive rows of one cloud.
template <auto Kern>
static int tpr_launch_t(const KnnParams& p, cudaStream_t stream, int threads, int unit_rows, size_t smem) {
  int dev = 0;
  cudaGetDevice(&dev);
  const cudaError_t e = raise_smem_once<Kern>(dev, KNN_SMEM_LIMIT);
  if (e != cudaSuccess) return (int)e;
  const long units = (long)p.B * (p.N / unit_rows);
  long grid = sm_count(dev);
  if (grid > units) grid = units;
  return knn_launch_pdl(Kern, grid, threads, smem, stream, p);
}

int knn_tpr_launch(const KnnParams& p, cudaStream_t stream) {
  const bool n1024 = tpr_npad(p.N) == 1024;
  if (p.N % 64 == 0 && duo_smem_bytes(p.N) <= KNN_SMEM_LIMIT) {
    const size_t smem = duo_smem_bytes(p.N);
    if (p.feat_out) {
      if (n1024 && p.k == 20) return tpr_launch_t<knn_duo_kernel<8, 20, true>>(p, stream, DUO_THREADS, 64, smem);
      return tpr_launch_t<knn_duo_kernel<0, 0, true>>(p, stream, DUO_THREADS, 64, smem);
    }
    if (n1024 && p.k == 20) return tpr_launch_t<knn_duo_kernel<8, 20, false>>(p, stream, DUO_THREADS, 64, smem);
    return tpr_launch_t<knn_duo_kernel<0, 0, false>>(p, stream, DUO_THREADS, 64, smem);
  }
  const size_t smem = tpr_smem_bytes(p.N);
  if (p.feat_out) {
    if (n1024 && p.k == 20) return tpr_launch_t<knn_tpr_kernel<8, 20, true>>(p, stream, TPR_THREADS, 32, smem);
    return tpr_launch_t<knn_tpr_kernel<0, 0, true>>(p, stream, TPR_THREADS, 32, smem);
  }
  if (n1024 && p.k == 20) return tpr_launch_t<knn_tpr_kernel<8, 20, false>>(p, stream, TPR_THREADS, 32, smem);
  return tpr_launch_t<knn_tpr_kernel<0, 0, false>>(p, stream, TPR_THREADS, 32, smem);
}

}  // namespace l3d

extern "C" void l3d_debug_knn_path(int path) { l3d::g_knn_path = (path == 1 || path == 2) ? path : 0; }
