// Soft correspondences of DCP's SVD head, fused (sm_100a: TMA + tcgen05 + TMEM).
//
// Replaces utils/svd.py:23-28:
//     scores   = softmax(src_emb^T . tgt_emb / sqrt(d_k), dim=2)      [B, Ns, Nt]   (134 MB at C3)
//     src_corr = tgt . scores^T                                        [B, 3, Ns]
// without ever writing the score matrix: one CTA owns 128 source points, walks the target points
// in tiles of 256 (TMA pipeline) / 128 (generic), and keeps a running (max, sum, sum*xyz) per source
// point — the flash-attention recurrence with a 3-wide V.
//
// Arithmetic: the score GEMM runs on the 5th-gen tensor cores as 3xTF32 — every fp32 operand x is
// split into hi + lo,  a.b ~= hi.hi + hi.lo + lo.hi  accumulated in fp32 in TMEM: relative error
// ~2^-21 per product, the same class as the fp32 SGEMM the reference calls (torch.matmul with TF32
// off).  exp() is ex2.approx on log2(e)-prescaled scores.
//
// Two operand pipelines, one epilogue / MMA structure:
//   TMA path (Ns, Nt multiples of 4, 16-byte aligned bases — every shape the models produce):
//     the embeddings are [d, n]-major in HBM, which IS an MN-major UMMA operand: 3-D tensor-map TMA
//     drops [16 d x 32 n] boxes (SWIZZLE_128B_ATOM_32B = UMMA layout 1, the only swizzle MN-major tf32
//     operands exist in) straight into shared memory and the tensor core reads them as the hi operand
//     (the hardware ignores the low 13 mantissa bits); four "splitter" warps only derive the lo tiles
//     (x - trunc(x), tf32-rounded) shared-to-shared.  No thread touches global memory for the GEMM
//     operands.  N = 256 MMAs: the kernel is shared-memory-bandwidth bound (DESIGN.md §3.6).
//   generic path (any shape): four producer warps load rows with LDG, split, and store K-major
//     swizzled tiles themselves.
//   warps 0-3  epilogue: tcgen05.ld the 128 x BN score tile (lane = source point), online softmax,
//              xyz accumulation; two accumulators in TMEM so it overlaps the next tile's MMAs
//   warps 4-7  splitters / producers
//   warp  8    one thread issues tcgen05.mma (M128 N256|128 K8, kind::tf32) and tcgen05.commit
//   warp  9    one thread issues the TMA loads (TMA path)
// Every mbarrier wait is bounded: a protocol bug surfaces as an error code, never as a hung GPU.
#include "common.cuh"
#include "tc05.cuh"
#include "../../include/l3d_b200.h"
#include "knn_matrix.h"
#include "launch_count.h"

#include <cuda.h>
#include <string.h>
#include <math.h>

namespace l3d {

constexpr int SC_EPI_THREADS = 128;
constexpr int SC_PROD_THREADS = 128;
constexpr int SC_THREADS = SC_EPI_THREADS + SC_PROD_THREADS + 64;   // + MMA warp + TMA warp
constexpr int SC_MAX_BN = 256, SC_MAX_STAGES = 6;

// Tile configuration per operand pipeline.  The kernel is shared-memory-bandwidth bound (TMA writes,
// the splitters' read + write and the tensor core's operand reads all cross the same 128 B/clk port), so
// the TMA path uses N = 256 MMAs: A is read once per 256 target points instead of once per 128.
// CTAS = 2: a CTA pair (cluster of 2, tcgen05 cta_group::2) computes a 256 x 256 tile per MMA; each CTA keeps
// its own 128 source rows and only HALF of the target columns, so the B-side TMA, split and operand-read
// traffic per SM halves (144 KB -> 96 KB of shared-memory traffic per 16-channel stage).
template <bool USE_TMA, int CTAS = 1>
struct SoftCorrCfg {
  static constexpr int BN = USE_TMA ? 256 : 128;      // target points per tile (UMMA N)
  static constexpr int BK = USE_TMA ? 16 : 32;        // embedding channels per stage
  static constexpr int STAGES = USE_TMA ? (CTAS == 2 ? 6 : 4) : 3;
  static constexpr int BN_LOCAL = BN / CTAS;          // target columns whose operands live in this CTA
  static constexpr int A_TILE = SC_BM * BK * 4;       // bytes: 8 KB / 16 KB
  static constexpr int B_TILE = BN_LOCAL * BK * 4;    // bytes: 16 KB (8 KB in a pair)
  static constexpr int STAGE = 2 * A_TILE + 2 * B_TILE;   // A_hi, A_lo, B_hi, B_lo: 48 / 32 / 64 KB
  static constexpr int TMEM_COLS = 2 * BN;            // two fp32 accumulators
  static constexpr int ATOM = 32 * BK * 4;            // TMA path: bytes of one [BK d x 32 n] box
};

struct SoftCorrParams {
  const float* src_emb;   // [B, D, Ns]
  const float* tgt_emb;   // [B, D, Nt]
  const float* tgt_xyz;   // [B, 3, Nt]
  float* out;             // [B, 3, Ns]
  float* dbg_scores;      // optional [B, Ns, Nt]: raw accumulator dump (debug entry point only)
  // EPI_KEYS (feature-space kNN): squared norms of the source / target columns and the key matrix
  const float* xx_a;      // [B, Ns]
  const float* xx_b;      // [B, Nt]
  float* keys;            // [B, Ns, Nt]   ((-|b_j|^2) + 2 a_i.b_j) - |a_i|^2
  // EPI_SQDIST (feature-space square_distance / RPMNet affinity): optional per-item affinity transform
  const float* aff_beta;  // [B] or null: out = -beta[b] * (dist - alpha[b])     (rpmnet.py:266-272)
  const float* aff_alpha; // [B]
  // EPI_STATS / EPI_PROBS_T (attention, utils/transformer.py:17-23): row statistics of softmax(a^T b / sqrt(D)) and
  // the TRANSPOSED probabilities P^T [B, Nt, Ns] (the B operand of the P.V GEMM, l3d_conv1x1_bn_relu_maxk)
  float* stats;           // [B, Ns, 2]: (running max in log2 units, sum of 2^(s - max))
  float* probs_t;         // [B, Nt, Ns]
  int single_pass;        // EPI_STATS: one TF32 MMA per k-step (hi.hi only): the row max to ~1e-3 relative is all the
                          // probability pass needs as its exponent reference
  int probs_unnormalized; // EPI_PROBS_T: write 2^(s c - m_i) WITHOUT the 1/l_i factor and store the exact row sums
                          // l_i = sum_j 2^(s c - m_i) into stats[.., 1] (the p.v GEMM divides its columns by them)
  // EPI_DS (backward of the soft correspondences): dS[i,j] = P[i,j] (g_i . tgt_j - g_i . corr_i) / sqrt(D)
  const float* grad_corr; // [B, 3, Ns]  dL/d src_corr
  const float* corr;      // [B, 3, Ns]  src_corr of the forward
  float* ds;              // optional [B, Ns, Nt]
  float* ds_t;            // optional [B, Nt, Ns]
  const int* cond_flag;   // EPI_STATS: when set and *cond_flag == 0 the launch returns at once (l3d_attention_stats_if)
  int tma4;               // TMA pipeline: the tensor maps are the chunked 4-D views (one instruction per operand tile)
  int kmajor;             // generic pipeline only: operands are [B, N, D] (channels contiguous) instead of [B, D, N]
  int* err;               // device error word (0 = ok)
  float* part;            // split target range only: partial softmax states [B, Ns, gridDim.z, 8]
  int tiles_per_split;    // target tiles handled by one CTA (all of them when gridDim.z == 1)
  int B, D, Ns, Nt;
  float c;                // log2(e) / sqrt(D)
};

struct SoftCorrShared {
  float4 xyz[2][SC_MAX_BN];
  uint64_t tma_full[SC_MAX_STAGES];   // TMA path: raw tiles landed
  uint64_t full[SC_MAX_STAGES];       // all four operand tiles of the stage are ready for the MMA
  uint64_t empty[SC_MAX_STAGES];      // the MMAs reading the stage have completed
  uint64_t acc_full[2];
  uint64_t acc_empty[2];
  uint32_t tmem_base;
  // EPI_KEYS: per-warp 32 x 32 transpose tile (row stride 36 floats: conflict-free 16-byte accesses both
  // ways) so that the key matrix is written as full 128-byte lines instead of 16-byte pieces of 32 rows
  alignas(16) float tbuf[SC_EPI_THREADS / 32][32][36];
};

__device__ int g_softcorr_error = 0;
__device__ float g_softcorr_dbg_tiles[SoftCorrCfg<true>::STAGE / 4];   // stage-0 operand tiles of CTA (0,0), debug entry only

constexpr int SC_GBK = SoftCorrCfg<false>::BK;   // generic pipeline: channels per stage (one 128 B swizzle row)

// byte offset of (row r, 16-byte chunk c) inside a K-major [128 x 32 fp32] swizzled tile
__device__ __forceinline__ uint32_t sc_swz(int r, int c) {
  return (uint32_t)(((r >> 3) << 10) | ((r & 7) << 7) | ((c ^ (r & 7)) << 4));
}

// ---- generic producer helpers -------------------------------------------------------------------
__device__ __forceinline__ void sc_load_row(const float* __restrict__ base, int D, int N, int d0,
                                            int n, float (&v)[SC_GBK], int kmajor = 0) {
  const bool nv = n < N;
  if (kmajor) {
    // [N, D] operand: the 32 channels of this row are contiguous (one 128-byte line per thread)
    const float* p = base + (size_t)(nv ? n : 0) * D + d0;
    if (nv && d0 + SC_GBK <= D && (D & 3) == 0) {
#pragma unroll
      for (int q = 0; q < SC_GBK / 4; ++q) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(p) + q);
        v[q * 4] = t.x; v[q * 4 + 1] = t.y; v[q * 4 + 2] = t.z; v[q * 4 + 3] = t.w;
      }
    } else {
#pragma unroll
      for (int dd = 0; dd < SC_GBK; ++dd) v[dd] = (nv && d0 + dd < D) ? __ldg(p + dd) : 0.f;
    }
    return;
  }
  const float* p = base + (size_t)d0 * N + (nv ? n : 0);
#pragma unroll
  for (int dd = 0; dd < SC_GBK; ++dd) v[dd] = (nv && d0 + dd < D) ? __ldg(p + (size_t)dd * N) : 0.f;
}
__device__ __forceinline__ void sc_store_row(uint32_t hi_tile, uint32_t lo_tile, int r, const float (&v)[SC_GBK]) {
#pragma unroll
  for (int c = 0; c < SC_GBK / 4; ++c) {
    uint32_t h[4], l[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float x = v[c * 4 + e];
      h[e] = rna_tf32_bits(__float_as_uint(x));
      l[e] = __float_as_uint(__fsub_rn(x, __uint_as_float(h[e])));
    }
    const uint32_t off = sc_swz(r, c);
    sts128(hi_tile + off, make_uint4(h[0], h[1], h[2], h[3]));
    sts128(lo_tile + off, make_uint4(l[0], l[1], l[2], l[3]));
  }
}

constexpr int EPI_SQDIST = 2;        // square_distance on C-dim features (+ RPMNet's affinity) -> keys [B,Ns,Nt]
// matrix-valued epilogues: what is written at (i, j) for the accumulator v = a_i . b_j
template <int EPI>
__device__ __forceinline__ float sc_matrix_value(float v, float xa_i, float xb_j, float beta, float alpha, bool aff) {
  if (EPI == EPI_SQDIST) {
    // dist = -2 * matmul(src, dst^T); dist += |src|^2; dist += |dst|^2      (ppfnet_util.py:45-47)
    const float d = __fadd_rn(fmaf(-2.0f, v, xa_i), xb_j);
    return aff ? __fmul_rn(-beta, __fsub_rn(d, alpha)) : d;               // -beta * (dist - alpha)
  }
  // pd = ((-|b_j|^2) + 2 a_i.b_j) - |a_i|^2  (model_common_utils.py:5-7, same association as knn.cu)
  return __fsub_rn(fmaf(2.0f, v, -xb_j), xa_i);
}
constexpr int EPI_STATS = 3;         // attention pass 1: online (max, sum) of the scaled score rows -> stats [B,Ns,2]
constexpr int EPI_PROBS_T = 4;       // attention pass 2: softmax probabilities, transposed -> probs_t [B,Nt,Ns]
constexpr int EPI_DS = 5;            // SVD head backward: gradient of the scaled scores, plain and transposed
constexpr int EPI_SOFTMAX_XYZ = 0;   // SVD head: online softmax, xyz-weighted sums  -> out [B,3,Ns]
constexpr int EPI_KEYS = 1;          // feature-space kNN: negated expansion distances -> keys [B,Ns,Nt]

template <bool USE_TMA, int EPI, int CTAS = 1>
__global__ void __launch_bounds__(SC_THREADS, 1)
softcorr_kernel(const SoftCorrParams p, const __grid_constant__ CUtensorMap tmap_a,
                const __grid_constant__ CUtensorMap tmap_b) {
  static_assert(CTAS == 1 || (CTAS == 2 && USE_TMA), "CTA pairs exist on the TMA pipeline only");
  using Cfg = SoftCorrCfg<USE_TMA, CTAS>;
  constexpr int SC_BN = Cfg::BN, SC_BK = Cfg::BK, SC_STAGES = Cfg::STAGES, SC_STAGE_BYTES = Cfg::STAGE;
  constexpr int A_TILE = Cfg::A_TILE, B_TILE = Cfg::B_TILE, SC_TMEM_COLS = Cfg::TMEM_COLS;
  constexpr bool PAIR = (CTAS == 2);
  const uint32_t crank = PAIR ? cluster_ctarank() : 0u;   // rank 0 of a pair issues the MMAs
  extern __shared__ unsigned char sc_raw[];
  // 1024-byte alignment: the swizzle XOR is applied to absolute shared addresses
  unsigned char* tiles = reinterpret_cast<unsigned char*>(
      (reinterpret_cast<uintptr_t>(sc_raw) + 1023) & ~(uintptr_t)1023);
  SoftCorrShared* sh = reinterpret_cast<SoftCorrShared*>(tiles + SC_STAGES * SC_STAGE_BYTES);
  const uint32_t tiles_s = smem_u32(tiles);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // conditional statistics pass: every thread of every CTA reads the same word before anything is set up
  if (EPI == EPI_STATS && p.cond_flag && *reinterpret_cast<const volatile int*>(p.cond_flag) == 0) return;
  const int b = blockIdx.y;
  const int i0 = blockIdx.x * SC_BM;
  // target tiles of this CTA: blockIdx.z selects a contiguous group of p.tiles_per_split tiles (small
  // batches split the target range over several CTAs / clusters so that the whole GPU is used; each
  // group leaves a partial softmax state that softcorr_merge_kernel combines).  jb below is LOCAL.
  const int jb0 = (int)blockIdx.z * p.tiles_per_split;
  const int num_jb = min(p.tiles_per_split, (p.Nt + SC_BN - 1) / SC_BN - jb0);
  const int num_kb = (p.D + SC_BK - 1) / SC_BK;
  const int total = num_jb * num_kb;

  if (tid == 0) {
    for (int s = 0; s < SC_STAGES; ++s) {
      mbar_init(&sh->tma_full[s], 1);
      // in a pair the leader's full / acc_empty barriers also collect the peer's splitters / epilogue
      // (one arrival per warp: every lane fences, __syncwarp orders them, lane 0 arrives)
      mbar_init(&sh->full[s], SC_PROD_THREADS / 32 * CTAS);
      mbar_init(&sh->empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) { mbar_init(&sh->acc_full[a], 1); mbar_init(&sh->acc_empty[a], SC_EPI_THREADS / 32 * CTAS); }
    fence_mbar_init();
  }
  if (warp == 0) {
    if (PAIR) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                       smem_u32(&sh->tmem_base)),
                   "n"(SC_TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                       smem_u32(&sh->tmem_base)),
                   "n"(SC_TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();   // both CTAs' barriers are initialised before any remote arrive / multicast commit
  tc_fence_after();
  const uint32_t tmem = sh->tmem_base;

  if (warp < 4) {
    // ------------------------------------------------ epilogue: online softmax over target tiles
    const int i = i0 + tid;
    const float c = p.c;
    float m = -INFINITY, l = 0.f, ax = 0.f, ay = 0.f, az = 0.f;
    constexpr bool MATRIX = (EPI == EPI_KEYS || EPI == EPI_SQDIST);
    const float xi = (MATRIX && i < p.Ns) ? __ldg(p.xx_a + (size_t)b * p.Ns + i) : 0.f;
    // EPI_PROBS_T: this row's softmax statistics from the EPI_STATS pass
    float pm = 0.f, pinv = 0.f;
    if (EPI == EPI_PROBS_T && i < p.Ns) {
      pm = __ldg(p.stats + ((size_t)b * p.Ns + i) * 2);
      pinv = __fdividef(1.f, __ldg(p.stats + ((size_t)b * p.Ns + i) * 2 + 1));
    }
    // EPI_DS: row statistics, upstream gradient of this row and its dot product with the forward output
    float gx = 0.f, gy = 0.f, gz = 0.f, gc = 0.f, dscale = 0.f;
    if (EPI == EPI_DS && i < p.Ns) {
      pm = __ldg(p.stats + ((size_t)b * p.Ns + i) * 2);
      pinv = __fdividef(1.f, __ldg(p.stats + ((size_t)b * p.Ns + i) * 2 + 1));
      const float* g = p.grad_corr + (size_t)b * 3 * p.Ns + i;
      const float* co = p.corr + (size_t)b * 3 * p.Ns + i;
      gx = __ldg(g); gy = __ldg(g + p.Ns); gz = __ldg(g + 2 * (size_t)p.Ns);
      gc = fmaf(gz, __ldg(co + 2 * (size_t)p.Ns), fmaf(gy, __ldg(co + p.Ns), gx * __ldg(co)));
      dscale = c * 0.6931471805599453f;          // c = log2(e)/sqrt(D)  ->  1/sqrt(D)
    }
    const bool aff = (EPI == EPI_SQDIST) && p.aff_beta != nullptr;
    const float a_beta = aff ? __ldg(p.aff_beta + b) : 0.f, a_alpha = aff ? __ldg(p.aff_alpha + b) : 0.f;
    bool ok = true;
    for (int jb = 0; jb < num_jb; ++jb) {
      const int a = jb & 1;
      const int j0 = (jb0 + jb) * SC_BN;
#pragma unroll
      for (int jj = tid; jj < ((EPI == EPI_STATS || EPI == EPI_PROBS_T) ? 0 : SC_BN); jj += SC_EPI_THREADS) {
        const int j = j0 + jj;
        float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
        if (j < p.Nt) {
          if (MATRIX) {
            q.x = __ldg(p.xx_b + (size_t)b * p.Nt + j);
          } else {
            const float* t = p.tgt_xyz + (size_t)b * 3 * p.Nt + j;
            q = make_float4(__ldg(t), __ldg(t + p.Nt), __ldg(t + 2 * (size_t)p.Nt), 0.f);
          }
        }
        sh->xyz[a][jj] = q;
      }
      if (EPI != EPI_STATS && EPI != EPI_PROBS_T) asm volatile("bar.sync 1, 128;" ::: "memory");
      if (!mbar_wait_bounded(&sh->acc_full[a], (uint32_t)((jb >> 1) & 1))) { ok = false; break; }
      __syncwarp();
      tc_fence_after();
      const int nvalid = min(SC_BN, p.Nt - j0);
#pragma unroll 1
      for (int ch = 0; ch < SC_BN / 32; ++ch) {
        float v[32];
        tc_ld32(tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)(a * SC_BN + ch * 32), v);
        if (p.dbg_scores && i < p.Ns) {
          for (int e = 0; e < 32; ++e)
            if (j0 + ch * 32 + e < p.Nt) p.dbg_scores[((size_t)b * p.Ns + i) * p.Nt + j0 + ch * 32 + e] = v[e];
        }
        if (ch * 32 >= nvalid) continue;
        if (MATRIX) {
          // thread = row i: 32 consecutive floats of its row of the output matrix, 16-byte stores when the row allows
          const float4* xz = &sh->xyz[a][ch * 32];
          const int nv = min(32, nvalid - ch * 32);
          if (nv == 32 && (p.Nt & 3) == 0) {
            // full chunk: transpose the warp's 32 x 32 block through shared memory, then every store
            // instruction writes four complete 128-byte lines (8 lanes x 16 B per row)
            float(*tb)[36] = sh->tbuf[warp];
#pragma unroll
            for (int e = 0; e < 32; e += 4) {
              float4 o;
              o.x = sc_matrix_value<EPI>(v[e], xi, xz[e].x, a_beta, a_alpha, aff);
              o.y = sc_matrix_value<EPI>(v[e + 1], xi, xz[e + 1].x, a_beta, a_alpha, aff);
              o.z = sc_matrix_value<EPI>(v[e + 2], xi, xz[e + 2].x, a_beta, a_alpha, aff);
              o.w = sc_matrix_value<EPI>(v[e + 3], xi, xz[e + 3].x, a_beta, a_alpha, aff);
              *reinterpret_cast<float4*>(&tb[lane][e]) = o;
            }
            __syncwarp();
            const int rr = lane >> 3, cc = (lane & 7) * 4;
            const int ibase = i0 + warp * 32;
#pragma unroll
            for (int r = 0; r < 32; r += 4) {
              const float4 o = *reinterpret_cast<const float4*>(&tb[r + rr][cc]);
              const int ir = ibase + r + rr;
              if (ir < p.Ns)
                *reinterpret_cast<float4*>(p.keys + ((size_t)b * p.Ns + ir) * p.Nt + j0 + ch * 32 + cc) = o;
            }
            __syncwarp();
          } else if (i < p.Ns) {
            float* dst = p.keys + ((size_t)b * p.Ns + i) * p.Nt + j0 + ch * 32;
#pragma unroll
            for (int e = 0; e < 32; ++e)
              if (e < nv) dst[e] = sc_matrix_value<EPI>(v[e], xi, xz[e].x, a_beta, a_alpha, aff);
          }
          continue;
        }
        if (EPI == EPI_DS) {
          // dS[i,j] = P[i,j] (g_i . tgt_j - g_i . corr_i) / sqrt(D); columns beyond Nt are never stored
          const float4* xz = &sh->xyz[a][ch * 32];
          const int nv = min(32, nvalid - ch * 32);
#pragma unroll
          for (int e = 0; e < 32; ++e) {
            const float pe = __fmul_rn(ex2_approx(fmaf(v[e], c, -pm)), pinv);
            const float4 q = xz[e];
            v[e] = pe * (fmaf(gz, q.z, fmaf(gy, q.y, gx * q.x)) - gc) * dscale;
          }
          if (p.ds_t && i < p.Ns) {
            float* dst = p.ds_t + ((size_t)b * p.Nt + j0 + ch * 32) * p.Ns + i;
#pragma unroll
            for (int e = 0; e < 32; ++e)
              if (e < nv) dst[(size_t)e * p.Ns] = v[e];
          }
          if (p.ds) {
            if (nv == 32 && (p.Nt & 3) == 0) {
              float(*tb)[36] = sh->tbuf[warp];
#pragma unroll
              for (int e = 0; e < 32; e += 4) *reinterpret_cast<float4*>(&tb[lane][e]) = make_float4(v[e], v[e + 1], v[e + 2], v[e + 3]);
              __syncwarp();
              const int rr = lane >> 3, cc = (lane & 7) * 4;
              const int ibase = i0 + warp * 32;
#pragma unroll
              for (int r = 0; r < 32; r += 4) {
                const float4 o = *reinterpret_cast<const float4*>(&tb[r + rr][cc]);
                const int ir = ibase + r + rr;
                if (ir < p.Ns) *reinterpret_cast<float4*>(p.ds + ((size_t)b * p.Ns + ir) * p.Nt + j0 + ch * 32 + cc) = o;
              }
              __syncwarp();
            } else if (i < p.Ns) {
              float* dst = p.ds + ((size_t)b * p.Ns + i) * p.Nt + j0 + ch * 32;
#pragma unroll
              for (int e = 0; e < 32; ++e)
                if (e < nv) dst[e] = v[e];
            }
          }
          continue;
        }
        if (EPI == EPI_PROBS_T) {
          // P[i, j] = 2^(s c - m_i) / l_i, stored TRANSPOSED: for a fixed column j the 32 lanes (rows i) write one
          // 128-byte line of probs_t[b, j, :]
          if (i < p.Ns) {
            float* dst = p.probs_t + ((size_t)b * p.Nt + j0 + ch * 32) * p.Ns + i;
#pragma unroll
            for (int e = 0; e < 32; ++e) {
              if (ch * 32 + e < nvalid) {
                const float pe = ex2_approx(fmaf(v[e], c, -pm));
                l = __fadd_rn(l, pe);
                dst[(size_t)e * p.Ns] = p.probs_unnormalized ? pe : __fmul_rn(pe, pinv);
              }
            }
          }
          continue;
        }
        if (nvalid - ch * 32 < 32) {
#pragma unroll
          for (int e = 0; e < 32; ++e)
            if (ch * 32 + e >= nvalid) v[e] = -INFINITY;
        }
        float cm = v[0];
#pragma unroll
        for (int e = 1; e < 32; ++e) cm = fmaxf(cm, v[e]);
        const float m_new = fmaxf(m, __fmul_rn(cm, c));
        const float alpha = ex2_approx(__fsub_rn(m, m_new));
        l = __fmul_rn(l, alpha); ax = __fmul_rn(ax, alpha); ay = __fmul_rn(ay, alpha); az = __fmul_rn(az, alpha);
        m = m_new;
        const float4* xz = &sh->xyz[a][ch * 32];
#pragma unroll
        for (int e = 0; e < 32; ++e) {
          const float pe = ex2_approx(fmaf(v[e], c, -m));
          l = __fadd_rn(l, pe);
          if (EPI != EPI_STATS) {
            const float4 q = xz[e];
            ax = fmaf(pe, q.x, ax); ay = fmaf(pe, q.y, ay); az = fmaf(pe, q.z, az);
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (PAIR) mbar_arrive_cluster(&sh->acc_empty[a], 0);   // the leader's MMA warp waits for both epilogues
        else mbar_arrive(&sh->acc_empty[a]);
      }
    }
    if (!ok) {
      // a timed-out pipeline must not look like a result: poison this row's outputs with NaN (R and t downstream
      // become NaN) and raise the sticky error word for l3d_soft_correspondence_status()
      atomicCAS(p.err, 0, 1);
      const float qnan = __int_as_float(0x7fc00000);
      if (EPI == EPI_SOFTMAX_XYZ && i < p.Ns) {
        if (p.part) {
          float* q = p.part + (((size_t)b * p.Ns + i) * gridDim.z + blockIdx.z) * 8;
          q[0] = qnan; q[1] = qnan; q[2] = qnan; q[3] = qnan; q[4] = qnan;
        } else {
          float* o = p.out + (size_t)b * 3 * p.Ns + i;
          o[0] = qnan; o[p.Ns] = qnan; o[2 * (size_t)p.Ns] = qnan;
        }
      }
      if ((EPI == EPI_KEYS || EPI == EPI_SQDIST) && i < p.Ns) {
        float* dst = p.keys + ((size_t)b * p.Ns + i) * p.Nt;
        for (int j = 0; j < p.Nt; ++j) dst[j] = qnan;
      }
    }
    if (EPI == EPI_STATS && i < p.Ns) {
      const float qn = __int_as_float(0x7fc00000);
      p.stats[((size_t)b * p.Ns + i) * 2] = ok ? m : qn;
      p.stats[((size_t)b * p.Ns + i) * 2 + 1] = ok ? l : qn;
    }
    if (EPI == EPI_PROBS_T && ok && p.probs_unnormalized && i < p.Ns) p.stats[((size_t)b * p.Ns + i) * 2 + 1] = l;
    if (EPI == EPI_PROBS_T && !ok && i < p.Ns) {
      for (int j = 0; j < p.Nt; ++j) p.probs_t[((size_t)b * p.Nt + j) * p.Ns + i] = __int_as_float(0x7fc00000);
    }
    if (EPI == EPI_SOFTMAX_XYZ && ok && i < p.Ns && p.part) {
      // split target range: leave (running max in log2 units, sum, sum*xyz) for the merge kernel
      float* q = p.part + (((size_t)b * p.Ns + i) * gridDim.z + blockIdx.z) * 8;
      *reinterpret_cast<float4*>(q) = make_float4(m, l, ax, ay);
      q[4] = az;
    } else if (EPI == EPI_SOFTMAX_XYZ && ok && i < p.Ns) {
      const float inv = __fdividef(1.f, l);
      float* o = p.out + (size_t)b * 3 * p.Ns + i;
      o[0] = __fmul_rn(ax, inv);
      o[p.Ns] = __fmul_rn(ay, inv);
      o[2 * (size_t)p.Ns] = __fmul_rn(az, inv);
    }
  } else if (warp < 8) {
    const int r = tid - SC_EPI_THREADS;
    bool ok = true;
    if (USE_TMA) {
      // -------------------------------------------- splitters: lo = tf32(x - trunc_tf32(x)), smem -> smem
      for (int it = 0; it < total; ++it) {
        const int s = it % SC_STAGES;
        const uint32_t n = (uint32_t)(it / SC_STAGES);
        const uint32_t st = tiles_s + s * SC_STAGE_BYTES;
        if (!mbar_wait_bounded(&sh->tma_full[s], n & 1u)) { ok = false; break; }
#pragma unroll
        for (int op = 0; op < (p.single_pass ? 0 : 2); ++op) {
          const uint32_t hi = st + (op ? 2 * A_TILE : 0), lo = hi + (op ? B_TILE : A_TILE);
#pragma unroll
          for (int q = 0; q < (op ? B_TILE : A_TILE) / 16 / SC_PROD_THREADS; ++q) {
            const uint32_t off = (uint32_t)(q * SC_PROD_THREADS + r) * 16u;
            const uint4 x = lds128(hi + off);
            uint4 y;
            y.x = rna_tf32_bits(__float_as_uint(__fsub_rn(__uint_as_float(x.x), __uint_as_float(x.x & 0xffffe000u))));
            y.y = rna_tf32_bits(__float_as_uint(__fsub_rn(__uint_as_float(x.y), __uint_as_float(x.y & 0xffffe000u))));
            y.z = rna_tf32_bits(__float_as_uint(__fsub_rn(__uint_as_float(x.z), __uint_as_float(x.z & 0xffffe000u))));
            y.w = rna_tf32_bits(__float_as_uint(__fsub_rn(__uint_as_float(x.w), __uint_as_float(x.w & 0xffffe000u))));
            sts128(lo + off, y);
          }
        }
        if (p.dbg_scores && it == 0 && blockIdx.x == 0 && blockIdx.y == 0) {
          for (int w = r; w < SC_STAGE_BYTES / 4; w += SC_PROD_THREADS)
            g_softcorr_dbg_tiles[w] = *reinterpret_cast<const float*>(tiles + s * SC_STAGE_BYTES + w * 4);
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
          if (PAIR) mbar_arrive_cluster(&sh->full[s], 0);   // the leader's MMA reads both CTAs' tiles
          else mbar_arrive(&sh->full[s]);
        }
      }
    } else {
      // -------------------------------------------- generic producers: LDG, split, K-major swizzled STS
      const float* A = p.src_emb + (size_t)b * p.D * p.Ns;
      const float* Bm = p.tgt_emb + (size_t)b * p.D * p.Nt;
      float va[SC_GBK], vb[SC_GBK];
      for (int it = 0; it < total; ++it) {
        const int jb = it / num_kb, kb = it - jb * num_kb;
        sc_load_row(A, p.D, p.Ns, kb * SC_BK, i0 + r, va, p.kmajor);
        sc_load_row(Bm, p.D, p.Nt, kb * SC_BK, (jb0 + jb) * SC_BN + r, vb, p.kmajor);
        const int s = it % SC_STAGES;
        const uint32_t n = (uint32_t)(it / SC_STAGES);
        const uint32_t st = tiles_s + s * SC_STAGE_BYTES;
        if (!mbar_wait_bounded(&sh->empty[s], (n & 1u) ^ 1u)) { ok = false; break; }
        sc_store_row(st, st + A_TILE, r, va);
        sc_store_row(st + 2 * A_TILE, st + 2 * A_TILE + B_TILE, r, vb);
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(&sh->full[s]);
      }
    }
    if (!ok) atomicCAS(p.err, 0, 2);
  } else if (warp == 8) {
    // ------------------------------------------------ MMA issuer
    bool ok = true;
    int it = 0;
    // in a pair only rank 0 issues: its MMAs (cta_group::2, M = 256) read A and half of B from EACH CTA's
    // shared memory and write each CTA's 128 accumulator rows into that CTA's tensor memory
    for (int jb = 0; jb < num_jb && ok && crank == 0; ++jb) {
      const int a = jb & 1;
      const uint32_t pe = (uint32_t)(((jb >> 1) & 1) ^ 1);
      if (!(PAIR ? mbar_wait_bounded_cluster(&sh->acc_empty[a], pe) : mbar_wait_bounded(&sh->acc_empty[a], pe))) { ok = false; break; }
      tc_fence_after();
      const uint32_t d_tmem = tmem + (uint32_t)(a * SC_BN);
      for (int kb = 0; kb < num_kb; ++kb, ++it) {
        const int s = it % SC_STAGES;
        const uint32_t n = (uint32_t)(it / SC_STAGES);
        if (!(PAIR ? mbar_wait_bounded_cluster(&sh->full[s], n & 1u) : mbar_wait_bounded(&sh->full[s], n & 1u))) { ok = false; break; }
        tc_fence_after();
        if (lane == 0) {
          const uint32_t sa = tiles_s + s * SC_STAGE_BYTES;
          // MN-major tf32 operands exist only in the 32-byte-atom flavour of the 128 B swizzle
          // (UMMA layout 1 = TMA SWIZZLE_128B_ATOM_32B): 4-channel groups 512 B apart.
          const uint32_t lbo = USE_TMA ? (uint32_t)Cfg::ATOM : 16u, sbo = USE_TMA ? 512u : 1024u, lay = USE_TMA ? 1u : 2u;
          constexpr uint32_t idesc = sc_idesc(SC_BN, USE_TMA, SC_BM * CTAS);
          const uint64_t a_hi = sc_desc(sa, lbo, sbo, lay), a_lo = sc_desc(sa + A_TILE, lbo, sbo, lay);
          const uint64_t b_hi = sc_desc(sa + 2 * A_TILE, lbo, sbo, lay), b_lo = sc_desc(sa + 2 * A_TILE + B_TILE, lbo, sbo, lay);
#pragma unroll
          for (int k = 0; k < SC_BK / SC_UK; ++k) {
            // K-major: +32 bytes inside the 128 B swizzle row; MN-major: next 8-channel group (+1024 B)
            const uint64_t adv = (uint64_t)((USE_TMA ? k * 1024 : k * SC_UK * 4) >> 4);
            if (p.single_pass) {
              if (PAIR) tc_mma_tf32_pair(d_tmem, a_hi + adv, b_hi + adv, idesc, (kb | k) != 0);
              else tc_mma_tf32(d_tmem, a_hi + adv, b_hi + adv, idesc, (kb | k) != 0);
            } else if (PAIR) {
              tc_mma_tf32_pair(d_tmem, a_lo + adv, b_hi + adv, idesc, (kb | k) != 0);
              tc_mma_tf32_pair(d_tmem, a_hi + adv, b_lo + adv, idesc, 1u);
              tc_mma_tf32_pair(d_tmem, a_hi + adv, b_hi + adv, idesc, 1u);
            } else {
              tc_mma_tf32(d_tmem, a_lo + adv, b_hi + adv, idesc, (kb | k) != 0);
              tc_mma_tf32(d_tmem, a_hi + adv, b_lo + adv, idesc, 1u);
              tc_mma_tf32(d_tmem, a_hi + adv, b_hi + adv, idesc, 1u);
            }
          }
          if (PAIR) {
            tc_commit_pair(&sh->empty[s]);                       // frees the stage in both CTAs
            if (kb == num_kb - 1) tc_commit_pair(&sh->acc_full[a]);
          } else {
            tc_commit(&sh->empty[s]);
            if (kb == num_kb - 1) tc_commit(&sh->acc_full[a]);
          }
        }
        __syncwarp();
      }
    }
    if (!ok && lane == 0) atomicCAS(p.err, 0, 3);
  } else if (USE_TMA) {
    // ------------------------------------------------ TMA issuer: 4 + 8 boxes of [16 d x 32 n] per stage
    bool ok = true;
    for (int it = 0; it < total; ++it) {
      const int jb = it / num_kb, kb = it - jb * num_kb;
      const int s = it % SC_STAGES;
      const uint32_t n = (uint32_t)(it / SC_STAGES);
      if (!mbar_wait_bounded(&sh->empty[s], (n & 1u) ^ 1u)) { ok = false; break; }
      if (lane == 0) {
        const uint32_t st = tiles_s + s * SC_STAGE_BYTES;
        mbar_arrive_expect_tx(&sh->tma_full[s], A_TILE + B_TILE);
        if (p.tma4) {
          // chunked 4-D maps (Ns, Nt multiples of 32): one instruction per operand tile
          tma_load_4d(st, &tmap_a, 0, kb * SC_BK, i0 / 32, b, &sh->tma_full[s]);
          tma_load_4d(st + 2 * A_TILE, &tmap_b, 0, kb * SC_BK, ((jb0 + jb) * SC_BN + (int)crank * Cfg::BN_LOCAL) / 32, b,
                      &sh->tma_full[s]);
        } else {
#pragma unroll
          for (int q = 0; q < SC_BM / 32; ++q)
            tma_load_3d(st + q * Cfg::ATOM, &tmap_a, i0 + 32 * q, kb * SC_BK, b, &sh->tma_full[s]);
          // a pair member fetches only its half of the 256 target columns
#pragma unroll
          for (int q = 0; q < Cfg::BN_LOCAL / 32; ++q)
            tma_load_3d(st + 2 * A_TILE + q * Cfg::ATOM, &tmap_b, (jb0 + jb) * SC_BN + (int)crank * Cfg::BN_LOCAL + 32 * q,
                        kb * SC_BK, b, &sh->tma_full[s]);
        }
      }
      __syncwarp();
    }
    if (!ok && lane == 0) atomicCAS(p.err, 0, 4);
  }

  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();   // the peer may still be arriving on our barriers / its MMAs reading our tiles
  if (warp == 0) {
    tc_fence_after();
    if (PAIR)
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(SC_TMEM_COLS) : "memory");
    else
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(SC_TMEM_COLS) : "memory");
  }
}

template <bool USE_TMA, int CTAS = 1>
size_t softcorr_smem_bytes() {
  return (size_t)SoftCorrCfg<USE_TMA, CTAS>::STAGES * SoftCorrCfg<USE_TMA, CTAS>::STAGE + sizeof(SoftCorrShared) + 1024;
}

// emb [B, D, N] fp32 as a 3-D tensor (n fastest); boxes of 32 n x BK d, 128B-swizzled; OOB -> 0
static bool make_emb_tmap(CUtensorMap* m, const float* emb, int B, int D, int N) {
  return make_dn_tmap(m, emb, B, D, N, SoftCorrCfg<true>::BK);
}

}  // namespace l3d

using namespace l3d;

static thread_local int g_softcorr_force_generic = 0;   // testing hooks are per host thread
static thread_local int g_softcorr_tma3 = 0;            // 1: keep the 3-D maps (32-point boxes) on aligned shapes too

// -1: never split the target range, 0: automatic (small batches), > 0: forced number of splits (testing hook)
static thread_local int g_softcorr_split = 0;

// Combines the partial softmax states of a split target range: state z = (m_z in log2 units, l_z, a_z[3]);
// out = sum_z a_z 2^(m_z - M) / sum_z l_z 2^(m_z - M), M = max_z m_z.
static __global__ void softcorr_merge_kernel(const float* __restrict__ part, int B, int Ns, int nsplit,
                                             float* __restrict__ out) {
  const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long)B * Ns) return;
  const float* q = part + (size_t)t * nsplit * 8;
  float M = -INFINITY;
  for (int z = 0; z < nsplit; ++z) M = fmaxf(M, q[z * 8]);
  float l = 0.f, ax = 0.f, ay = 0.f, az = 0.f;
  for (int z = 0; z < nsplit; ++z) {
    const float w = ex2_approx(__fsub_rn(q[z * 8], M));
    l = fmaf(w, q[z * 8 + 1], l);
    ax = fmaf(w, q[z * 8 + 2], ax); ay = fmaf(w, q[z * 8 + 3], ay); az = fmaf(w, q[z * 8 + 4], az);
  }
  const int b = (int)(t / Ns), i = (int)(t - (long)b * Ns);
  const float inv = __fdividef(1.f, l);
  float* o = out + (size_t)b * 3 * Ns + i;
  o[0] = __fmul_rn(ax, inv); o[Ns] = __fmul_rn(ay, inv); o[2 * (size_t)Ns] = __fmul_rn(az, inv);
}

// Launches the GEMM pipeline with epilogue EPI on an already filled parameter block (src_emb, tgt_emb,
// B, D, Ns, Nt and the epilogue's own pointers).
template <int EPI>
static int sc_launch(SoftCorrParams p, void* stream) {
  if (p.B > 65535) return L3D_ERR_UNSUPPORTED;
  const size_t smem_t = softcorr_smem_bytes<true>(), smem_g = softcorr_smem_bytes<false>();
  const size_t smem_p = softcorr_smem_bytes<true, 2>();
  int dev = 0;
  cudaGetDevice(&dev);
  {
    cudaError_t e = raise_smem_once<softcorr_kernel<true, EPI>>(dev, smem_t);
    if (e == cudaSuccess) e = raise_smem_once<softcorr_kernel<false, EPI>>(dev, smem_g);
    if (e == cudaSuccess) e = raise_smem_once<softcorr_kernel<true, EPI, 2>>(dev, smem_p);
    if (e != cudaSuccess) return (int)e;
  }
  p.c = (float)(1.4426950408889634 / sqrt((double)p.D));
  void* errp = nullptr;
  cudaError_t e = cudaGetSymbolAddress(&errp, g_softcorr_error);
  if (e != cudaSuccess) return (int)e;
  p.err = (int*)errp;
  dim3 grid((p.Ns + SC_BM - 1) / SC_BM, p.B);

  // TMA needs 16-byte global strides and bases
  bool tma = g_softcorr_force_generic != 1 && !p.kmajor && (p.Ns % 4 == 0) && (p.Nt % 4 == 0) &&
             (((uintptr_t)p.src_emb | (uintptr_t)p.tgt_emb) & 15) == 0;
  CUtensorMap ma, mb;
  memset(&ma, 0, sizeof(ma)); memset(&mb, 0, sizeof(mb));
  const bool pair = tma && g_softcorr_force_generic != 2 && p.Ns > SC_BM;
  p.tma4 = 0;
  if (tma && g_softcorr_tma3 == 0 && (p.Ns % 32 == 0) && (p.Nt % 32 == 0)) {
    constexpr int BK = SoftCorrCfg<true>::BK;
    const int bchunks = (pair ? SoftCorrCfg<true, 2>::BN_LOCAL : SoftCorrCfg<true>::BN_LOCAL) / 32;
    if (make_dn_tmap4(&ma, p.src_emb, p.B, p.D, p.Ns, BK, SC_BM / 32) && make_dn_tmap4(&mb, p.tgt_emb, p.B, p.D, p.Nt, BK, bchunks))
      p.tma4 = 1;
  }
  if (tma && !p.tma4) tma = make_emb_tmap(&ma, p.src_emb, p.B, p.D, p.Ns) && make_emb_tmap(&mb, p.tgt_emb, p.B, p.D, p.Nt);

  // Small batches: with one CTA (pair) per 128 (256) source rows a B = 2 call would occupy 8 of 74 TPCs.
  // Split the target tiles over gridDim.z so that about one wave of CTAs exists; each split leaves a
  // partial softmax state per row (EPI_SOFTMAX_XYZ), combined by softcorr_merge_kernel.
  const int bn = tma ? SoftCorrCfg<true>::BN : SoftCorrCfg<false>::BN;
  const int tiles = (p.Nt + bn - 1) / bn;
  const long units = pair ? (long)((p.Ns + 2 * SC_BM - 1) / (2 * SC_BM)) * p.B : (long)grid.x * p.B;
  const int sms = sm_count(dev);
  const long slots = pair ? sms / 2 : sms;             // 1 CTA per SM; a pair needs both SMs of a TPC
  int jsplit = 1;
  if (EPI != EPI_STATS && EPI != EPI_DS && !(EPI == EPI_PROBS_T && p.probs_unnormalized) && g_softcorr_split >= 0 &&
      tiles > 1 && units * 2 <= slots) {
    jsplit = (int)((slots + units - 1) / units);
    if (g_softcorr_split > 0) jsplit = g_softcorr_split;
    if (jsplit > tiles) jsplit = tiles;
  }
  p.tiles_per_split = (tiles + jsplit - 1) / jsplit;
  jsplit = (tiles + p.tiles_per_split - 1) / p.tiles_per_split;     // no empty split
  p.part = nullptr;
  if (EPI == EPI_SOFTMAX_XYZ && jsplit > 1) {
    // stream-ordered scratch from the device's default pool; keep freed blocks cached in the pool (the
    // default release threshold of 0 hands them back to the driver at every sync: ~100 us per call)
    static thread_local int pool_dev = -1;
    if (pool_dev != dev) {
      cudaMemPool_t pool;
      if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
        uint64_t keep = UINT64_MAX;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
      }
      pool_dev = dev;
    }
    cudaError_t me = cudaMallocAsync((void**)&p.part, (size_t)p.B * p.Ns * jsplit * 8 * sizeof(float),
                                     (cudaStream_t)stream);
    if (me != cudaSuccess) return (int)me;
  }
  grid.z = jsplit;
  if (pair) {
    // CTA pairs: cluster (2,1,1), two adjacent 128-row blocks of one batch item (an odd last block gets an
    // all-out-of-range partner: TMA zero-fills its tiles and its epilogue stores nothing)
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * ((p.Ns + 2 * SC_BM - 1) / (2 * SC_BM)), p.B, jsplit);
    cfg.blockDim = dim3(SC_THREADS);
    cfg.dynamicSmemBytes = smem_p;
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    cudaError_t le = cudaLaunchKernelEx(&cfg, softcorr_kernel<true, EPI, 2>, p, ma, mb);
    if (le != cudaSuccess) {
      if (p.part) cudaFreeAsync(p.part, (cudaStream_t)stream);
      return (int)le;
    }
  } else if (tma)
    softcorr_kernel<true, EPI><<<grid, SC_THREADS, smem_t, (cudaStream_t)stream>>>(p, ma, mb);
  else
    softcorr_kernel<false, EPI><<<grid, SC_THREADS, smem_g, (cudaStream_t)stream>>>(p, ma, mb);
  count_launch();
  {
    const cudaError_t le2 = cudaGetLastError();
    if (le2 != cudaSuccess) {
      if (p.part) cudaFreeAsync(p.part, (cudaStream_t)stream);   // do not leak the scratch on a failed launch
      return (int)le2;
    }
  }
  if (p.part) {
    const long rows = (long)p.B * p.Ns;
    softcorr_merge_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, (cudaStream_t)stream>>>(p.part, p.B, p.Ns,
                                                                                            jsplit, p.out);
    count_launch();
    cudaError_t fe = cudaFreeAsync(p.part, (cudaStream_t)stream);
    L3D_LAUNCH_CHECK();
    if (fe != cudaSuccess) return (int)fe;
  }
  return L3D_OK;
}

static int softcorr_launch(const float* src_emb, const float* tgt_emb, const float* tgt_xyz, int B, int D,
                           int Ns, int Nt, float* src_corr, float* dbg_scores, void* stream) {
  if (B < 0 || D < 0 || Ns < 0 || Nt < 0) return L3D_ERR_INVALID;
  if (B == 0 || Ns == 0) return L3D_OK;
  if (!src_emb || !tgt_emb || !tgt_xyz || !src_corr) return L3D_ERR_INVALID;
  if (Nt == 0 || D == 0) return L3D_ERR_INVALID;      // softmax over an empty row is undefined
  SoftCorrParams p;
  memset(&p, 0, sizeof(p));
  p.src_emb = src_emb; p.tgt_emb = tgt_emb; p.tgt_xyz = tgt_xyz; p.out = src_corr; p.dbg_scores = dbg_scores;
  p.B = B; p.D = D; p.Ns = Ns; p.Nt = Nt;
  return sc_launch<EPI_SOFTMAX_XYZ>(p, stream);
}

// ---- feature-space kNN: knn() of utils/model_common_utils.py:3-9 for C != 3 -----------------------------
// xx[b,n] = sum_c x[b,c,n]^2, accumulated in channel order (torch.sum(x**2, dim=1), :6)
// 256 threads = 32 points x 8 channel slices: coalesced over points, 8 partial sums per point combined
// in slice order (deterministic; the row is toleranced anyway, §3.7)
static __global__ void sqnorm_kernel(const float* __restrict__ x, int B, int C, int N, float* __restrict__ xx) {
  __shared__ float part[8][33];
  const int ln = threadIdx.x & 31, sl = threadIdx.x >> 5;
  const long t = (long)blockIdx.x * 32 + ln;            // flattened (b, n)
  float acc = 0.f;
  if (t < (long)B * N) {
    const int b = (int)(t / N), n = (int)(t - (long)b * N);
    const float* p = x + (size_t)b * C * N + n;
    const int c0 = (int)((long)C * sl / 8), c1 = (int)((long)C * (sl + 1) / 8);
    for (int c = c0; c < c1; ++c) {
      const float v = __ldg(p + (size_t)c * N);
      acc = __fadd_rn(acc, __fmul_rn(v, v));
    }
  }
  part[sl][ln] = acc;
  __syncthreads();
  if (sl == 0 && t < (long)B * N) {
    float s = part[0][ln];
#pragma unroll
    for (int k = 1; k < 8; ++k) s = __fadd_rn(s, part[k][ln]);
    xx[t] = s;
  }
}

// |x_n|^2 for [B, N, C] rows (channels contiguous): torch.sum(x ** 2, dim=-1), accumulated in channel order
static __global__ void sqnorm_rows_kernel(const float* __restrict__ x, long rows, int C, float* __restrict__ xx) {
  const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= rows) return;
  const float* p = x + (size_t)t * C;
  float acc = 0.f;
  for (int c = 0; c < C; ++c) acc = __fadd_rn(acc, __fmul_rn(p[c], p[c]));
  xx[t] = acc;
}

extern "C" size_t l3d_feature_square_distance_ws_bytes(int B, int N, int M) {
  if (B < 1 || N < 1 || M < 1) return 0;
  return sizeof(float) * (size_t)B * ((size_t)N + M);
}

// square_distance(src, dst) of utils/ppfnet_util.py:29-48 / model_common_utils.py:19-38 for C-dimensional features
// (RPMNet's match_features, models/rpmnet.py:130-154): src [B,N,C], dst [B,M,C] -> out [B,N,M], Gram matrix on
// tcgen05 (3xTF32).  With beta/alpha ([B] each) the epilogue writes RPMNet's affinity -beta*(dist - alpha) instead.
extern "C" int l3d_feature_square_distance(const float* src_dev, const float* dst_dev, int B, int N, int M, int C,
                                           const float* beta_dev, const float* alpha_dev, float* out_dev,
                                           void* ws_dev, void* stream) {
  if (B < 0 || N < 0 || M < 0 || C < 1) return L3D_ERR_INVALID;
  if (B == 0 || N == 0 || M == 0) return L3D_OK;
  if (!src_dev || !dst_dev || !out_dev || !ws_dev || ((beta_dev == nullptr) != (alpha_dev == nullptr))) return L3D_ERR_INVALID;
  float* xa = reinterpret_cast<float*>(ws_dev);
  float* xb = xa + (size_t)B * N;
  const long ra = (long)B * N, rb = (long)B * M;
  sqnorm_rows_kernel<<<(unsigned)((ra + 255) / 256), 256, 0, (cudaStream_t)stream>>>(src_dev, ra, C, xa);
  count_launch();
  L3D_LAUNCH_CHECK();
  sqnorm_rows_kernel<<<(unsigned)((rb + 255) / 256), 256, 0, (cudaStream_t)stream>>>(dst_dev, rb, C, xb);
  count_launch();
  L3D_LAUNCH_CHECK();
  SoftCorrParams p;
  memset(&p, 0, sizeof(p));
  p.src_emb = src_dev; p.tgt_emb = dst_dev; p.xx_a = xa; p.xx_b = xb; p.keys = out_dev;
  p.aff_beta = beta_dev; p.aff_alpha = alpha_dev; p.kmajor = 1;
  p.B = B; p.D = C; p.Ns = N; p.Nt = M;
  return sc_launch<EPI_SQDIST>(p, stream);
}

static size_t knn_features_keys_bytes(int B, int N) {
  return (((size_t)B * N * N * sizeof(float)) + 255) & ~(size_t)255;
}

extern "C" size_t l3d_knn_features_ws_bytes(int B, int C, int N) {
  (void)C;
  if (B <= 0 || N <= 0) return 0;
  return knn_features_keys_bytes(B, N) + (size_t)B * N * sizeof(float);
}

extern "C" int l3d_knn_features(const float* x_dev, int B, int C, int N, int k, int64_t* idx_dev, void* ws_dev,
                                void* stream) {
  if (B < 0 || C < 1 || N < 0 || k < 1) return L3D_ERR_INVALID;
  if (B == 0 || N == 0) return L3D_OK;
  if (!x_dev || !idx_dev || !ws_dev || k > N) return L3D_ERR_INVALID;
  if (((uintptr_t)ws_dev & 15) != 0) return L3D_ERR_INVALID;
  float* keys = reinterpret_cast<float*>(ws_dev);
  float* xx = reinterpret_cast<float*>(reinterpret_cast<unsigned char*>(ws_dev) + knn_features_keys_bytes(B, N));
  const long rows = (long)B * N;
  sqnorm_kernel<<<(unsigned)((rows + 31) / 32), 256, 0, (cudaStream_t)stream>>>(x_dev, B, C, N, xx);
  count_launch();
  L3D_LAUNCH_CHECK();
  SoftCorrParams p;
  memset(&p, 0, sizeof(p));
  p.src_emb = x_dev; p.tgt_emb = x_dev; p.xx_a = xx; p.xx_b = xx; p.keys = keys;
  p.B = B; p.D = C; p.Ns = N; p.Nt = N;
  int rc = sc_launch<EPI_KEYS>(p, stream);
  if (rc != L3D_OK) return rc;
  return knn_select_from_matrix(keys, rows, N, k, reinterpret_cast<long long*>(idx_dev), (cudaStream_t)stream);
}

// ---- attention (utils/transformer.py:17-23): softmax(q k^T / sqrt(d_k)) in two passes over the tcgen05 score
// pipeline; the probabilities leave the kernel transposed, ready to be the activation operand of the P.V GEMM.
// q_dev [BH, D, Nq], k_dev [BH, D, Nk] (channel-major per batch x head) -> stats_dev [BH, Nq, 2]
// precise = 0: the row max from ONE TF32 pass (the exponent reference only has to be close to the true max; the
// row sum slot is then meaningless and is rewritten by l3d_attention_probs_t(normalized = 0) with the exact sums)
extern "C" int l3d_attention_stats(const float* q_dev, const float* k_dev, int BH, int D, int Nq, int Nk, int precise,
                                   float* stats_dev, void* stream) {
  if (BH < 0 || D < 1 || Nq < 0 || Nk < 1) return L3D_ERR_INVALID;
  if (BH == 0 || Nq == 0) return L3D_OK;
  if (!q_dev || !k_dev || !stats_dev) return L3D_ERR_INVALID;
  SoftCorrParams p;
  memset(&p, 0, sizeof(p));
  p.src_emb = q_dev; p.tgt_emb = k_dev; p.stats = stats_dev;
  p.B = BH; p.D = D; p.Ns = Nq; p.Nt = Nk;
  p.single_pass = precise ? 0 : 1;
  return sc_launch<EPI_STATS>(p, stream);
}
// ---- bound-referenced softmax -----------------------------------------------------------------------------------
// The exponent reference of a softmax row does not have to be the row maximum: any m_i with
// max_j s_ij - m_i in (-~100, 0] (log2 units) gives the same probabilities after normalisation, without overflow or
// underflow.  Cauchy-Schwarz supplies one for free:  |q_i . k_j| <= |q_i| max_j |k_j|, so
// m_i = |q_i| * max_j |k_j| * log2(e) / sqrt(D) >= every scaled score of the row, and the row maximum is at least
// -m_i.  Whenever m_i <= ATTN_BOUND_MAX for every row of the call (2 m_i <= 80: the largest term is >= 2^-80), the
// statistics pass is unnecessary; otherwise a device flag is raised and l3d_attention_stats_if computes the true
// maxima.  Nothing comes back to the host.
constexpr float ATTN_BOUND_MAX = 40.0f;

// thread = key j: |k_j| over the D channels of x [BH, D, N] (coalesced over j); block max -> atomicMax on the bits
static __global__ void attn_colnorm_max_kernel(const float* __restrict__ x, int D, int N, unsigned int* __restrict__ out_max) {
  const int bh = blockIdx.y;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  float acc = 0.f;
  if (j < N) {
    const float* px = x + (size_t)bh * D * N + j;
    for (int d = 0; d < D; ++d) { const float v = px[(size_t)d * N]; acc = fmaf(v, v, acc); }
  }
  float nrm = sqrtf(acc);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) nrm = fmaxf(nrm, __shfl_xor_sync(L3D_FULL_MASK, nrm, o));
  if ((threadIdx.x & 31) == 0 && !(nrm <= 0.f)) atomicMax(out_max + bh, __float_as_uint(nrm));   // NaN propagates too
}

// thread = query i: m_i = |q_i| * kmax[bh] * c (rounded up a little) -> stats[(bh, i), 0]; raises *flag when too large
static __global__ void attn_row_bound_kernel(const float* __restrict__ q, int D, int N, const unsigned int* __restrict__ kmax,
                                             float c, float* __restrict__ stats, int* __restrict__ flag) {
  const int bh = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  const float* pq = q + (size_t)bh * D * N + i;
  float acc = 0.f;
  for (int d = 0; d < D; ++d) { const float v = pq[(size_t)d * N]; acc = fmaf(v, v, acc); }
  const float m = sqrtf(acc) * __uint_as_float(kmax[bh]) * c * 1.0001f;
  stats[((size_t)bh * N + i) * 2] = m;
  if (!(m <= ATTN_BOUND_MAX)) atomicOr(flag, 1);      // also raised by NaN / Inf
}

extern "C" size_t l3d_attention_bounds_ws_bytes(int BH) { return BH < 0 ? 0 : sizeof(int) * ((size_t)BH + 1); }

// q_dev [BH, D, Nq], k_dev [BH, D, Nk] -> stats_dev[(bh, i), 0] = the row's exponent reference (an upper bound of its
// scaled scores); ws_dev (l3d_attention_bounds_ws_bytes) receives max_j |k_j| per head and, in its LAST int, the flag
// "some row's bound is too loose: run the statistics pass" consumed by l3d_attention_stats_if.
extern "C" int l3d_attention_bounds(const float* q_dev, const float* k_dev, int BH, int D, int Nq, int Nk, float* stats_dev,
                                    void* ws_dev, void* stream) {
  if (BH < 0 || D < 1 || Nq < 0 || Nk < 1) return L3D_ERR_INVALID;
  if (BH == 0 || Nq == 0) return L3D_OK;
  if (!q_dev || !k_dev || !stats_dev || !ws_dev) return L3D_ERR_INVALID;
  if (BH > 65535) return L3D_ERR_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  unsigned int* kmax = (unsigned int*)ws_dev;
  int* flag = (int*)ws_dev + BH;
  cudaError_t e = cudaMemsetAsync(ws_dev, 0, sizeof(int) * ((size_t)BH + 1), st);
  if (e != cudaSuccess) return (int)e;
  attn_colnorm_max_kernel<<<dim3((unsigned)((Nk + 255) / 256), (unsigned)BH), 256, 0, st>>>(k_dev, D, Nk, kmax);
  count_launch();
  L3D_LAUNCH_CHECK();
  const float c = (float)(1.4426950408889634 / sqrt((double)D));
  attn_row_bound_kernel<<<dim3((unsigned)((Nq + 255) / 256), (unsigned)BH), 256, 0, st>>>(q_dev, D, Nq, kmax, c, stats_dev, flag);
  count_launch();
  L3D_LAUNCH_CHECK();
  return L3D_OK;
}

// l3d_attention_stats(precise = 0) that runs only if *flag_dev != 0 (flag_dev = the last int of l3d_attention_bounds'
// workspace); when it runs it replaces the bounds in stats_dev[.., 0] by the true row maxima.
extern "C" int l3d_attention_stats_if(const float* q_dev, const float* k_dev, int BH, int D, int Nq, int Nk,
                                      const int* flag_dev, float* stats_dev, void* stream) {
  if (BH < 0 || D < 1 || Nq < 0 || Nk < 1) return L3D_ERR_INVALID;
  if (BH == 0 || Nq == 0) return L3D_OK;
  if (!q_dev || !k_dev || !stats_dev || !flag_dev) return L3D_ERR_INVALID;
  SoftCorrParams p;
  memset(&p, 0, sizeof(p));
  p.src_emb = q_dev; p.tgt_emb = k_dev; p.stats = stats_dev;
  p.B = BH; p.D = D; p.Ns = Nq; p.Nt = Nk;
  p.single_pass = 1;
  p.cond_flag = flag_dev;
  return sc_launch<EPI_STATS>(p, stream);
}

// ... + stats_dev -> probs_t_dev [BH, Nk, Nq] = softmax(q^T k / sqrt(D), over k) transposed
extern "C" int l3d_attention_probs_t(const float* q_dev, const float* k_dev, float* stats_dev, int BH, int D, int Nq,
                                     int Nk, int normalized, float* probs_t_dev, void* stream) {
  if (BH < 0 || D < 1 || Nq < 0 || Nk < 1) return L3D_ERR_INVALID;
  if (BH == 0 || Nq == 0) return L3D_OK;
  if (!q_dev || !k_dev || !stats_dev || !probs_t_dev) return L3D_ERR_INVALID;
  SoftCorrParams p;
  memset(&p, 0, sizeof(p));
  p.src_emb = q_dev; p.tgt_emb = k_dev; p.stats = stats_dev; p.probs_t = probs_t_dev;
  p.B = BH; p.D = D; p.Ns = Nq; p.Nt = Nk;
  p.probs_unnormalized = normalized ? 0 : 1;
  return sc_launch<EPI_PROBS_T>(p, stream);
}

// Backward of l3d_soft_correspondence w.r.t. the SCALED-score logits: with P = softmax(src_emb^T tgt_emb / sqrt(D)),
// dS[i,j] = P[i,j] (g_i . tgt_j - g_i . src_corr_i) / sqrt(D) is written once plain (ds_dev [B,Ns,Nt]) and once
// transposed (ds_t_dev [B,Nt,Ns]); either may be NULL.  The two embedding gradients are then plain GEMMs
//   d src_emb = tgt_emb . dS^T,   d tgt_emb = src_emb . dS      (l3d_linear_cm with per-item weights).
// stats_dev [B,Ns,2] comes from l3d_attention_stats(src_emb, tgt_emb).
extern "C" int l3d_soft_correspondence_dscores(const float* src_emb, const float* tgt_emb, const float* tgt_xyz,
                                               const float* stats_dev, const float* grad_corr_dev,
                                               const float* corr_dev, int B, int D, int Ns, int Nt, float* ds_dev,
                                               float* ds_t_dev, void* stream) {
  if (B < 0 || D < 1 || Ns < 0 || Nt < 1) return L3D_ERR_INVALID;
  if (B == 0 || Ns == 0) return L3D_OK;
  if (!src_emb || !tgt_emb || !tgt_xyz || !stats_dev || !grad_corr_dev || !corr_dev || (!ds_dev && !ds_t_dev))
    return L3D_ERR_INVALID;
  SoftCorrParams p;
  memset(&p, 0, sizeof(p));
  p.src_emb = src_emb; p.tgt_emb = tgt_emb; p.tgt_xyz = tgt_xyz; p.stats = const_cast<float*>(stats_dev);
  p.grad_corr = grad_corr_dev; p.corr = corr_dev; p.ds = ds_dev; p.ds_t = ds_t_dev;
  p.B = B; p.D = D; p.Ns = Ns; p.Nt = Nt;
  return sc_launch<EPI_DS>(p, stream);
}

extern "C" int l3d_soft_correspondence(const float* src_emb, const float* tgt_emb, const float* tgt_xyz,
                                       int B, int D, int Ns, int Nt, float* src_corr, void* stream) {
  return softcorr_launch(src_emb, tgt_emb, tgt_xyz, B, D, Ns, Nt, src_corr, nullptr, stream);
}

// Debug variant: additionally dumps the raw (unscaled) score accumulators to scores_dev [B,Ns,Nt].
extern "C" int l3d_debug_soft_correspondence_scores(const float* src_emb, const float* tgt_emb,
                                                    const float* tgt_xyz, int B, int D, int Ns, int Nt,
                                                    float* src_corr, float* scores_dev, void* stream) {
  if (!scores_dev) return L3D_ERR_INVALID;
  return softcorr_launch(src_emb, tgt_emb, tgt_xyz, B, D, Ns, Nt, src_corr, scores_dev, stream);
}

// Debug aid: copies the stage-0 operand tiles (A_hi, A_lo, B_hi, B_lo; 4 x 4096 floats, shared-memory image)
// that CTA (0,0) of the last l3d_debug_soft_correspondence_scores launch saw on the TMA path.
extern "C" int l3d_debug_soft_correspondence_tiles(float* host_out) {
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) return (int)e;
  return (int)cudaMemcpyFromSymbol(host_out, g_softcorr_dbg_tiles, sizeof(float) * SoftCorrCfg<true>::STAGE / 4);
}

// Testing hook: nonzero forces the generic (LDG producer) operand pipeline even for TMA-eligible shapes.
// 0: automatic, 1: generic (non-TMA) pipeline, 2: TMA without CTA pairs, 3: automatic but with the 3-D tensor maps
// (32-point boxes) on shapes that would take the chunked 4-D maps — also honoured by edgeconv.cu
extern "C" void l3d_debug_soft_correspondence_force_generic(int on) {
  g_softcorr_force_generic = (on == 3) ? 0 : on;
  g_softcorr_tma3 = (on == 3) ? 1 : 0;
}
namespace l3d { int tma3_boxes_forced() { return g_softcorr_tma3; } }

// Testing hook: -1 = never split the target range over CTAs, 0 = automatic, n > 0 = force n splits.
extern "C" void l3d_debug_soft_correspondence_split(int n) { g_softcorr_split = n; }

// Synchronises the device and returns the pipeline error word of l3d_soft_correspondence
// (0 = ok; 1/2/3/4 = an epilogue / producer / MMA-issuer / TMA-issuer wait ran out).  Test and debug aid.
extern "C" int l3d_soft_correspondence_status(void) {
  int v = 0;
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) return (int)e;
  e = cudaMemcpyFromSymbol(&v, g_softcorr_error, sizeof(int));
  if (e != cudaSuccess) return (int)e;
  if (v != 0) {                    // report once, then clear: the word is not sticky across calls
    const int zero = 0;
    cudaMemcpyToSymbol(g_softcorr_error, &zero, sizeof(int));
  }
  return v;
}
