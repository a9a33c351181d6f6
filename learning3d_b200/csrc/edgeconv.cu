// DGCNN's EdgeConv stack on the 5th-gen tensor cores (sm_100a: TMA + tcgen05 + TMEM), SURVEY.md §8f rank 1.
//
// Replaces models/dgcnn.py:32-48 in eval mode:
//     x = get_graph_feature(xyz)                                [B, 6, N, k]   never written here
//     x = relu(bn_i(conv_i(x)));  out_i = x.max(dim=-1)          i = 1..4       (64, 64, 128, 256 channels)
//     y = relu(bn5(conv5(cat(out_1..out_4))))                                   [B, emb, N]
//
// Layer 1 (K = 6) is CUDA-core work straight from the kNN indices and the [B,3,N] cloud (edge_l1_kernel:
// gather-on-load, the concatenated graph feature never exists).  Layers 2-4 and conv5 are GEMMs
//     D[C_out, positions] = W[C_out, C_in] . X[C_in, positions]
// with positions = (point, neighbour) pairs, run by ONE persistent kernel design (edge_gemm_kernel):
//   * "swap-AB": the weights are the M-side operand (lane of the accumulator = output channel), the activations
//     the N-side operand.  Both are MN-major fp32 in HBM exactly as torch holds them (W^T [C_in, C_out] prepared
//     once per module, X = [B, C_in, N*k]), so 3-D tensor-map TMA drops [16 ch x 32] boxes into shared memory
//     and the tensor core reads them in place (SWIZZLE_128B_ATOM_32B = UMMA layout 1) — no transposes.
//   * fp32-class accuracy: 3xTF32 (hi.hi + hi.lo + lo.hi, fp32 accumulate in TMEM) like softcorr.cu: the raw fp32
//     tile is the hi operand, four splitter warps derive the lo tiles shared-to-shared.
//   * epilogue in the accumulator's own layout: thread = output channel, registers = consecutive positions, so
//     folded BatchNorm + ReLU is one FFMA + FMNMX per value and the max over the k neighbours of a point is a
//     running max over k consecutive registers — no shuffles, no atomics.  Tiles advance by a multiple of k
//     positions (240 of the 256 MMA columns at k = 20) so that a group never straddles two tiles.
//   * C_out = 256 / conv5: CTA pairs (cluster of 2, tcgen05 cta_group::2, M = 256): each CTA keeps 128 output
//     channels and stages only half of the activation columns.
//   * persistent: one CTA (pair) per SM (TPC), static round-robin over (batch item, position tile, channel
//     block) units; two 256-column accumulators in TMEM so the epilogue of unit i overlaps the MMAs of i+1.
// Every mbarrier wait is bounded; a timed-out pipeline writes NaN to everything it still owed and raises the
// error word read by l3d_edgeconv_status().
#include "common.cuh"
#include "tc05.cuh"
#include "../../include/l3d_b200.h"
#include "launch_count.h"

#include <math.h>
#include <string.h>

namespace l3d {

constexpr int EC_EPI_THREADS = 128;   // one epilogue group = 4 warps = the 128 TMEM lanes of an accumulator
constexpr int EC_EPI_GROUPS = 2;      // group g drains accumulator g (even / odd tiles)
constexpr int EC_SPLIT_THREADS = 128;
// warps 0-3 epilogue group 0 | 4-7 splitters | 8 MMA issuer | 9 TMA issuer | 10-13 epilogue group 1
constexpr int EC_THREADS = EC_EPI_THREADS + EC_SPLIT_THREADS + 64 + EC_EPI_THREADS;
constexpr int EC_BN = 256;           // positions per MMA (UMMA N)
constexpr int EC_BK = 16;            // input channels per pipeline stage
constexpr int EC_MAX_GROUPS = 32;    // pooled groups (points) per tile
constexpr int EC_MAX_STAGES = 6;

template <int CTAS>
struct EdgeCfg {
  static constexpr int STAGES = CTAS == 2 ? 6 : 4;
  static constexpr int BN_LOCAL = EC_BN / CTAS;            // activation columns staged by this CTA
  static constexpr int A_TILE = SC_BM * EC_BK * 4;         // 8 KB   [16 ch x 128 out-channels]
  static constexpr int B_TILE = BN_LOCAL * EC_BK * 4;      // 16 / 8 KB
  static constexpr int STAGE = 2 * A_TILE + 2 * B_TILE;    // W_hi, W_lo, X_hi, X_lo: 48 / 32 KB
  static constexpr int ATOM = 32 * EC_BK * 4;              // one [16 ch x 32] TMA box
  static constexpr int TMEM_COLS = 2 * EC_BN;
};

struct EdgeParams {
  const float* scale;    // [M] folded BatchNorm scale  gamma / sqrt(var + eps)
  const float* shift;    // [M] folded shift            beta - mean * scale
  float* h_out;          // optional [B, M, P]: relu(bn(conv(x)))
  float* pool_out;       // optional: max over each group of G positions -> pool_out[b*pool_bstride + (pool_coff+c)*pool_n + n]
  long pool_bstride;
  int pool_coff, pool_n;
  int* err;
  int B, M, K, P;        // batch, output channels, input channels, positions per item
  int G, TS;             // positions per pooled group; tile stride in positions (multiple of G, <= 256)
  int tiles_per_item, m_blocks, units;
  int relu;
  const float* residual; // optional [B, M, P]: added after the activation (transformer sublayers: x + f(norm(x)))
  const float* col_div;  // optional [B, P]: every output column p is divided by col_div[b, p] (attention: p.v / row sum)
  int out_t;             // linear layers: h_out is written transposed, [B, P, M] (v^T for the attention p.v product)
  int w4, x4;            // chunked 4-D tensor maps: weights; activations (bit 0: tiles at 32-position multiples, bit 1: +16)
  int w_heads;           // 0: one weight matrix for every item.  h > 0: item b uses rows (b % h)*M.. of weight batch b / h
};

struct EdgeShared {
  uint64_t tma_full[EC_MAX_STAGES];
  uint64_t full[EC_MAX_STAGES];
  uint64_t empty[EC_MAX_STAGES];
  uint64_t acc_full[2];
  uint64_t acc_empty[2];
  uint32_t tmem_base;
  // per-epilogue-warp 32 x 32 transpose tile for the h_out stores, XOR-swizzled 16-byte chunks (no padding);
  // the generic-G pooling path keeps a thread's <= 16 pooled values of the current tile in its own row
  alignas(16) float tbuf[EC_EPI_GROUPS * EC_EPI_THREADS / 32][32][32];
};
// tile stride (owned positions per tile) for a group size G: whole groups only, at most EC_MAX_GROUPS of them
__host__ __device__ constexpr int edge_tile_stride(int G) {
  return G * ((EC_BN / G) < EC_MAX_GROUPS ? (EC_BN / G) : EC_MAX_GROUPS);
}

__device__ int g_edgeconv_error = 0;

struct EdgeUnit { int b, j0, m0; };
__device__ __forceinline__ EdgeUnit edge_unit(const EdgeParams& p, int u, int ctas, uint32_t crank) {
  EdgeUnit r;
  const int mb = u % p.m_blocks, q = u / p.m_blocks;
  const int jt = q % p.tiles_per_item;
  r.b = q / p.tiles_per_item;
  r.j0 = jt * p.TS;
  r.m0 = mb * (SC_BM * ctas) + (int)crank * SC_BM;
  return r;
}

// GT: compile-time pooling group size for the epilogue's fast path (20 = DGCNN's k; 1 = the generic path only)
int tma3_boxes_forced();   // softcorr.cu: testing hook (l3d_debug_soft_correspondence_force_generic(3))

template <int CTAS, int GT>
__global__ void __launch_bounds__(EC_THREADS, 1)
edge_gemm_kernel(const EdgeParams p, const __grid_constant__ CUtensorMap tmap_w,
                 const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_x4a,
                 const __grid_constant__ CUtensorMap tmap_x4b) {
  using Cfg = EdgeCfg<CTAS>;
  constexpr int STAGES = Cfg::STAGES, STAGE_BYTES = Cfg::STAGE, A_TILE = Cfg::A_TILE, B_TILE = Cfg::B_TILE;
  constexpr bool PAIR = (CTAS == 2);
  const uint32_t crank = PAIR ? cluster_ctarank() : 0u;
  extern __shared__ unsigned char ec_raw[];
  unsigned char* tiles = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(ec_raw) + 1023) & ~(uintptr_t)1023);
  EdgeShared* sh = reinterpret_cast<EdgeShared*>(tiles + STAGES * STAGE_BYTES);
  const uint32_t tiles_s = smem_u32(tiles);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int cluster_id = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int n_clusters = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  const int my_tiles = (p.units > cluster_id) ? (p.units - cluster_id + n_clusters - 1) / n_clusters : 0;
  const int num_kb = (p.K + EC_BK - 1) / EC_BK;
  const int total = my_tiles * num_kb;

  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&sh->tma_full[s], 1);
      mbar_init(&sh->full[s], EC_SPLIT_THREADS / 32 * CTAS);
      mbar_init(&sh->empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) { mbar_init(&sh->acc_full[a], 1); mbar_init(&sh->acc_empty[a], EC_EPI_THREADS / 32 * CTAS); }
    fence_mbar_init();
  }
  if (warp == 0) {
    if (PAIR) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&sh->tmem_base)),
                   "n"(Cfg::TMEM_COLS) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&sh->tmem_base)),
                   "n"(Cfg::TMEM_COLS) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem = sh->tmem_base;

  if (warp < 4 || warp >= 10) {
    // ------------------------------------------------ epilogue: BN + ReLU, max over groups of G positions, stores
    // two groups of four warps: group g drains accumulator g, i.e. the tiles t = g, g+2, ... of this CTA
    const int grp = warp < 4 ? 0 : 1;
    const int w4 = warp & 3;                        // TMEM lane quarter this warp may read (warp id % 4)
    const int row = w4 * 32 + lane;                 // accumulator lane = output channel within the block
    float(*tb)[32] = sh->tbuf[grp * 4 + w4];
    const float qnan = __int_as_float(0x7fc00000);
    bool ok = true;
    for (int t = grp; t < my_tiles; t += EC_EPI_GROUPS) {
      const EdgeUnit un = edge_unit(p, cluster_id + t * n_clusters, CTAS, crank);
      const int a = grp;
      const int c = un.m0 + row;                    // this thread's output channel
      const bool vrow = c < p.M;
      const int nvalid = min(p.TS, p.P - un.j0);    // positions this tile owns
      const bool vec = ((p.P & 3) == 0) && ((un.j0 & 3) == 0) && ((nvalid & 3) == 0);
      if (ok && !mbar_wait_bounded(&sh->acc_full[a], (uint32_t)((t >> 1) & 1))) {
        ok = false;
        atomicCAS(p.err, 0, 1);
      }
      if (!ok) {
        // the pipeline is dead: everything this thread still owed becomes NaN so that no caller mistakes
        // uninitialised memory for a result
        if (vrow) {
          if (p.h_out) {
            float* dst = p.h_out + ((size_t)un.b * p.M + c) * p.P + un.j0;
            for (int e = 0; e < nvalid; ++e) dst[e] = qnan;
          }
          if (p.pool_out) {
            float* dst = p.pool_out + (size_t)un.b * p.pool_bstride + (size_t)(p.pool_coff + c) * p.pool_n + un.j0 / p.G;
            for (int g = 0; g < nvalid / p.G; ++g) dst[g] = qnan;
          }
        }
        continue;
      }
      __syncwarp();
      tc_fence_after();
      const float s = vrow ? (p.scale ? __ldg(p.scale + c) : 1.f) : 0.f, sf = (vrow && p.shift) ? __ldg(p.shift + c) : 0.f;
      const uint32_t tacc = tmem + ((uint32_t)(w4 * 32) << 16) + (uint32_t)(a * EC_BN);
      float* pdst = p.pool_out ? p.pool_out + (size_t)un.b * p.pool_bstride + (size_t)(p.pool_coff + c) * p.pool_n + un.j0 / p.G
                               : nullptr;
      // one 32-column chunk: folded BN (+ ReLU) in place, and the transposed, coalesced h_out store
      auto chunk = [&](int ch, float (&v)[32], int nv) {
        tc_ld32(tacc + (uint32_t)(ch * 32), v);
#pragma unroll
        for (int e = 0; e < 32; ++e) {
          const float y = fmaf(v[e], s, sf);
          v[e] = p.relu ? fmaxf(y, 0.f) : y;
        }
        if (GT == 1 && p.col_div) {          // linear layers only: keeps the pooled kernels' epilogue free of it
          const float* cd = p.col_div + (size_t)un.b * p.P + un.j0 + ch * 32;      // same address in every lane
#pragma unroll
          for (int e = 0; e < 32; ++e)
            if (e < nv) v[e] = __fdividef(v[e], __ldg(cd + e));
        }
        if (!p.h_out) return;
        if (GT == 1 && p.out_t) {
          // [B, P, M]: for a fixed position the 32 lanes (consecutive channels) write one 128-byte line
          if (vrow) {
            float* dst = p.h_out + ((size_t)un.b * p.P + un.j0 + ch * 32) * p.M + c;
#pragma unroll
            for (int e = 0; e < 32; ++e)
              if (e < nv) dst[(size_t)e * p.M] = v[e];
          }
          return;
        }
        if (vec) {
          // transpose the warp's 32 x 32 block through shared memory (16-byte chunk q of row r lives at chunk
          // q ^ (r & 7): conflict-free both ways): every store instruction then writes four 128-byte lines
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<float4*>(&tb[lane][((q ^ (lane & 7)) << 2)]) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
          __syncwarp();
          const int rr = lane >> 3, cq = lane & 7;
          const int cbase = un.m0 + w4 * 32;
#pragma unroll
          for (int r = 0; r < 32; r += 4) {
            float4 o = *reinterpret_cast<const float4*>(&tb[r + rr][((cq ^ ((r + rr) & 7)) << 2)]);
            const int cr = cbase + r + rr;
            if (cr < p.M && cq * 4 < nv) {
              const size_t off = ((size_t)un.b * p.M + cr) * p.P + un.j0 + ch * 32 + cq * 4;
              if (GT == 1 && p.residual) {
                const float4 rz = __ldg(reinterpret_cast<const float4*>(p.residual + off));
                o.x += rz.x; o.y += rz.y; o.z += rz.z; o.w += rz.w;
              }
              *reinterpret_cast<float4*>(p.h_out + off) = o;
            }
          }
          __syncwarp();
        } else if (vrow) {
          const size_t off = ((size_t)un.b * p.M + c) * p.P + un.j0 + ch * 32;
#pragma unroll
          for (int e = 0; e < 32; ++e)
            if (e < nv) p.h_out[off + e] = (GT == 1 && p.residual) ? v[e] + __ldg(p.residual + off + e) : v[e];
        }
      };
      auto release = [&]() {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (PAIR) mbar_arrive_cluster(&sh->acc_empty[a], 0);
          else mbar_arrive(&sh->acc_empty[a]);
        }
      };
      if (un.m0 + w4 * 32 >= p.M) {
        // none of this warp's 32 accumulator lanes is an output channel (C_out = 64 fills half of the 128 lanes):
        // nothing to read or store, only the accumulator hand-back
        release();
        continue;
      }
      if (GT > 1 && nvalid == edge_tile_stride(GT > 1 ? GT : 2)) {
        // full tile, compile-time group size: every index below is static after unrolling — the pooled maxima
        // live in registers, the max chains of different groups are independent (ILP), no branches
        constexpr int TSS = edge_tile_stride(GT > 1 ? GT : 2);
        constexpr int NG = TSS / (GT > 1 ? GT : 2);
        float pool[NG];
#pragma unroll
        for (int g = 0; g < NG; ++g) pool[g] = -INFINITY;
#pragma unroll
        for (int ch = 0; ch < (TSS + 31) / 32; ++ch) {
          float v[32];
          chunk(ch, v, (TSS - ch * 32) < 32 ? (TSS - ch * 32) : 32);
          if (pdst) {
#pragma unroll
            for (int e = 0; e < 32; ++e)
              if (ch * 32 + e < TSS) pool[(ch * 32 + e) / (GT > 1 ? GT : 2)] = fmaxf(pool[(ch * 32 + e) / (GT > 1 ? GT : 2)], v[e]);
          }
        }
        release();
        if (pdst && vrow) {
#pragma unroll
          for (int g = 0; g < NG; ++g) pdst[g] = pool[g];
        }
      } else {
        // generic: run-time group size and / or a short last tile
        float gm = -INFINITY;
        int cnt = 0, gi = 0;
        // a kernel with a compile-time group size only comes here for a short last tile: fewer than EC_BN / GT groups
        constexpr int PLN = GT > 1 ? EC_BN / GT : EC_MAX_GROUPS;
        float pl[PLN];
#pragma unroll
        for (int g = 0; g < PLN; ++g) pl[g] = 0.f;
#pragma unroll 1
        for (int ch = 0; ch < EC_BN / 32; ++ch) {
          if (ch * 32 >= nvalid) break;
          float v[32];
          const int nv = min(32, nvalid - ch * 32);
          chunk(ch, v, nv);
          if (pdst) {
#pragma unroll
            for (int e = 0; e < 32; ++e) {
              if (e < nv) {
                gm = fmaxf(gm, v[e]);
                if (++cnt == p.G) {
#pragma unroll
                  for (int g = 0; g < PLN; ++g) if (g == gi) pl[g] = gm;
                  ++gi; gm = -INFINITY; cnt = 0;
                }
              }
            }
          }
        }
        release();
        if (pdst && vrow) {
#pragma unroll
          for (int g = 0; g < PLN; ++g) if (g < gi) pdst[g] = pl[g];
        }
      }
    }
  } else if (warp < 8) {
    // ------------------------------------------------ splitters: lo = tf32(x - trunc_tf32(x)), smem -> smem
    const int r = tid - EC_EPI_THREADS;
    bool ok = true;
    for (int it = 0; it < total; ++it) {
      const int s = it % STAGES;
      const uint32_t n = (uint32_t)(it / STAGES);
      const uint32_t st = tiles_s + s * STAGE_BYTES;
      if (!mbar_wait_bounded(&sh->tma_full[s], n & 1u)) { ok = false; break; }
#pragma unroll
      for (int op = 0; op < 2; ++op) {
        const uint32_t hi = st + (op ? 2 * A_TILE : 0), lo = hi + (op ? B_TILE : A_TILE);
#pragma unroll
        for (int q = 0; q < (op ? B_TILE : A_TILE) / 16 / EC_SPLIT_THREADS; ++q) {
          const uint32_t off = (uint32_t)(q * EC_SPLIT_THREADS + r) * 16u;
          const uint4 x = lds128(hi + off);
          uint4 y;
          y.x = rna_tf32_bits(__float_as_uint(__fsub_rn(__uint_as_float(x.x), __uint_as_float(x.x & 0xffffe000u))));
          y.y = rna_tf32_bits(__float_as_uint(__fsub_rn(__uint_as_float(x.y), __uint_as_float(x.y & 0xffffe000u))));
          y.z = rna_tf32_bits(__float_as_uint(__fsub_rn(__uint_as_float(x.z), __uint_as_float(x.z & 0xffffe000u))));
          y.w = rna_tf32_bits(__float_as_uint(__fsub_rn(__uint_as_float(x.w), __uint_as_float(x.w & 0xffffe000u))));
          sts128(lo + off, y);
        }
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) {
        if (PAIR) mbar_arrive_cluster(&sh->full[s], 0);
        else mbar_arrive(&sh->full[s]);
      }
    }
    if (!ok) atomicCAS(p.err, 0, 2);
  } else if (warp == 8) {
    // ------------------------------------------------ MMA issuer (rank 0 of a pair issues for both CTAs)
    bool ok = true;
    int it = 0;
    for (int t = 0; t < my_tiles && ok && crank == 0; ++t) {
      const int a = t & 1;
      const uint32_t pe = (uint32_t)(((t >> 1) & 1) ^ 1);
      if (!(PAIR ? mbar_wait_bounded_cluster(&sh->acc_empty[a], pe) : mbar_wait_bounded(&sh->acc_empty[a], pe))) { ok = false; break; }
      tc_fence_after();
      const uint32_t d_tmem = tmem + (uint32_t)(a * EC_BN);
      for (int kb = 0; kb < num_kb; ++kb, ++it) {
        const int s = it % STAGES;
        const uint32_t n = (uint32_t)(it / STAGES);
        if (!(PAIR ? mbar_wait_bounded_cluster(&sh->full[s], n & 1u) : mbar_wait_bounded(&sh->full[s], n & 1u))) { ok = false; break; }
        tc_fence_after();
        if (lane == 0) {
          const uint32_t sa = tiles_s + s * STAGE_BYTES;
          // MN-major tf32 operands: UMMA layout 1 (128 B swizzle, 32-byte atoms): 4-channel groups 512 B apart,
          // the next 32 rows / columns one TMA box (ATOM bytes) further
          constexpr uint32_t lbo = (uint32_t)Cfg::ATOM, sbo = 512u, lay = 1u;
          constexpr uint32_t idesc = sc_idesc(EC_BN, true, SC_BM * CTAS);
          const uint64_t a_hi = sc_desc(sa, lbo, sbo, lay), a_lo = sc_desc(sa + A_TILE, lbo, sbo, lay);
          const uint64_t b_hi = sc_desc(sa + 2 * A_TILE, lbo, sbo, lay), b_lo = sc_desc(sa + 2 * A_TILE + B_TILE, lbo, sbo, lay);
#pragma unroll
          for (int k = 0; k < EC_BK / SC_UK; ++k) {
            const uint64_t adv = (uint64_t)((k * 1024) >> 4);     // next 8-channel group
            if (PAIR) {
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
            tc_commit_pair(&sh->empty[s]);
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
  } else {
    // ------------------------------------------------ TMA issuer: 4 weight boxes + 8 (4 in a pair) activation boxes
    bool ok = true;
    int it = 0;
    // Tried and rejected (profiles/r02/README.md): prefetching the activation boxes 12 stages beyond the ring into L2
    // (UTMAPF.L2).  The prefetches queue in the same TMA pipe ahead of the ring's own loads and made every layer
    // slower (layer 2: 108 -> 183 us, p.v: 188 -> 310 us).  The experiment was removed; its code is in git history
    // before the change that removed it.
    for (int t = 0; t < my_tiles && ok; ++t) {
      const EdgeUnit un = edge_unit(p, cluster_id + t * n_clusters, CTAS, crank);
      for (int kb = 0; kb < num_kb; ++kb, ++it) {
        const int s = it % STAGES;
        const uint32_t n = (uint32_t)(it / STAGES);
        if (!mbar_wait_bounded(&sh->empty[s], (n & 1u) ^ 1u)) { ok = false; break; }
        if (lane == 0) {
          const uint32_t st = tiles_s + s * STAGE_BYTES;
          mbar_arrive_expect_tx(&sh->tma_full[s], A_TILE + B_TILE);
          const int wm0 = un.m0 + (p.w_heads ? (un.b % p.w_heads) * p.M : 0), wb = p.w_heads ? un.b / p.w_heads : 0;
          // chunked 4-D maps (tc05.cuh: make_dn_tmap4): a whole operand tile per instruction.  The activation tile
          // starts at a multiple of 32 positions (map a) or 16 past one (map b, base shifted by 16 floats: k = 20 tiles
          // advance by 240); a shifted tile that would run past the row takes the 32-point boxes, which zero-fill.
          if (p.w4) {
            tma_load_4d(st, &tmap_w, 0, kb * EC_BK, wm0 / 32, wb, &sh->tma_full[s]);
          } else {
#pragma unroll
            for (int q = 0; q < SC_BM / 32; ++q)
              tma_load_3d(st + q * Cfg::ATOM, &tmap_w, wm0 + 32 * q, kb * EC_BK, wb, &sh->tma_full[s]);
          }
          const int jl = un.j0 + (int)crank * Cfg::BN_LOCAL;
          if ((p.x4 & 1) && (jl & 31) == 0) {
            tma_load_4d(st + 2 * A_TILE, &tmap_x4a, 0, kb * EC_BK, jl / 32, un.b, &sh->tma_full[s]);
          } else if ((p.x4 & 2) && (jl & 31) == 16 && jl + Cfg::BN_LOCAL <= p.P) {
            tma_load_4d(st + 2 * A_TILE, &tmap_x4b, 0, kb * EC_BK, jl / 32, un.b, &sh->tma_full[s]);
          } else {
#pragma unroll
            for (int q = 0; q < Cfg::BN_LOCAL / 32; ++q)
              tma_load_3d(st + 2 * A_TILE + q * Cfg::ATOM, &tmap_x, jl + 32 * q, kb * EC_BK, un.b, &sh->tma_full[s]);
          }
        }
        __syncwarp();
      }
    }
    if (!ok && lane == 0) atomicCAS(p.err, 0, 4);
  }

  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();
  if (warp == 0) {
    tc_fence_after();
    if (PAIR)
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(Cfg::TMEM_COLS) : "memory");
    else
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(Cfg::TMEM_COLS) : "memory");
  }
}

template <int CTAS>
static size_t edge_smem_bytes() {
  return (size_t)EdgeCfg<CTAS>::STAGES * EdgeCfg<CTAS>::STAGE + sizeof(EdgeShared) + 1024;
}

// ---- layer 1: conv(6 -> C1) + BN + ReLU straight from the kNN indices (gather-on-load) ------------------------
// h1[b, c, n*k + j] = relu(scale_c * (W[c,0:3] . x[idx[b,n,j]] + W[c,3:6] . x[n]) + shift_c)
// (get_graph_feature's channel order: neighbour xyz, then centre xyz — model_common_utils.py:149-154).
// Weights travel as a kernel parameter (constant bank): every FFMA reads its weight as an immediate-like operand.
constexpr int EC_C1 = 64;
struct EdgeL1Weights {
  float w[EC_C1 * 6];
  float scale[EC_C1];
  float shift[EC_C1];
};

__device__ __forceinline__ float edge_l1_value(const EdgeL1Weights& W, int c, float nx, float ny, float nz, float cx,
                                               float cy, float cz) {
  float v = __fmul_rn(W.w[c * 6 + 0], nx);
  v = fmaf(W.w[c * 6 + 1], ny, v);
  v = fmaf(W.w[c * 6 + 2], nz, v);
  v = fmaf(W.w[c * 6 + 3], cx, v);
  v = fmaf(W.w[c * 6 + 4], cy, v);
  v = fmaf(W.w[c * 6 + 5], cz, v);
  return fmaxf(fmaf(v, W.scale[c], W.shift[c]), 0.f);
}

// thread = position (n, j): 64 coalesced stores
__global__ void __launch_bounds__(256) edge_l1_kernel(const __grid_constant__ EdgeL1Weights W, const float* __restrict__ x,
                                                      const long long* __restrict__ idx, int N, int k,
                                                      float* __restrict__ h1) {
  const int b = blockIdx.y;
  const long P = (long)N * k;
  const long pos = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (pos >= P) return;
  const int n = (int)(pos / k);
  const float* xb = x + (size_t)b * 3 * N;
  long j = idx[(size_t)b * P + pos];
  if ((unsigned long)j >= (unsigned long)N) j = n;            // never produced by l3d_knn_*; keeps the loads in bounds
  const float nx = __ldg(xb + j), ny = __ldg(xb + N + j), nz = __ldg(xb + 2 * (size_t)N + j);
  const float cx = __ldg(xb + n), cy = __ldg(xb + N + n), cz = __ldg(xb + 2 * (size_t)N + n);
  float* o = h1 + (size_t)b * EC_C1 * P + pos;
#pragma unroll
  for (int c = 0; c < EC_C1; ++c) o[(size_t)c * P] = edge_l1_value(W, c, nx, ny, nz, cx, cy, cz);
}

// thread = (point n, quarter of the channels): max over the point's k neighbours of the same expression
// (bit-identical values), coalesced over n.  32 points x 4 channel quarters per CTA.
constexpr int EC_L1P_Q = 4;
__global__ void __launch_bounds__(32 * EC_L1P_Q) edge_l1_pool_kernel(const __grid_constant__ EdgeL1Weights W,
                                                                     const float* __restrict__ x, const long long* __restrict__ idx,
                                                                     int N, int k, float* __restrict__ pool, long pool_bstride,
                                                                     int pool_coff) {
  constexpr int CQ = EC_C1 / EC_L1P_Q;
  const int b = blockIdx.y;
  const int n = blockIdx.x * 32 + (threadIdx.x & 31);
  const int cq = threadIdx.x >> 5;
  if (n >= N) return;
  const float* xb = x + (size_t)b * 3 * N;
  const float cx = __ldg(xb + n), cy = __ldg(xb + N + n), cz = __ldg(xb + 2 * (size_t)N + n);
  float m[CQ];
#pragma unroll
  for (int c = 0; c < CQ; ++c) m[c] = 0.f;                      // values are >= 0 after the ReLU
  const long long* ip = idx + ((size_t)b * N + n) * k;
  for (int jj = 0; jj < k; ++jj) {
    long j = ip[jj];
    if ((unsigned long)j >= (unsigned long)N) j = n;
    const float nx = __ldg(xb + j), ny = __ldg(xb + N + j), nz = __ldg(xb + 2 * (size_t)N + j);
#pragma unroll
    for (int q = 0; q < EC_L1P_Q; ++q) {
      if (q == cq) {                                             // warp-uniform: weights stay constant-bank operands
#pragma unroll
        for (int c = 0; c < CQ; ++c) m[c] = fmaxf(m[c], edge_l1_value(W, q * CQ + c, nx, ny, nz, cx, cy, cz));
      }
    }
  }
  float* o = pool + (size_t)b * pool_bstride + (size_t)(pool_coff + cq * CQ) * N + n;
#pragma unroll
  for (int c = 0; c < CQ; ++c) o[(size_t)c * N] = m[c];
}

}  // namespace l3d

using namespace l3d;

extern "C" int l3d_edgeconv_layer1(const float* x_dev, const int64_t* idx_dev, const float* w_host,
                                   const float* scale_host, const float* shift_host, int B, int N, int k, int C1,
                                   float* h1_dev, float* pool_dev, long long pool_bstride, int pool_coff,
                                   void* stream) {
  if (B < 0 || N < 1 || k < 1 || k > N) return L3D_ERR_INVALID;
  if (C1 != EC_C1) return L3D_ERR_UNSUPPORTED;
  if (B == 0) return L3D_OK;
  if (!x_dev || !idx_dev || !w_host || !scale_host || !shift_host || (!h1_dev && !pool_dev) || B > 65535)
    return L3D_ERR_INVALID;
  EdgeL1Weights W;
  memcpy(W.w, w_host, sizeof(W.w));
  memcpy(W.scale, scale_host, sizeof(W.scale));
  memcpy(W.shift, shift_host, sizeof(W.shift));
  const long P = (long)N * k;
  if (h1_dev) {
    edge_l1_kernel<<<dim3((unsigned)((P + 255) / 256), B), 256, 0, (cudaStream_t)stream>>>(
        W, x_dev, reinterpret_cast<const long long*>(idx_dev), N, k, h1_dev);
    count_launch();
    L3D_LAUNCH_CHECK();
  }
  if (pool_dev) {
    edge_l1_pool_kernel<<<dim3((unsigned)((N + 31) / 32), B), 32 * EC_L1P_Q, 0, (cudaStream_t)stream>>>(
        W, x_dev, reinterpret_cast<const long long*>(idx_dev), N, k, pool_dev, (long)pool_bstride, pool_coff);
    count_launch();
    L3D_LAUNCH_CHECK();
  }
  return L3D_OK;
}

// relu(scale * (W . X) + shift) for X [B, K, P], W^T [K, M]; optional full output h_out [B, M, P] and optional max
// over every group of G consecutive positions -> pool_out[b*pool_bstride + (pool_coff + c)*(P/G) + n].
template <int GT>
static cudaError_t edge_set_attrs_gt(int dev) {
  cudaError_t e = raise_smem_once<edge_gemm_kernel<1, GT>>(dev, edge_smem_bytes<1>());
  if (e != cudaSuccess) return e;
  return raise_smem_once<edge_gemm_kernel<2, GT>>(dev, edge_smem_bytes<2>());
}
static cudaError_t edge_set_attrs(int dev) {
  cudaError_t e = edge_set_attrs_gt<1>(dev);
  if (e == cudaSuccess) e = edge_set_attrs_gt<20>(dev);
  if (e == cudaSuccess) e = edge_set_attrs_gt<16>(dev);
  if (e == cudaSuccess) e = edge_set_attrs_gt<8>(dev);
  if (e == cudaSuccess) e = edge_set_attrs_gt<64>(dev);
  return e;
}

static int edge_gemm_launch(const float* wt_dev, const float* x_dev, const float* scale_dev, const float* shift_dev,
                            const float* residual_dev, const float* col_div_dev, int w_heads, int B, int M, int K, int P,
                            int G, int relu,
                            float* h_out_dev, float* pool_out_dev, long long pool_bstride, int pool_coff,
                            void* stream) {
  if (B < 0 || M < 1 || K < 1 || P < 1 || G < 1) return L3D_ERR_INVALID;
  if (B == 0) return L3D_OK;
  if (!wt_dev || !x_dev || (!h_out_dev && !pool_out_dev) || w_heads < 0) return L3D_ERR_INVALID;
  if (w_heads > 0 && (M % SC_BM != 0 || B % w_heads != 0)) return L3D_ERR_UNSUPPORTED;   // whole 128-row blocks per head
  if (pool_out_dev && (P % G != 0 || G > EC_BN)) return L3D_ERR_INVALID;
  // TMA: 16-byte global strides and bases
  if ((P & 3) || (M & 3) || ((((uintptr_t)wt_dev) | ((uintptr_t)x_dev)) & 15)) return L3D_ERR_UNSUPPORTED;
  if (B > 65535) return L3D_ERR_UNSUPPORTED;
  EdgeParams p;
  memset(&p, 0, sizeof(p));
  p.scale = scale_dev; p.shift = shift_dev; p.h_out = h_out_dev; p.pool_out = pool_out_dev;
  p.pool_bstride = (long)pool_bstride; p.pool_coff = pool_coff;
  p.B = B; p.M = M; p.K = K; p.P = P; p.G = G; p.relu = relu & 1; p.out_t = (relu >> 1) & 1;   // bit 1: transposed output
  p.residual = residual_dev; p.w_heads = w_heads; p.col_div = col_div_dev;
  if (pool_out_dev) {
    p.TS = edge_tile_stride(G);
    p.pool_n = P / G;
  } else {
    p.TS = EC_BN;
    p.pool_n = 0;
  }
  const bool pair = M > SC_BM;
  p.tiles_per_item = (P + p.TS - 1) / p.TS;
  p.m_blocks = (M + (pair ? 2 : 1) * SC_BM - 1) / ((pair ? 2 : 1) * SC_BM);
  const long units = (long)B * p.tiles_per_item * p.m_blocks;
  if (units > 0x7fffffffL) return L3D_ERR_UNSUPPORTED;
  p.units = (int)units;

  int dev = 0;
  cudaGetDevice(&dev);
  {
    const cudaError_t e = edge_set_attrs(dev);
    if (e != cudaSuccess) return (int)e;
  }
  void* errp = nullptr;
  cudaError_t e = cudaGetSymbolAddress(&errp, g_edgeconv_error);
  if (e != cudaSuccess) return (int)e;
  p.err = (int*)errp;

  CUtensorMap mw, mx;
  memset(&mw, 0, sizeof(mw)); memset(&mx, 0, sizeof(mx));
  // weights: [K, M] shared by every item, or (w_heads > 0) [B / w_heads, K, w_heads * M] with one head per item
  const bool wok = w_heads ? make_dn_tmap(&mw, wt_dev, B / w_heads, K, w_heads * M, EC_BK) : make_dn_tmap(&mw, wt_dev, 1, K, M, EC_BK);
  if (!wok || !make_dn_tmap(&mx, x_dev, B, K, P, EC_BK)) return L3D_ERR_UNSUPPORTED;
  CUtensorMap mx4a, mx4b;
  memset(&mx4a, 0, sizeof(mx4a)); memset(&mx4b, 0, sizeof(mx4b));
  if (!tma3_boxes_forced()) {
    const int xchunks = (pair ? EdgeCfg<2>::BN_LOCAL : EdgeCfg<1>::BN_LOCAL) / 32;
    CUtensorMap mw4;
    const bool w4 = w_heads ? make_dn_tmap4(&mw4, wt_dev, B / w_heads, K, w_heads * M, EC_BK, SC_BM / 32)
                            : make_dn_tmap4(&mw4, wt_dev, 1, K, M, EC_BK, SC_BM / 32);
    if (w4) { mw = mw4; p.w4 = 1; }
    const int step = p.TS & 31;                                  // tile starts modulo 32: always 0, or alternating 0 / 16
    if ((step == 0 || step == 16) && (P & 31) == 0) {
      if (make_dn_tmap4(&mx4a, x_dev, B, K, P, EC_BK, xchunks)) p.x4 |= 1;
      // the +16 view: same strides from a base 16 floats in; only chunks that lie wholly inside a row are declared
      if (step == 16 && P >= 64) {
        EncodeTiledFn fn = encode_tiled_fn();
        cuuint64_t dims[4] = {32, (cuuint64_t)K, (cuuint64_t)((P - 16) / 32), (cuuint64_t)B};
        cuuint64_t strides[3] = {(cuuint64_t)P * 4, 128, (cuuint64_t)P * (cuuint64_t)K * 4};
        cuuint32_t box[4] = {32, (cuuint32_t)EC_BK, (cuuint32_t)xchunks, 1};
        cuuint32_t estr[4] = {1, 1, 1, 1};
        if (fn && fn(&mx4b, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (void*)(x_dev + 16), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS)
          p.x4 |= 2;
      }
    }
  }

  const int sms = sm_count(dev);
  // (the compile-time-G kernels carry no residual / column-divide code)
  const int gt = (pool_out_dev != nullptr && !residual_dev && !col_div_dev && (G == 20 || G == 16 || G == 8 || G == 64)) ? G : 1;
  if (pair) {
    long clusters = sms / 2;
    if (clusters > units) clusters = units;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(2 * clusters));
    cfg.blockDim = dim3(EC_THREADS);
    cfg.dynamicSmemBytes = edge_smem_bytes<2>();
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    // group sizes with a compile-time epilogue (static group boundaries): DGCNN's k = 20, FlowNet3D's 8 / 16 / 64
    cudaError_t le;
    switch (gt) {
      case 20: le = cudaLaunchKernelEx(&cfg, edge_gemm_kernel<2, 20>, p, mw, mx, mx4a, mx4b); break;
      case 16: le = cudaLaunchKernelEx(&cfg, edge_gemm_kernel<2, 16>, p, mw, mx, mx4a, mx4b); break;
      case 8: le = cudaLaunchKernelEx(&cfg, edge_gemm_kernel<2, 8>, p, mw, mx, mx4a, mx4b); break;
      case 64: le = cudaLaunchKernelEx(&cfg, edge_gemm_kernel<2, 64>, p, mw, mx, mx4a, mx4b); break;
      default: le = cudaLaunchKernelEx(&cfg, edge_gemm_kernel<2, 1>, p, mw, mx, mx4a, mx4b);
    }
    if (le != cudaSuccess) return (int)le;
  } else {
    long grid = sms;
    if (grid > units) grid = units;
    const size_t sm1 = edge_smem_bytes<1>();
    cudaStream_t st = (cudaStream_t)stream;
    switch (gt) {
      case 20: edge_gemm_kernel<1, 20><<<(unsigned)grid, EC_THREADS, sm1, st>>>(p, mw, mx, mx4a, mx4b); break;
      case 16: edge_gemm_kernel<1, 16><<<(unsigned)grid, EC_THREADS, sm1, st>>>(p, mw, mx, mx4a, mx4b); break;
      case 8: edge_gemm_kernel<1, 8><<<(unsigned)grid, EC_THREADS, sm1, st>>>(p, mw, mx, mx4a, mx4b); break;
      case 64: edge_gemm_kernel<1, 64><<<(unsigned)grid, EC_THREADS, sm1, st>>>(p, mw, mx, mx4a, mx4b); break;
      default: edge_gemm_kernel<1, 1><<<(unsigned)grid, EC_THREADS, sm1, st>>>(p, mw, mx, mx4a, mx4b);
    }
  }
  count_launch();
  L3D_LAUNCH_CHECK();
  return L3D_OK;
}

extern "C" int l3d_conv1x1_bn_relu_maxk(const float* wt_dev, const float* x_dev, const float* scale_dev,
                                        const float* shift_dev, int B, int M, int K, int P, int G, int relu,
                                        float* h_out_dev, float* pool_out_dev, long long pool_bstride, int pool_coff,
                                        void* stream) {
  if (!scale_dev) return L3D_ERR_INVALID;
  return edge_gemm_launch(wt_dev, x_dev, scale_dev, shift_dev, nullptr, nullptr, 0, B, M, K, P, G, relu ? 1 : 0, h_out_dev,
                          pool_out_dev, pool_bstride, pool_coff, stream);
}

// Channel-major linear layer  out[b, m, p] = act(sum_k wt[.., k, m] x[b, k, p] + bias[m]) (+ residual[b, m, p])
// on the same tcgen05 pipeline (the transformer's nn.Linear layers with activations kept as [B, d_model, N]).
// w_heads = 0: wt_dev [K, M] shared by all items.  w_heads = h > 0 ("one head per item", the P.V product of
// attention): x_dev has B = batch*h items, wt_dev is [batch, K, h*M] and item b uses columns (b % h)*M.. of weight
// batch b / h; M must be a multiple of 128.
// col_div_dev (optional, [B, P]): every output column is divided by it — the attention row sums when x_dev holds
// unnormalised probabilities.
extern "C" int l3d_linear_cm(const float* wt_dev, const float* x_dev, const float* bias_dev, const float* residual_dev,
                             const float* col_div_dev, int B, int M, int K, int P, int relu, int w_heads,
                             float* out_dev, void* stream) {
  if (!out_dev) return L3D_ERR_INVALID;
  if ((M * w_heads) & 3) return L3D_ERR_UNSUPPORTED;
  return edge_gemm_launch(wt_dev, x_dev, nullptr, bias_dev, residual_dev, col_div_dev, w_heads, B, M, K, P, 1, relu ? 1 : 0,
                          out_dev, nullptr, 0, 0, stream);
}

// l3d_linear_cm with the output written transposed: out_dev [B, P, M] (positions major).  The attention value
// projection uses it to produce v^T [B, N_k, h * d_v] — the per-head weight operand of the p.v product — without a
// separate transpose pass.  No residual / column divide on this form.
extern "C" int l3d_linear_cm_t(const float* wt_dev, const float* x_dev, const float* bias_dev, int B, int M, int K, int P,
                               int relu, float* out_dev, void* stream) {
  if (!out_dev) return L3D_ERR_INVALID;
  return edge_gemm_launch(wt_dev, x_dev, nullptr, bias_dev, nullptr, nullptr, 0, B, M, K, P, 1, (relu ? 1 : 0) | 2, out_dev,
                          nullptr, 0, 0, stream);
}

// Synchronises the device and returns (then clears) the pipeline error word of l3d_conv1x1_bn_relu_maxk:
// 0 = ok; 1/2/3/4 = an epilogue / splitter / MMA-issuer / TMA-issuer wait ran out (outputs were set to NaN).
extern "C" int l3d_edgeconv_status(void) {
  int v = 0;
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) return (int)e;
  e = cudaMemcpyFromSymbol(&v, g_edgeconv_error, sizeof(int));
  if (e != cudaSuccess) return (int)e;
  if (v != 0) {
    const int zero = 0;
    cudaMemcpyToSymbol(g_edgeconv_error, &zero, sizeof(int));
  }
  return v;
}
