// In-register sorting networks and the 62-bit (key, index) composites of the thread-per-row selections
// (knn_tpr.cu: knn() on xyz clouds).
#pragma once
#include "common.cuh"

namespace l3d {

// ---- in-register sorting networks (every index is a compile-time constant after unrolling) ----------------
// cex(x, y) is the compare-exchange: the larger element ends in x.  cex_f32 for group maxima, tpr_cex for the
// composites below.
// Sorting network: Batcher's merge exchange (Knuth 5.2.2 M) — 191 exchanges for 32 keys against 240 for the
// bitonic sorter; the larger key ends at the lower index.
template <int N, typename T, typename Cex>
__device__ __forceinline__ void reg_sort_desc(T (&a)[N], Cex cex) {
#pragma unroll
  for (int p = N / 2; p >= 1; p >>= 1) {
#pragma unroll
    for (int i = 0; i < N - p; ++i)
      if ((i & p) == 0) cex(a[i], a[i + p]);
#pragma unroll
    for (int q = N / 2; q > p; q >>= 1) {
      const int d = q - p;
#pragma unroll
      for (int i = 0; i < N - d; ++i)
        if ((i & p) == p) cex(a[i], a[i + d]);
    }
  }
}
template <int N, typename T, typename Cex>
__device__ __forceinline__ void reg_merge_desc(T (&a)[N], Cex cex) {   // a is bitonic -> descending
#pragma unroll
  for (int j = N >> 1; j > 0; j >>= 1) {
#pragma unroll
    for (int i = 0; i < N; ++i) {
      const int l = i ^ j;
      if (l > i) cex(a[i], a[l]);
    }
  }
}
__device__ __forceinline__ void cex_f32(float& x, float& y) {
  const float hi = fmaxf(x, y), lo = fminf(x, y);
  x = hi;
  y = lo;
}

// ---- final sort of the composites ---------------------------------------------------------------------------
// The composite is 62 bits, (ordered key << 30) | (~index & 0x3fffffff), so as an IEEE double it is a non-negative
// finite number (or zero / denormal) whose numeric order is its bit-pattern order: one DSETP on the fp64 pipe
// replaces the ISETP + ISETP.EX pair of a 64-bit integer comparison on the (busier) ALU pipe.
__device__ __forceinline__ unsigned long long tpr_composite(float key, uint32_t idx) {
  return ((unsigned long long)f32_order(key + 0.0f) << 30) | (unsigned long long)(~idx & 0x3fffffffu);
}
__device__ __forceinline__ uint32_t tpr_comp_index(unsigned long long c) { return ~(uint32_t)c & 0x3fffffffu; }
__device__ __forceinline__ float tpr_comp_key(unsigned long long c) { return f32_unorder((uint32_t)(c >> 30)); }
__device__ __forceinline__ void tpr_cex(unsigned long long& x, unsigned long long& y) {
  unsigned long long hi, lo;
  asm("{\n\t.reg .pred p;\n\t.reg .f64 a, b;\n\tmov.b64 a, %2;\n\tmov.b64 b, %3;\n\tsetp.gt.f64 p, a, b;\n\t"
      "selp.b64 %0, %2, %3, p;\n\tselp.b64 %1, %3, %2, p;\n\t}"
      : "=l"(hi), "=l"(lo) : "l"(x), "l"(y));
  x = hi;
  y = lo;
}

}  // namespace l3d
