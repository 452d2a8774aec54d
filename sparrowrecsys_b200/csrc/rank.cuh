// rank.cuh - the ranking order and the "emb" similarity shared by the ranking tail (topk.cu), the
// cosine scorer (util.cu) and candidate retrieval (retrieve.cu), so that all three agree bit for bit.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace srs {

constexpr uint64_t kPadKey = ~0ull;     // sorts after every real key

// A score and its position packed into one 64-bit key whose ascending order is the ranking:
// descending score, NaN first (Double.compareTo: NaN is the greatest value), -0.0 after 0.0,
// equal scores by lower position.
__device__ __forceinline__ uint64_t rank_key(float s, uint32_t i) {
  uint32_t u = __float_as_uint(s);
  if (s != s) u = 0xFFFFFFFFu;                                    // NaN: greatest
  else u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);            // monotone float -> uint
  return ((uint64_t)(~u) << 32) | i;                              // ascending key = descending score
}

// compare-exchange of the pair (i, i | j) for the bitonic stage of width k
__device__ __forceinline__ void cmpx(uint64_t& a, uint64_t& b, bool ascending) {
  if ((a > b) == ascending) {
    const uint64_t t = a; a = b; b = t;
  }
}

// position of the t-th pair's lower element: t with a zero inserted at bit log2(j)
__device__ __forceinline__ uint32_t pair_lo(uint32_t t, uint32_t j) {
  return ((t & ~(j - 1)) << 1) | (t & (j - 1));
}

// Cosine similarity of q and v, computed by a whole warp; the result is lane 0's.
// Reference: online/model/Embedding.java:33-47 - float products accumulated in double,
// dot / (sqrt(n1) * sqrt(n2)).  Lane l sums the elements l, l + 32, ...; the partial sums
// meet in a butterfly, so the association order (and with it every bit of the result) is fixed.
__device__ __forceinline__ float cosine_warp(const float* __restrict__ q, const float* __restrict__ v,
                                             int dim, int lane) {
  double dot = 0.0, n1 = 0.0, n2 = 0.0;
  for (int k = lane; k < dim; k += 32) {
    const float a = __ldg(q + k), bb = __ldg(v + k);
    dot += (double)__fmul_rn(a, bb);
    n1 += (double)__fmul_rn(a, a);
    n2 += (double)__fmul_rn(bb, bb);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    dot += __shfl_xor_sync(0xffffffffu, dot, o);
    n1 += __shfl_xor_sync(0xffffffffu, n1, o);
    n2 += __shfl_xor_sync(0xffffffffu, n2, o);
  }
  return (float)(dot / (sqrt(n1) * sqrt(n2)));
}

}  // namespace srs
