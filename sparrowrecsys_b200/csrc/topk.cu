// topk.cu - rank candidate scores on the device: descending score, first k.
//
// Reference: the `ranker` tail shared by RecForYouProcess.java:92-94 and
// SimilarMovieProcess.java:133-135 -
//   candidateScoreMap.entrySet().stream().sorted(comparingByValue(reverseOrder()))
// followed by `rankedList.subList(0, size)` (RecForYouProcess.java:56-59).  The Java sort
// compares boxed Doubles (Double.compareTo: NaN is the greatest value, -0.0 < 0.0); equal
// scores come out in HashMap iteration order (identity hash codes, i.e. unspecified).  Here
// ties are broken by the candidate's position (lower index first), which is one of the
// orders the reference can produce and the only deterministic one.
//
// A score and its position are packed into one 64-bit key whose ascending order is the
// wanted ranking; the keys are sorted by a bitonic network: one CTA in shared memory for
// n <= 4096 (the reference ranks 800 candidates), shared-memory chunks plus global
// compare-exchange steps above that.
#include "kernels.h"
#include "rank.cuh"

namespace srs {

namespace {

constexpr int kSortChunk = 4096;            // keys one CTA sorts in shared memory (32 KB)
constexpr int kSortThreads = 1024;

// n <= NP <= kSortChunk: the whole ranking in one CTA.
__global__ void __launch_bounds__(kSortThreads)
topk_cta_kernel(const float* __restrict__ scores, int n, int NP, int k,
                int32_t* __restrict__ top_idx, float* __restrict__ top_scores) {
  extern __shared__ uint64_t keys[];
  for (int i = threadIdx.x; i < NP; i += kSortThreads)
    keys[i] = i < n ? rank_key(scores[i], (uint32_t)i) : kPadKey;
  __syncthreads();
  for (uint32_t w = 2; w <= (uint32_t)NP; w <<= 1)
    for (uint32_t j = w >> 1; j > 0; j >>= 1) {
      for (uint32_t t = threadIdx.x; t < (uint32_t)NP / 2; t += kSortThreads) {
        const uint32_t lo = pair_lo(t, j);
        uint64_t a = keys[lo], b = keys[lo | j];
        cmpx(a, b, (lo & w) == 0);
        keys[lo] = a; keys[lo | j] = b;
      }
      __syncthreads();
    }
  for (int r = threadIdx.x; r < k; r += kSortThreads) {
    const uint32_t idx = (uint32_t)keys[r];
    top_idx[r] = (int32_t)idx;
    if (top_scores) top_scores[r] = scores[idx];
  }
}

// n <= 1024: one key per thread, the compare-exchange steps of distance < 32 by warp shuffles, the
// others through shared memory (the reference ranks 800 candidates: RecForYouProcess.java:34).
// Optional tail for the latency path (model.cu): `done` is a host-mapped record the caller spins on
// instead of synchronising the stream; the error word is moved into it and cleared.
__global__ void __launch_bounds__(1024)
topk_small_kernel(const float* __restrict__ scores, int n, int k, int32_t* __restrict__ top_idx,
                  float* __restrict__ top_scores, int* err_flag, volatile uint32_t* done, uint32_t seq) {
  __shared__ uint64_t keys[2][1024];
  const uint32_t tid = threadIdx.x, NP = blockDim.x;
  uint64_t key = tid < (uint32_t)n ? rank_key(scores[tid], tid) : kPadKey;
  int buf = 0;
  for (uint32_t w = 2; w <= NP; w <<= 1) {
    const bool up = (tid & w) == 0;
    for (uint32_t j = w >> 1; j > 0; j >>= 1) {
      uint64_t other;
      if (j >= 32) {
        keys[buf][tid] = key;
        __syncthreads();
        other = keys[buf][tid ^ j];
        buf ^= 1;                                    // the next exchange writes the other buffer: one barrier per step
      } else {
        other = __shfl_xor_sync(0xffffffffu, key, j);
      }
      const bool lower = (tid & j) == 0;
      key = (lower == up) ? (key < other ? key : other) : (key > other ? key : other);
    }
  }
  if (tid < (uint32_t)k) {
    const uint32_t idx = (uint32_t)key;
    top_idx[tid] = (int32_t)idx;
    if (top_scores) top_scores[tid] = scores[idx];
  }
  if (done) {
    __threadfence_system();
    __syncthreads();
    if (tid == 0) {
      done[1] = err_flag ? (uint32_t)atomicExch(err_flag, 0) : 0u;
      __threadfence_system();
      done[0] = seq;
    }
  }
}

// Tail of a latency-path call that does not end in topk_small_kernel: publish the error word and the
// sequence number to the host-mapped record.
__global__ void finish_kernel(int* err_flag, volatile uint32_t* done, uint32_t seq) {
  if (threadIdx.x == 0) {
    __threadfence_system();
    done[1] = err_flag ? (uint32_t)atomicExch(err_flag, 0) : 0u;
    __threadfence_system();
    done[0] = seq;
  }
}

// ---- n > kSortChunk -----------------------------------------------------------------------
__global__ void make_keys_kernel(const float* __restrict__ scores, int n, int NP,
                                 uint64_t* __restrict__ keys) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < NP) keys[i] = i < n ? rank_key(scores[i], (uint32_t)i) : kPadKey;
}

// One CTA per chunk of kSortChunk keys.  first_w == 2: every stage up to width kSortChunk (a full
// sort of the chunk, direction by the chunk's place in the stage of width kSortChunk);
// otherwise the steps j = kSortChunk/2 .. 1 of the single stage of width first_w.
__global__ void __launch_bounds__(kSortThreads)
chunk_sort_kernel(uint64_t* __restrict__ gkeys, uint32_t first_w) {
  __shared__ uint64_t keys[kSortChunk];
  const uint32_t base = blockIdx.x * kSortChunk;
  for (int i = threadIdx.x; i < kSortChunk; i += kSortThreads) keys[i] = gkeys[base + i];
  __syncthreads();
  const uint32_t w_end = first_w == 2 ? (uint32_t)kSortChunk : first_w;
  for (uint32_t w = first_w; w <= w_end; w <<= 1) {
    for (uint32_t j = (w > (uint32_t)kSortChunk ? (uint32_t)kSortChunk : w) >> 1; j > 0; j >>= 1) {
      for (uint32_t t = threadIdx.x; t < kSortChunk / 2; t += kSortThreads) {
        const uint32_t lo = pair_lo(t, j);
        uint64_t a = keys[lo], b = keys[lo | j];
        cmpx(a, b, ((base + lo) & w) == 0);
        keys[lo] = a; keys[lo | j] = b;
      }
      __syncthreads();
    }
    if (w == w_end) break;              // w <<= 1 would overflow for w = 2^31
  }
  for (int i = threadIdx.x; i < kSortChunk; i += kSortThreads) gkeys[base + i] = keys[i];
}

// One compare-exchange step (distance j >= kSortChunk) of the stage of width w, in global memory.
__global__ void global_step_kernel(uint64_t* __restrict__ keys, uint32_t half, uint32_t j,
                                   uint32_t w) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= half) return;
  const uint32_t lo = pair_lo(t, j);
  uint64_t a = keys[lo], b = keys[lo | j];
  const uint64_t a0 = a;
  cmpx(a, b, (lo & w) == 0);
  if (a != a0) {
    keys[lo] = a; keys[lo | j] = b;
  }
}

__global__ void emit_topk_kernel(const uint64_t* __restrict__ keys, const float* __restrict__ scores,
                                 int k, int32_t* __restrict__ top_idx,
                                 float* __restrict__ top_scores) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= k) return;
  const uint32_t idx = (uint32_t)keys[r];
  top_idx[r] = (int32_t)idx;
  if (top_scores) top_scores[r] = scores[idx];
}

}  // namespace

// Scratch bytes launch_topk needs for n scores (0 for n <= kSortChunk).
size_t topk_scratch_bytes(int n) {
  if (n <= kSortChunk) return 0;
  size_t NP = kSortChunk;
  while (NP < (size_t)n) NP <<= 1;
  return NP * sizeof(uint64_t);
}

// top_idx / top_scores receive min(k, n) entries.  `scratch` (device, topk_scratch_bytes(n))
// may be null when n <= kSortChunk.
cudaError_t launch_finish(int* err_flag, uint32_t* done, uint32_t seq, cudaStream_t s) {
  finish_kernel<<<1, 32, 0, s>>>(err_flag, done, seq);
  ++g_launch_count;
  return cudaGetLastError();
}

// `done` != nullptr: the last kernel also publishes {seq, error word} to that host-mapped record.
cudaError_t launch_topk_done(const float* scores, int n, int k, int32_t* top_idx, float* top_scores,
                             void* scratch, int* err_flag, uint32_t* done, uint32_t seq, cudaStream_t s) {
  if (n <= 0 || k <= 0) return done ? launch_finish(err_flag, done, seq, s) : cudaSuccess;
  if (k > n) k = n;
  if (n <= 1024) {
    int NP = 32;
    while (NP < n) NP <<= 1;
    topk_small_kernel<<<1, NP, 0, s>>>(scores, n, k, top_idx, top_scores, err_flag, done, seq);
    ++g_launch_count;
    return cudaGetLastError();
  }
  cudaError_t e = launch_topk(scores, n, k, top_idx, top_scores, scratch, s);
  if (e == cudaSuccess && done) e = launch_finish(err_flag, done, seq, s);
  return e;
}

cudaError_t launch_topk(const float* scores, int n, int k, int32_t* top_idx, float* top_scores,
                        void* scratch, cudaStream_t s) {
  if (n <= 0 || k <= 0) return cudaSuccess;
  if (k > n) k = n;
  if (n <= 1024) return launch_topk_done(scores, n, k, top_idx, top_scores, scratch, nullptr, nullptr, 0, s);
  if (n <= kSortChunk) {
    int NP = 32;
    while (NP < n) NP <<= 1;
    topk_cta_kernel<<<1, kSortThreads, NP * sizeof(uint64_t), s>>>(scores, n, NP, k, top_idx,
                                                              top_scores);
    ++g_launch_count;
    return cudaGetLastError();
  }
  if (!scratch) return cudaErrorInvalidValue;
  uint32_t NP = kSortChunk;
  while (NP < (uint32_t)n) NP <<= 1;
  uint64_t* keys = static_cast<uint64_t*>(scratch);
  make_keys_kernel<<<NP / 256, 256, 0, s>>>(scores, n, (int)NP, keys);
  chunk_sort_kernel<<<NP / kSortChunk, kSortThreads, 0, s>>>(keys, 2u);
  g_launch_count += 2;
  for (uint32_t w = 2u * kSortChunk; w <= NP; w <<= 1) {
    for (uint32_t j = w >> 1; j >= (uint32_t)kSortChunk; j >>= 1) {
      global_step_kernel<<<NP / 2 / 256, 256, 0, s>>>(keys, NP / 2, j, w);
      ++g_launch_count;
    }
    chunk_sort_kernel<<<NP / kSortChunk, kSortThreads, 0, s>>>(keys, w);
    ++g_launch_count;
    if (w == NP) break;
  }
  emit_topk_kernel<<<(k + 255) / 256, 256, 0, s>>>(keys, scores, k, top_idx, top_scores);
  ++g_launch_count;
  return cudaGetLastError();
}

}  // namespace srs
