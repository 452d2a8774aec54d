// util.cu - small device utilities around the forward path.
#include "kernels.h"
#include "rank.cuh"

namespace srs {

int64_t g_launch_count = 0;

// Counter-based uniform fill (splitmix64 of seed + (i+1)*golden): the synthetic
// 10^8-row movie table of BASELINE cfg 5 is generated in place in HBM; the oracle
// regenerates any row it needs from the same formula.
__global__ void fill_uniform_kernel(float* __restrict__ x, int64_t n, uint64_t seed, float lo,
                                    float hi) {
  const float span = hi - lo;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    uint64_t z = seed + (uint64_t)(i + 1) * 0x9E3779B97F4A7C15ULL;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    z = z ^ (z >> 31);
    const float u = (float)(uint32_t)(z >> 40) * (1.0f / 16777216.0f);
    x[i] = __fadd_rn(lo, __fmul_rn(span, u));
  }
}

cudaError_t launch_fill_uniform(float* x, int64_t n, uint64_t seed, float lo, float hi,
                                cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  const int threads = 256;
  int64_t blocks = (n + threads - 1) / threads;
  if (blocks > 148 * 32) blocks = 148 * 32;
  fill_uniform_kernel<<<(int)blocks, threads, 0, s>>>(x, n, seed, lo, hi);
  ++g_launch_count;
  return cudaGetLastError();
}

// uint16 -> int32 history ids (srs_batch::hist16): the narrow form crosses PCIe, the kernels
// read int32.  `src` is 4-byte aligned (packed layout); two ids per thread.
__global__ void widen_u16_kernel(const uint16_t* __restrict__ src, int32_t* __restrict__ dst,
                                 int64_t n) {
  const int64_t pairs = n >> 1;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < pairs;
       i += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t v = __ldg(reinterpret_cast<const uint32_t*>(src) + i);
    *reinterpret_cast<int2*>(dst + 2 * i) = make_int2((int)(v & 0xFFFFu), (int)(v >> 16));
  }
  if ((n & 1) && blockIdx.x == 0 && threadIdx.x == 0) dst[n - 1] = src[n - 1];
}

cudaError_t launch_widen_u16(const uint16_t* src, int32_t* dst, int64_t n, cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  const int threads = 256;
  int64_t blocks = ((n >> 1) + threads - 1) / threads;
  if (blocks < 1) blocks = 1;
  if (blocks > 148 * 8) blocks = 148 * 8;
  widen_u16_kernel<<<(int)blocks, threads, 0, s>>>(src, dst, n);
  ++g_launch_count;
  return cudaGetLastError();
}

// Ranking request "one user x n candidates" (RecForYouProcess.java:46-59): the request ships the user's
// feature row and n candidate movie ids; the movie-side features (the `mf:<movieId>` hashes,
// FeatureEngForRecModel.scala:130-174) are resident in HBM, 32 bytes per movie:
//   {movieGenre1..3 (vocabulary index, -1 missing), movieAvgRating, movieRatingCount, movieRatingStddev,
//    releaseYear, -}.
// This kernel expands both into the packed batch the forward kernels read: user columns broadcast,
// movie columns gathered by candidate id.  req = [userId | userGenre1..5 | userAvgRating,
// userRatingCount, userRatingStddev | hist[hc] | candidate ids[n]]  (32-bit words).
__global__ void assemble_request_kernel(const int32_t* __restrict__ req, const int4* __restrict__ movie_feats,
                                        int n_table, int n, int hc, int dense, int32_t* __restrict__ movie_id,
                                        int32_t* __restrict__ user_id, int32_t* __restrict__ hist,
                                        int32_t* __restrict__ movie_genre, int32_t* __restrict__ user_genre,
                                        float* __restrict__ numerics, int* err_flag) {
  const int words = 2 + hc + (dense ? 15 : 0);              // per row
  const int32_t* cand = req + 9 + hc;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (int64_t)n * words;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int row = (int)(i / words), w = (int)(i - (int64_t)row * words);
    if (w == 0) movie_id[row] = __ldg(cand + row);
    else if (w == 1) user_id[row] = __ldg(req);
    else if (w < 2 + hc) hist[(size_t)row * hc + (w - 2)] = __ldg(req + 9 + (w - 2));
    else {
      const int f = w - 2 - hc;                              // 0..2 movie genres, 3..7 user genres, 8..14 numerics
      if (f >= 3 && f < 8) { user_genre[row * 5 + (f - 3)] = __ldg(req + 1 + (f - 3)); continue; }
      if (f >= 12) { numerics[row * 7 + (f - 8)] = __int_as_float(__ldg(req + 6 + (f - 12))); continue; }
      const int id = __ldg(cand + row);
      int4 a = make_int4(-1, -1, -1, 0), bq = make_int4(0, 0, 0, 0);
      if ((unsigned)id < (unsigned)n_table) {
        a = __ldg(movie_feats + 2 * (size_t)id);
        bq = __ldg(movie_feats + 2 * (size_t)id + 1);
      } else if (err_flag) {
        atomicExch(err_flag, 1);
      }
      if (f < 3) movie_genre[row * 3 + f] = f == 0 ? a.x : (f == 1 ? a.y : a.z);
      else numerics[row * 7 + (f - 8)] = __int_as_float(f == 8 ? a.w : (f == 9 ? bq.x : (f == 10 ? bq.y : bq.z)));
    }
  }
}

cudaError_t launch_assemble_request(const int32_t* req, const void* movie_feats, int n_table, int n, int hc,
                                    int dense, int32_t* movie_id, int32_t* user_id, int32_t* hist,
                                    int32_t* movie_genre, int32_t* user_genre, float* numerics, int* err_flag,
                                    cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  const int words = 2 + hc + (dense ? 15 : 0);
  const int threads = 256;
  int64_t blocks = ((int64_t)n * words + threads - 1) / threads;
  if (blocks > 148 * 8) blocks = 148 * 8;
  assemble_request_kernel<<<(int)blocks, threads, 0, s>>>(req, static_cast<const int4*>(movie_feats), n_table, n, hc,
                                                         dense, movie_id, user_id, hist, movie_genre, user_genre,
                                                         numerics, err_flag);
  ++g_launch_count;
  return cudaGetLastError();
}

// Cosine similarity of one query against n candidates, one warp per candidate.
// Reference: online/model/Embedding.java:33-47 - float products accumulated in double,
// dot / (sqrt(n1) * sqrt(n2)).
__global__ void cosine_kernel(const float* __restrict__ q, const float* __restrict__ c, int n,
                              int dim, float* __restrict__ out) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= n) return;
  const float r = cosine_warp(q, c + (size_t)warp * dim, dim, lane);
  if (lane == 0) out[warp] = r;
}

cudaError_t launch_cosine(const float* q, const float* c, int n, int dim, float* out,
                          cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  const int threads = 256;
  const int blocks = (n * 32 + threads - 1) / threads;
  cosine_kernel<<<blocks, threads, 0, s>>>(q, c, n, dim, out);
  ++g_launch_count;
  return cudaGetLastError();
}

}  // namespace srs
