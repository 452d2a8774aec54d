// retrieve.cu - exact top-k retrieval over an item index resident in HBM (dot or cosine).
//
// Reference: the recall stage before ranking - SimilarMovieProcess.retrievalCandidatesByEmbedding
// (SimilarMovieProcess.java:91-112) scores the whole catalog by embedding cosine; the two-tower model
// (NeuralCF.py:57-70) is the standard recall model with one query vector per user.
//
// One search = for each query the best min(k, eligible) item positions in the rank_key order of
// rank.cuh, with exact scores (dot: fp32 fmaf chain over k = 0..dim-1; cosine: cosine_warp, bit for bit
// the value srs_cosine_scores_device gives).  Queries go in blocks of <= 256:
//   1. seed: the first kSample rows are scored exactly and ranked; their k-th key tau is a lower bound
//      on every query's k-th key, and their top k opens each query's candidate list;
//   2. scan: a persistent tcgen05 kernel multiplies 128-row bf16 tiles of the remaining rows by the
//      bf16 query block (fp32 accumulators in tensor memory) and appends an item to query j's list
//      unless its approximate score is provably below tau_j: s~ < tau_j - m |q_j| |x_i| (DESIGN.md
//      "Candidate retrieval" derives m);
//   3. select: the list is rescored exactly and ranked by one CTA per query (bitonic, rank.cuh).
// A list holds kCap entries; past that the scan only counts.  An overflowing query raises tau to the
// exact k-th key among its captured entries and is scanned again; when the bf16 filter stops making
// progress (near ties below bf16 resolution, equal rows) it switches to exact passes that keep items
// whose exact key is <= tau, which is correct by construction and shrinks tau on every pass.
// Scratch is fixed per index (lists of one query block) and does not depend on n.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <mutex>
#include <vector>

#include "../../include/srs_ctr.h"
#include "kernels.h"
#include "rank.cuh"
#include "rt_common.cuh"

namespace srs {
int report_error(int code, const char* msg);

namespace {

constexpr int kQBlock = 256;          // queries per scan (MMA N <= 256)
constexpr int kCap = 16384;           // candidate list entries per query (and the select CTA's sort width)
constexpr int kSample = 16384;        // seed rows: >= max(8 k, 16384) for k <= 1024
constexpr int kMaxK = 1024;
constexpr int kMaxDim = 128;
constexpr int kScanThreads = 320;     // warp 0 loads, warp 1 issues MMAs, warps 2..9 filter
constexpr int kSelThreads = 1024;
constexpr float kNormPad = 0x1p-50f;  // added to every norm: covers subnormal flushes in the scan
constexpr float kNormHuge = 0x1p60f;  // a norm this large may overflow the bf16 product sums: keep all

enum { SEL_SEED = 0, SEL_FINAL = 1, SEL_TAU = 2 };

// K-major operand tiles: K blocks of W bf16 per row (W = 64: SWIZZLE_128B, 32: SWIZZLE_64B,
// 16: SWIZZLE_32B), 8-row atoms of 8 * 2W bytes; the 16-byte chunk c of row r is stored at chunk
// c ^ (r's swizzle bits).  The scan copy is stored in global memory in exactly this layout, so one
// bulk copy per tile lands it ready for tcgen05.mma.
__host__ __device__ __forceinline__ uint32_t tile_offset(uint32_t row, uint32_t chunk, int W) {
  const uint32_t x = W == 64 ? (row & 7u) : W == 32 ? ((row >> 1) & 3u) : ((row >> 2) & 1u);
  return row * (uint32_t)(2 * W) + ((chunk ^ x) << 4);
}
__device__ __forceinline__ uint64_t smem_desc_kmajor(uint32_t addr, int W) {
  uint64_t d = 0;
  d |= (uint64_t)((addr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;                                      // leading byte offset: unused for swizzled K-major
  d |= (uint64_t)((16u * W) >> 4) << 32;                       // stride byte offset: one 8-row atom
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)(W == 64 ? 2 : W == 32 ? 4 : 6) << 61;        // SWIZZLE_128B / 64B / 32B
  return d;
}
int kblock_width(int Dp) { return Dp % 64 == 0 ? 64 : Dp % 32 == 0 ? 32 : 16; }

__device__ __forceinline__ float dot_exact(const float* __restrict__ q, const float* __restrict__ x, int dim) {
  float s = 0.f;
  for (int k = 0; k < dim; ++k) s = fmaf(__ldg(q + k), __ldg(x + k), s);
  return s;
}
// the score of a key (inverse of rank_key; NaN for the NaN key)
__device__ __forceinline__ float key_score(uint64_t key) {
  const uint32_t u = ~(uint32_t)(key >> 32);
  if (u == 0xFFFFFFFFu) return __int_as_float(0x7FFFFFFF);
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u);
}

// ---- index build --------------------------------------------------------------------------------
__device__ __forceinline__ double sumsq_f(const float* x, int dim) {   // cosine_warp's n2 terms
  double s = 0.0;
  for (int k = 0; k < dim; ++k) s += (double)__fmul_rn(x[k], x[k]);
  return s;
}

// dot: |x| rounded up, plus kNormPad; rows whose products could overflow get +inf.  cosine: 1.
__global__ void index_norms_kernel(const float* __restrict__ rows, int64_t n, int dim, int metric,
                                   float* __restrict__ norms) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    if (metric == SRS_COSINE) { norms[i] = 1.f; continue; }
    const float* x = rows + i * dim;
    double s = 0.0;
    for (int k = 0; k < dim; ++k) s += (double)x[k] * (double)x[k];
    float nr = __fadd_ru(__double2float_ru(sqrt(s) * (1.0 + 1e-12)), kNormPad);
    if (nr >= kNormHuge) nr = __int_as_float(0x7F800000);
    norms[i] = nr;
  }
}

// bf16 scan copy, one thread per (row, 8-element chunk).  Cosine rows are normalised; a row whose cosine
// is NaN for every query (zero or non-finite) is stored as NaN so that the filter always keeps it.
__global__ void index_tiles_kernel(const float* __restrict__ rows, int64_t n, int dim, int Dp, int W,
                                   int metric, int64_t total_rows, uint8_t* __restrict__ scan) {
  const int cpr = Dp / 8;
  const uint32_t tile_bytes = 128u * Dp * 2u;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total_rows * cpr;
       t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = t / cpr;
    const int cc = (int)(t - r * cpr);
    float v[8];
    double scale = 1.0;
    bool bad = false;
    if (r < n && metric == SRS_COSINE) {
      const double s = sumsq_f(rows + r * dim, dim);
      bad = !(s > 0.0) || !isfinite(s);
      scale = 1.0 / sqrt(s);
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int k = cc * 8 + e;
      float x = (r < n && k < dim) ? rows[r * dim + k] : 0.f;
      if (metric == SRS_COSINE && r < n) x = bad ? __int_as_float(0x7FC00000) : (k < dim ? (float)((double)x * scale) : 0.f);
      v[e] = x;
    }
    uint4 pk;
    __nv_bfloat162 h0 = __floats2bfloat162_rn(v[0], v[1]), h1 = __floats2bfloat162_rn(v[2], v[3]);
    __nv_bfloat162 h2 = __floats2bfloat162_rn(v[4], v[5]), h3 = __floats2bfloat162_rn(v[6], v[7]);
    pk.x = *reinterpret_cast<uint32_t*>(&h0); pk.y = *reinterpret_cast<uint32_t*>(&h1);
    pk.z = *reinterpret_cast<uint32_t*>(&h2); pk.w = *reinterpret_cast<uint32_t*>(&h3);
    const int kb = cc / (W / 8), c = cc % (W / 8);
    const int64_t tile = r >> 7;
    uint8_t* dst = scan + tile * tile_bytes + (size_t)kb * 128 * W * 2 + tile_offset((uint32_t)(r & 127), c, W);
    *reinterpret_cast<uint4*>(dst) = pk;
  }
}

// ---- one query block: bf16 operand, slack multipliers, exclude check -------------------------------
__global__ void prep_queries_kernel(const float* __restrict__ q, int nq, int N, int dim, int Dp, int W, int metric,
                                    float m, const int32_t* __restrict__ excl, int64_t n,
                                    uint8_t* __restrict__ bop, float* __restrict__ mq, int* err) {
  const int cpr = Dp / 8;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= N * cpr) return;
  const int r = t / cpr, cc = t % cpr;
  float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (r < nq) {
    const float* x = q + (size_t)r * dim;
    double scale = 1.0;
    bool bad = false;
    if (metric == SRS_COSINE) {
      const double s = sumsq_f(x, dim);
      bad = !(s > 0.0) || !isfinite(s);
      scale = 1.0 / sqrt(s);
    }
    for (int e = 0; e < 8; ++e) {
      const int k = cc * 8 + e;
      if (k < dim) v[e] = metric == SRS_COSINE ? (bad ? __int_as_float(0x7FC00000) : (float)((double)x[k] * scale)) : x[k];
    }
    if (cc == 0) {
      if (metric == SRS_COSINE) {
        mq[r] = m;
      } else {
        double s = 0.0;
        for (int k = 0; k < dim; ++k) s += (double)x[k] * (double)x[k];
        float nr = __fadd_ru(__double2float_ru(sqrt(s) * (1.0 + 1e-12)), kNormPad);
        if (nr >= kNormHuge) nr = __int_as_float(0x7F800000);
        mq[r] = __fmul_ru(m, nr);
      }
      if (excl) {
        const int32_t e = excl[r];
        if (e != -1 && (e < 0 || (int64_t)e >= n)) atomicExch(err, 1);
      }
    }
  }
  uint4 pk;
  __nv_bfloat162 h0 = __floats2bfloat162_rn(v[0], v[1]), h1 = __floats2bfloat162_rn(v[2], v[3]);
  __nv_bfloat162 h2 = __floats2bfloat162_rn(v[4], v[5]), h3 = __floats2bfloat162_rn(v[6], v[7]);
  pk.x = *reinterpret_cast<uint32_t*>(&h0); pk.y = *reinterpret_cast<uint32_t*>(&h1);
  pk.z = *reinterpret_cast<uint32_t*>(&h2); pk.w = *reinterpret_cast<uint32_t*>(&h3);
  const int kb = cc / (W / 8), c = cc % (W / 8);
  *reinterpret_cast<uint4*>(bop + (size_t)kb * N * W * 2 + tile_offset((uint32_t)r, c, W)) = pk;
}

// ---- exact rescoring + ranking, one CTA per query ------------------------------------------------------
struct SelParams {
  int mode, metric, dim, k, C, range;
  const float* rows;
  const float* queries;        // block base [nb][dim]
  const int32_t* excl;         // block base or nullptr
  const int32_t* qset;         // block-local query indices, one per CTA
  int32_t* list;               // [nb][C]
  int32_t* counts;             // [nb]
  int32_t* seedpos;            // [nb][kMaxK]
  int32_t* nseed;              // [nb]
  int32_t* state;              // [nb]: 0 scan, 1 nothing beyond the seed can rank
  int32_t* prog;               // [nb]: SEL_TAU: tau improved (and is not NaN)
  uint64_t* tau_key;           // [nb]
  float* tau_score;            // [nb]
  int32_t* out_pos;            // block base [nb][k]
  float* out_score;
};

__global__ void __launch_bounds__(kSelThreads) select_kernel(SelParams p) {
  extern __shared__ uint64_t keys[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int j = p.qset[blockIdx.x];
  const float* q = p.queries + (size_t)j * p.dim;
  const int ex = p.excl ? p.excl[j] : -1;
  const int32_t* lst = p.mode == SEL_SEED ? nullptr : p.list + (size_t)j * p.C;
  const int m = p.mode == SEL_SEED ? p.range : min(p.counts[j], p.C);
  uint32_t NP = 2;
  while (NP < (uint32_t)m) NP <<= 1;
  for (uint32_t c = tid; c < NP; c += kSelThreads) keys[c] = kPadKey;
  __syncthreads();
  if (p.metric == SRS_DOT) {
    for (int c = tid; c < m; c += kSelThreads) {
      const int pos = lst ? lst[c] : c;
      if (pos != ex) keys[c] = rank_key(dot_exact(q, p.rows + (size_t)pos * p.dim, p.dim), (uint32_t)pos);
    }
  } else {
    for (int c = warp; c < m; c += kSelThreads / 32) {
      const int pos = lst ? lst[c] : c;
      if (pos == ex) continue;
      const float s = cosine_warp(q, p.rows + (size_t)pos * p.dim, p.dim, lane);
      if (lane == 0) keys[c] = rank_key(s, (uint32_t)pos);
    }
  }
  __syncthreads();
  for (uint32_t w = 2; w <= NP; w <<= 1)
    for (uint32_t jj = w >> 1; jj > 0; jj >>= 1) {
      for (uint32_t t = tid; t < NP / 2; t += kSelThreads) {
        const uint32_t lo = pair_lo(t, jj);
        uint64_t a = keys[lo], b = keys[lo | jj];
        cmpx(a, b, (lo & w) == 0);
        keys[lo] = a; keys[lo | jj] = b;
      }
      __syncthreads();
    }
  const int k = p.k;
  const int kvalid = __syncthreads_count(tid < k && tid < (int)NP && keys[tid] != kPadKey);
  if (p.mode == SEL_TAU) {
    if (tid == 0) {
      const uint64_t nk = keys[k - 1];
      const float ns = key_score(nk);
      p.prog[j] = (nk < p.tau_key[j] && ns == ns) ? 1 : 0;
      p.tau_key[j] = nk;
      p.tau_score[j] = ns;
    }
    return;
  }
  // outputs: positions, exact scores (recomputed by the same code), -1 / 0 past the eligible items
  int32_t* op = p.out_pos + (size_t)j * k;
  float* os = p.out_score + (size_t)j * k;
  for (int r = tid; r < k; r += kSelThreads) {
    const int pos = r < kvalid ? (int)(uint32_t)keys[r] : -1;
    op[r] = pos;
    if (pos < 0) os[r] = 0.f;
    else if (p.metric == SRS_DOT) os[r] = dot_exact(q, p.rows + (size_t)pos * p.dim, p.dim);
    if (p.mode == SEL_SEED && r < kvalid) {
      p.list[(size_t)j * p.C + r] = pos;
      p.seedpos[(size_t)j * kMaxK + r] = pos;
    }
  }
  if (p.metric == SRS_COSINE)
    for (int r = warp; r < kvalid; r += kSelThreads / 32) {
      const int pos = (int)(uint32_t)keys[r];
      const float s = cosine_warp(q, p.rows + (size_t)pos * p.dim, p.dim, lane);
      if (lane == 0) os[r] = s;
    }
  if (p.mode == SEL_SEED && tid == 0) {
    p.counts[j] = kvalid;
    p.nseed[j] = kvalid;
    if (kvalid == k) {
      const uint64_t tk = keys[k - 1];
      const float ts = key_score(tk);
      p.tau_key[j] = tk;
      p.tau_score[j] = ts;
      p.state[j] = ts != ts ? 1 : 0;     // k NaN scores in the sample: no later position can rank before them
    } else {
      p.tau_key[j] = kPadKey;
      p.tau_score[j] = -INFINITY;
      p.state[j] = 0;
    }
  }
}

// ---- the filtered scan (tcgen05) ------------------------------------------------------------------------
struct ScanParams {
  const uint8_t* scan;         // bf16 tiles
  const float* norms;          // [n]
  const uint8_t* bop;          // query block operand [Dp/W][N rows][W]
  const float* tau_score;
  const float* mq;
  const int32_t* excl;         // or nullptr
  const int32_t* state;
  int32_t* list;
  int32_t* counts;
  int64_t n;
  int tile_begin, tile_end;
  int Dp, W, N, nq, C, stages;
  uint32_t tile_bytes, b_bytes, b_pad, tmem_cols;
};

__global__ void __launch_bounds__(kScanThreads, 1) scan_kernel(ScanParams p) {
  extern __shared__ uint8_t raw[];
  __shared__ uint64_t full[8], empty[8], tfull[2], tempty[2], bbar;
  __shared__ uint32_t tmem_slot;
  __shared__ float s_tau[kQBlock], s_mq[kQBlock];
  __shared__ int s_ex[kQBlock];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  uint8_t* base = raw + ((1024u - (smem_u32(raw) & 1023u)) & 1023u);
  uint8_t* sB = base;
  uint8_t* ring = base + p.b_pad;
  for (int j = tid; j < p.N; j += kScanThreads) {
    const bool on = j < p.nq && p.state[j] == 0;
    s_tau[j] = on ? p.tau_score[j] : 0.f;
    s_mq[j] = on ? p.mq[j] : 0.f;
    s_ex[j] = on ? (p.excl ? p.excl[j] : -1) : -2;              // -2: column not filtered
  }
  if (warp == 0) tmem_alloc(&tmem_slot, p.tmem_cols);
  if (tid == 0) {
    for (int s = 0; s < p.stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&tfull[a], 1); mbar_init(&tempty[a], 8); }
    mbar_init(&bbar, 1);
    fence_mbar_init();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tbase = tmem_slot;
  const int ST = p.stages;

  if (warp == 0) {
    if (elect_one()) {
      mbar_arrive_expect_tx(&bbar, p.b_bytes);
      bulk_g2s(sB, p.bop, p.b_bytes, &bbar);
      int it = 0;
      for (int t = p.tile_begin + blockIdx.x; t < p.tile_end; t += gridDim.x, ++it) {
        const int s = it % ST;
        if (it >= ST) mbar_wait(&empty[s], ((it / ST) - 1) & 1);
        mbar_arrive_expect_tx(&full[s], p.tile_bytes);
        bulk_g2s(ring + (size_t)s * p.tile_bytes, p.scan + (size_t)t * p.tile_bytes, p.tile_bytes, &full[s]);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    mbar_wait(&bbar, 0);
    __syncwarp();
    const uint32_t idesc = idesc_bf16(128, p.N);
    const int KB = p.Dp / p.W, KS = p.W / 16;
    int it = 0;
    for (int t = p.tile_begin + blockIdx.x; t < p.tile_end; t += gridDim.x, ++it) {
      const int s = it % ST, a = it & 1;
      mbar_wait(&full[s], (it / ST) & 1);
      if (it >= 2) mbar_wait(&tempty[a], ((it >> 1) - 1) & 1);
      __syncwarp();
      tc_fence_after();
      if (elect_one()) {
        const uint32_t a_addr = smem_u32(ring + (size_t)s * p.tile_bytes), b_addr = smem_u32(sB);
        for (int kb = 0; kb < KB; ++kb) {
          const uint64_t ad = smem_desc_kmajor(a_addr + kb * 128 * p.W * 2, p.W);
          const uint64_t bd = smem_desc_kmajor(b_addr + kb * p.N * p.W * 2, p.W);
          for (int ks = 0; ks < KS; ++ks)
            mma_ss(tbase + a * p.N, ad + 2 * ks, bd + 2 * ks, idesc, (kb | ks) != 0);
        }
        mma_commit(&empty[s]);
        mma_commit(&tfull[a]);
      }
      __syncwarp();
    }
  } else {
    const int g = warp & 3, h = (warp - 2) >> 2;           // TMEM lane quarter, column half
    const int half = p.N >> 1;
    const uint32_t lt_mask = (1u << lane) - 1u;
    int it = 0;
    for (int t = p.tile_begin + blockIdx.x; t < p.tile_end; t += gridDim.x, ++it) {
      const int a = it & 1;
      mbar_wait(&tfull[a], (it >> 1) & 1);
      __syncwarp();
      tc_fence_after();
      const int64_t i = (int64_t)t * 128 + g * 32 + lane;
      const bool valid = i < p.n;
      const float xn = valid ? __ldg(p.norms + i) : 0.f;
      for (int c0 = h * half; c0 < (h + 1) * half; c0 += 8) {
        uint32_t r[8];
        tmem_ld8(tmem_addr(tbase + a * p.N, g * 32, c0), r);
        tmem_ld_wait();
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) {
          const int j = c0 + jj;
          const int ex = s_ex[j];
          if (ex == -2) continue;
          const float s = __uint_as_float(r[jj]);
          const float thr = __fsub_rd(s_tau[j], __fmul_ru(s_mq[j], xn));
          const bool keep = valid && i != ex && !(s < thr);
          const uint32_t bal = __ballot_sync(0xffffffffu, keep);
          if (bal) {
            const int leader = __ffs(bal) - 1;
            int b0 = 0;
            if (lane == leader) b0 = atomicAdd(p.counts + j, __popc(bal));
            b0 = __shfl_sync(0xffffffffu, b0, leader);
            const int slot = b0 + __popc(bal & lt_mask);
            if (keep && slot < p.C) p.list[(size_t)j * p.C + slot] = (int32_t)i;
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[a]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tbase, p.tmem_cols);
}

// ---- overflow: list reset and the exact pass ---------------------------------------------------------------
__global__ void reset_lists_kernel(const int32_t* qset, int from_seed, int C, int32_t* list, int32_t* counts,
                                   const int32_t* seedpos, const int32_t* nseed) {
  const int j = qset[blockIdx.x];
  const int ns = from_seed ? nseed[j] : 0;
  for (int r = threadIdx.x; r < ns; r += blockDim.x) list[(size_t)j * C + r] = seedpos[(size_t)j * kMaxK + r];
  if (threadIdx.x == 0) counts[j] = ns;
}

// every row whose exact key is <= tau_key (ranks at or before the current bound) is appended
__global__ void exact_pass_kernel(const float* __restrict__ rows, int64_t n, int dim, int metric,
                                  const float* __restrict__ queries, const int32_t* excl, const int32_t* qset,
                                  const uint64_t* tau_key, int C, int32_t* list, int32_t* counts) {
  const int j = qset[blockIdx.y];
  const float* q = queries + (size_t)j * dim;
  const int ex = excl ? excl[j] : -1;
  const uint64_t tk = tau_key[j];
  const int lane = threadIdx.x & 31;
  if (metric == SRS_DOT) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i0 = (int64_t)blockIdx.x * blockDim.x; i0 < n; i0 += stride) {   // warp-uniform trip count
      const int64_t i = i0 + threadIdx.x;
      bool keep = false;
      if (i < n && i != ex) keep = rank_key(dot_exact(q, rows + i * dim, dim), (uint32_t)i) <= tk;
      const uint32_t bal = __ballot_sync(0xffffffffu, keep);
      if (bal) {
        const int leader = __ffs(bal) - 1;
        int b0 = 0;
        if (lane == leader) b0 = atomicAdd(counts + j, __popc(bal));
        b0 = __shfl_sync(0xffffffffu, b0, leader);
        const int slot = b0 + __popc(bal & ((1u << lane) - 1u));
        if (keep && slot < C) list[(size_t)j * C + slot] = (int32_t)i;
      }
    }
  } else {
    const int64_t nw = (int64_t)gridDim.x * blockDim.x / 32;
    for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / 32; i < n; i += nw) {
      if (i == ex) continue;
      const float s = cosine_warp(q, rows + i * dim, dim, lane);
      if (lane == 0 && rank_key(s, (uint32_t)i) <= tk) {
        const int slot = atomicAdd(counts + j, 1);
        if (slot < C) list[(size_t)j * C + slot] = (int32_t)i;
      }
    }
  }
}

// Bound m on |bf16 scan score - exact score| / (|q| |x|) (DESIGN.md "Candidate retrieval"):
// bf16 rounding of both operands (unit roundoff u = 2^-8), fp32 accumulation of Dp exact products in
// the tensor core in any order with any rounding (2^-23 per addition), and the fp32 fmaf chain of the
// exact score (2^-24), times a safety factor for the fp32 norms.
double gamma_n(int n, double u) { return n * u / (1.0 - n * u); }
float margin(int Dp, int metric) {
  const double u = std::ldexp(1.0, -8);
  double m = 2 * u + u * u + (1 + u) * (1 + u) * gamma_n(Dp, std::ldexp(1.0, -23)) + gamma_n(Dp, std::ldexp(1.0, -24));
  m *= 1.0 + std::ldexp(1.0, -10);
  // cosine: the operands are the rows scaled to unit length in fp32 (|x^| <= 1 + 2^-20), and the exact score
  // is the double-precision cosine rounded to float
  if (metric == SRS_COSINE) m = m * (1.0 + std::ldexp(1.0, -18)) + std::ldexp(1.0, -21);
  return (float)std::nextafter((float)m, INFINITY);
}

int grid_for(int64_t work, int threads, int cap) {
  int64_t b = (work + threads - 1) / threads;
  if (b < 1) b = 1;
  return (int)(b > cap ? cap : b);
}

}  // namespace
}  // namespace srs

using namespace srs;

struct srs_index {
  int device = 0, metric = 0, dim = 0, Dp = 0, W = 0, sms = 148;
  int64_t n = 0;
  int ntiles = 0;
  float* rows = nullptr;
  bool own_rows = false;
  uint8_t* scan = nullptr;
  float* norms = nullptr;
  float m = 0.f;
  // scratch of one query block (independent of n)
  uint8_t* scratch = nullptr;
  int32_t *list = nullptr, *counts = nullptr, *seedpos = nullptr, *nseed = nullptr, *state = nullptr, *prog = nullptr;
  int32_t *qsets = nullptr, *err = nullptr;
  uint64_t* tau_key = nullptr;
  float *tau_score = nullptr, *mq = nullptr;
  uint8_t* bop = nullptr;
  int32_t* pin = nullptr;      // pinned: counts | prog | err | 5 query sets | state
  cudaStream_t stream = nullptr;      // srs_index_search_host's stream
  cudaEvent_t done = nullptr;         // recorded at the end of every search: the next one, on any stream, waits for it
  uint8_t* stage = nullptr;           // srs_index_search_host's device staging (grows)
  size_t stage_bytes = 0;
  std::mutex mu;
};

namespace {

int fail_fmt(int code, const char* fmt, ...) __attribute__((format(printf, 2, 3)));
int fail_fmt(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  return report_error(code, buf);
}

#define RT_TRY(expr)                                                                               \
  do {                                                                                             \
    cudaError_t e__ = (expr);                                                                      \
    if (e__ != cudaSuccess)                                                                        \
      return fail_fmt(SRS_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, \
                      __LINE__);                                                                   \
  } while (0)

enum { PIN_COUNTS = 0, PIN_PROG = kQBlock, PIN_ERR = 2 * kQBlock, PIN_SETS = 2 * kQBlock + 32,
       PIN_STATE = PIN_SETS + 5 * kQBlock, PIN_WORDS = PIN_STATE + kQBlock };
enum { SET_ALL = 0, SET_FINAL, SET_TAU, SET_BF, SET_EXACT };

cudaError_t setup_retrieve_attributes() {
  cudaError_t e = cudaFuncSetAttribute(scan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024);   // + static smem <= 227 KB
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kCap * 8);
  return e;
}

int alloc_scratch(srs_index* ix) {
  size_t off = 0;
  auto take = [&](size_t bytes) { const size_t o = off; off += (bytes + 1023) & ~(size_t)1023; return o; };
  const size_t o_list = take((size_t)kQBlock * kCap * 4), o_counts = take(kQBlock * 4), o_seed = take((size_t)kQBlock * kMaxK * 4),
               o_nseed = take(kQBlock * 4), o_state = take(kQBlock * 4), o_prog = take(kQBlock * 4),
               o_sets = take(5 * kQBlock * 4), o_err = take(64), o_tk = take(kQBlock * 8), o_ts = take(kQBlock * 4),
               o_mq = take(kQBlock * 4), o_bop = take((size_t)kQBlock * kMaxDim * 2);
  RT_TRY(cudaMalloc(&ix->scratch, off));
  uint8_t* b = ix->scratch;
  ix->list = reinterpret_cast<int32_t*>(b + o_list);
  ix->counts = reinterpret_cast<int32_t*>(b + o_counts);
  ix->seedpos = reinterpret_cast<int32_t*>(b + o_seed);
  ix->nseed = reinterpret_cast<int32_t*>(b + o_nseed);
  ix->state = reinterpret_cast<int32_t*>(b + o_state);
  ix->prog = reinterpret_cast<int32_t*>(b + o_prog);
  ix->qsets = reinterpret_cast<int32_t*>(b + o_sets);
  ix->err = reinterpret_cast<int32_t*>(b + o_err);
  ix->tau_key = reinterpret_cast<uint64_t*>(b + o_tk);
  ix->tau_score = reinterpret_cast<float*>(b + o_ts);
  ix->mq = reinterpret_cast<float*>(b + o_mq);
  ix->bop = b + o_bop;
  RT_TRY(cudaMallocHost(&ix->pin, PIN_WORDS * 4));
  RT_TRY(cudaStreamCreateWithFlags(&ix->stream, cudaStreamNonBlocking));
  RT_TRY(cudaEventCreateWithFlags(&ix->done, cudaEventDisableTiming));
  return SRS_OK;
}

void free_index(srs_index* ix) {
  if (!ix) return;
  cudaSetDevice(ix->device);
  if (ix->own_rows) cudaFree(ix->rows);
  cudaFree(ix->scan);
  cudaFree(ix->norms);
  cudaFree(ix->scratch);
  if (ix->pin) cudaFreeHost(ix->pin);
  if (ix->stream) cudaStreamDestroy(ix->stream);
  if (ix->done) cudaEventDestroy(ix->done);
  cudaFree(ix->stage);
  delete ix;
}

SelParams sel_params(srs_index* ix, int mode, int k, const float* q, const int32_t* excl, int32_t* out_pos,
                     float* out_score, int set) {
  SelParams p{};
  p.mode = mode; p.metric = ix->metric; p.dim = ix->dim; p.k = k; p.C = kCap;
  p.range = (int)std::min<int64_t>(ix->n, kSample);
  p.rows = ix->rows; p.queries = q; p.excl = excl; p.qset = ix->qsets + set * kQBlock;
  p.list = ix->list; p.counts = ix->counts; p.seedpos = ix->seedpos; p.nseed = ix->nseed; p.state = ix->state;
  p.prog = ix->prog; p.tau_key = ix->tau_key; p.tau_score = ix->tau_score;
  p.out_pos = out_pos; p.out_score = out_score;
  return p;
}

// copy a query set to the device (pinned region `set`; each region is written at most once between two
// stream synchronisations, so an earlier asynchronous copy from it has completed)
cudaError_t put_set(srs_index* ix, int set, const std::vector<int>& v, cudaStream_t s) {
  int32_t* h = ix->pin + PIN_SETS + set * kQBlock;
  for (size_t i = 0; i < v.size(); ++i) h[i] = v[i];
  return cudaMemcpyAsync(ix->qsets + set * kQBlock, h, v.size() * 4, cudaMemcpyHostToDevice, s);
}

cudaError_t launch_select(const SelParams& p, int nset, cudaStream_t s) {
  if (nset == 0) return cudaSuccess;
  select_kernel<<<nset, kSelThreads, kCap * 8, s>>>(p);
  ++g_launch_count;
  return cudaGetLastError();
}

cudaError_t launch_scan(srs_index* ix, int nq, const int32_t* excl, cudaStream_t s) {
  ScanParams p{};
  const int N = (nq + 15) & ~15;
  p.scan = ix->scan; p.norms = ix->norms; p.bop = ix->bop; p.tau_score = ix->tau_score; p.mq = ix->mq;
  p.excl = excl; p.state = ix->state; p.list = ix->list; p.counts = ix->counts; p.n = ix->n;
  p.tile_begin = kSample / 128; p.tile_end = ix->ntiles;
  p.Dp = ix->Dp; p.W = ix->W; p.N = N; p.nq = nq; p.C = kCap;
  p.tile_bytes = 128u * ix->Dp * 2u;
  p.b_bytes = (uint32_t)N * ix->Dp * 2u;
  p.b_pad = (p.b_bytes + 1023u) & ~1023u;
  uint32_t cols = 32;
  while (cols < 2u * N) cols <<= 1;
  p.tmem_cols = cols;
  const uint32_t budget = 200u * 1024u - p.b_pad;
  p.stages = (int)std::min<uint32_t>(8u, budget / p.tile_bytes);
  // at least 120 KB so that one CTA holds an SM (and its tensor memory) alone
  const size_t smem = std::max<size_t>(1024 + p.b_pad + (size_t)p.stages * p.tile_bytes, 120 * 1024);
  const int tiles = p.tile_end - p.tile_begin;
  if (tiles <= 0) return cudaSuccess;
  const int grid = std::min(tiles, ix->sms);
  scan_kernel<<<grid, kScanThreads, smem, s>>>(p);
  ++g_launch_count;
  return cudaGetLastError();
}

// One block of nb <= 256 queries.  Synchronises the stream (reads the exclude check and the list counts).
int search_block(srs_index* ix, const float* q, int nb, int k, const int32_t* excl, int32_t* out_pos,
                 float* out_score, cudaStream_t s) {
  const int N = (nb + 15) & ~15;
  const int cpr = ix->Dp / 8;
  RT_TRY(cudaMemsetAsync(ix->err, 0, 4, s));
  prep_queries_kernel<<<grid_for((int64_t)N * cpr, 256, 1 << 20), 256, 0, s>>>(
      q, nb, N, ix->dim, ix->Dp, ix->W, ix->metric, ix->m, excl, ix->n, ix->bop, ix->mq, ix->err);
  ++g_launch_count;
  RT_TRY(cudaGetLastError());
  RT_TRY(cudaMemcpyAsync(ix->pin + PIN_ERR, ix->err, 4, cudaMemcpyDeviceToHost, s));
  RT_TRY(cudaStreamSynchronize(s));
  if (ix->pin[PIN_ERR]) return fail_fmt(SRS_ERR_INVALID, "an exclude position is outside 0..%lld (-1 = none)",
                                        (long long)ix->n - 1);
  std::vector<int> all(nb);
  for (int j = 0; j < nb; ++j) all[j] = j;
  RT_TRY(put_set(ix, SET_ALL, all, s));
  RT_TRY(launch_select(sel_params(ix, SEL_SEED, k, q, excl, out_pos, out_score, SET_ALL), nb, s));
  if (ix->n <= kSample) return SRS_OK;            // the sample is the catalog: the seed ranking is the answer
  RT_TRY(launch_scan(ix, nb, excl, s));
  int32_t* hc = ix->pin + PIN_COUNTS;
  RT_TRY(cudaMemcpyAsync(hc, ix->counts, nb * 4, cudaMemcpyDeviceToHost, s));
  RT_TRY(cudaStreamSynchronize(s));
  std::vector<int> fits, over;
  for (int j = 0; j < nb; ++j) (hc[j] <= kCap ? fits : over).push_back(j);
  RT_TRY(put_set(ix, SET_FINAL, fits, s));
  RT_TRY(launch_select(sel_params(ix, SEL_FINAL, k, q, excl, out_pos, out_score, SET_FINAL), (int)fits.size(), s));
  std::vector<int> last(hc, hc + nb), exact(nb, 0);
  while (!over.empty()) {
    RT_TRY(put_set(ix, SET_TAU, over, s));
    RT_TRY(launch_select(sel_params(ix, SEL_TAU, k, q, excl, out_pos, out_score, SET_TAU), (int)over.size(), s));
    int32_t* hp = ix->pin + PIN_PROG;
    RT_TRY(cudaMemcpyAsync(hp, ix->prog, nb * 4, cudaMemcpyDeviceToHost, s));
    RT_TRY(cudaStreamSynchronize(s));
    std::vector<int> bf, ex;
    for (int j : over) {
      // bf16 passes go on while tau rises and each pass keeps fewer rows than the one before; when tau stays,
      // or the bf16 scores cannot tell the rows apart any more (near ties, equal rows), exact passes take over
      if (!exact[j] && hp[j]) bf.push_back(j);
      else { exact[j] = 1; ex.push_back(j); }
    }
    if (!bf.empty()) {
      int32_t* hs = ix->pin + PIN_STATE;
      for (int j = 0; j < nb; ++j) hs[j] = 1;
      for (int j : bf) hs[j] = 0;
      RT_TRY(cudaMemcpyAsync(ix->state, hs, nb * 4, cudaMemcpyHostToDevice, s));
      RT_TRY(put_set(ix, SET_BF, bf, s));
      reset_lists_kernel<<<(int)bf.size(), 256, 0, s>>>(ix->qsets + SET_BF * kQBlock, 1, kCap, ix->list, ix->counts,
                                                       ix->seedpos, ix->nseed);
      ++g_launch_count;
      RT_TRY(cudaGetLastError());
      RT_TRY(launch_scan(ix, nb, excl, s));
    }
    if (!ex.empty()) {
      RT_TRY(put_set(ix, SET_EXACT, ex, s));
      reset_lists_kernel<<<(int)ex.size(), 256, 0, s>>>(ix->qsets + SET_EXACT * kQBlock, 0, kCap, ix->list, ix->counts,
                                                       ix->seedpos, ix->nseed);
      ++g_launch_count;
      const int bx = grid_for(ix->n, 256, std::max(1, 4 * ix->sms / (int)ex.size()));
      exact_pass_kernel<<<dim3(bx, (unsigned)ex.size()), 256, 0, s>>>(
          ix->rows, ix->n, ix->dim, ix->metric, q, excl, ix->qsets + SET_EXACT * kQBlock, ix->tau_key, kCap, ix->list,
          ix->counts);
      ++g_launch_count;
      RT_TRY(cudaGetLastError());
    }
    RT_TRY(cudaMemcpyAsync(hc, ix->counts, nb * 4, cudaMemcpyDeviceToHost, s));
    RT_TRY(cudaStreamSynchronize(s));
    std::vector<int> done, left;
    for (int j : over) {
      (hc[j] <= kCap ? done : left).push_back(j);
      if (!exact[j] && hc[j] >= last[j]) exact[j] = 1;
      last[j] = hc[j];
    }
    RT_TRY(put_set(ix, SET_FINAL, done, s));
    RT_TRY(launch_select(sel_params(ix, SEL_FINAL, k, q, excl, out_pos, out_score, SET_FINAL), (int)done.size(), s));
    over.swap(left);
  }
  return SRS_OK;
}

// The caller holds ix->mu.  Every search waits for the previous one (ix->done), whatever stream either runs on:
// the scratch lists and the pinned staging are per index.
int search_locked(srs_index* ix, const float* queries, int32_t q, int32_t dim, int32_t k, const int32_t* exclude,
                  int32_t* top_pos, float* top_scores, cudaStream_t s) {
  RT_TRY(cudaSetDevice(ix->device));
  RT_TRY(cudaStreamWaitEvent(s, ix->done, 0));
  for (int b0 = 0; b0 < q; b0 += kQBlock) {
    const int nb = std::min(kQBlock, q - b0);
    const int rc = search_block(ix, queries + (size_t)b0 * dim, nb, k, exclude ? exclude + b0 : nullptr,
                                top_pos + (size_t)b0 * k, top_scores + (size_t)b0 * k, s);
    if (rc != SRS_OK) {
      cudaEventRecord(ix->done, s);
      return rc;
    }
  }
  RT_TRY(cudaEventRecord(ix->done, s));
  return SRS_OK;
}

int check_search(const srs_index* ix, int32_t q, int32_t dim, int32_t k) {
  if (!ix) return fail_fmt(SRS_ERR_INVALID, "null index");
  if (k < 1 || k > kMaxK) return fail_fmt(SRS_ERR_INVALID, "k must be in 1..%d", kMaxK);
  if (dim != ix->dim) return fail_fmt(SRS_ERR_INVALID, "query dim %d != index dim %d", dim, ix->dim);
  if (q < 0) return fail_fmt(SRS_ERR_INVALID, "negative query count");
  return SRS_OK;
}

}  // namespace

extern "C" {

int srs_index_create(const float* items, int64_t n, int32_t dim, int32_t metric, int32_t location, int32_t device,
                     srs_index** out) {
  if (!out || !items) return fail_fmt(SRS_ERR_INVALID, "null argument");
  *out = nullptr;
  if (n < 1 || n >= ((int64_t)1 << 31)) return fail_fmt(SRS_ERR_INVALID, "n must be in 1..2^31-1");
  if (dim < 1 || dim > kMaxDim) return fail_fmt(SRS_ERR_INVALID, "dim must be in 1..%d", kMaxDim);
  if (metric != SRS_DOT && metric != SRS_COSINE) return fail_fmt(SRS_ERR_INVALID, "unknown metric %d", metric);
  if (location != SRS_HOST && location != SRS_DEVICE_BORROWED)
    return fail_fmt(SRS_ERR_INVALID, "unknown location %d", location);
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail_fmt(SRS_ERR_CUDA, "no CUDA device available; this library has no CPU path");
  if (device < 0 || device >= ndev) return fail_fmt(SRS_ERR_INVALID, "device %d out of range", device);
  RT_TRY(cudaSetDevice(device));
  srs_index* ix = new srs_index();
  ix->device = device; ix->metric = metric; ix->dim = dim; ix->n = n;
  ix->Dp = (dim + 15) & ~15;
  ix->W = kblock_width(ix->Dp);
  ix->ntiles = (int)((n + 127) / 128);
  ix->m = margin(ix->Dp, metric);
  cudaDeviceGetAttribute(&ix->sms, cudaDevAttrMultiProcessorCount, device);
  int rc = SRS_OK;
  auto bail = [&](int code) { free_index(ix); return code; };
  cudaError_t e = setup_retrieve_attributes();
  if (e != cudaSuccess) return bail(fail_fmt(SRS_ERR_CUDA, "kernel attribute setup failed: %s", cudaGetErrorString(e)));
  const size_t row_bytes = (size_t)n * dim * 4;
  if (location == SRS_DEVICE_BORROWED) {
    ix->rows = const_cast<float*>(items);
  } else {
    e = cudaMalloc(&ix->rows, row_bytes);
    if (e != cudaSuccess) return bail(fail_fmt(SRS_ERR_NOMEM, "cudaMalloc(%zu) failed: %s", row_bytes, cudaGetErrorString(e)));
    ix->own_rows = true;
    e = cudaMemcpy(ix->rows, items, row_bytes, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) return bail(fail_fmt(SRS_ERR_CUDA, "item upload failed: %s", cudaGetErrorString(e)));
  }
  const size_t scan_bytes = (size_t)ix->ntiles * 128 * ix->Dp * 2;
  e = cudaMalloc(&ix->scan, scan_bytes);
  if (e == cudaSuccess) e = cudaMalloc(&ix->norms, (size_t)n * 4);
  if (e != cudaSuccess) return bail(fail_fmt(SRS_ERR_NOMEM, "index allocation failed: %s", cudaGetErrorString(e)));
  rc = alloc_scratch(ix);
  if (rc != SRS_OK) return bail(rc);
  index_norms_kernel<<<grid_for(n, 256, 148 * 16), 256, 0, ix->stream>>>(ix->rows, n, dim, metric, ix->norms);
  index_tiles_kernel<<<grid_for((int64_t)ix->ntiles * 128 * (ix->Dp / 8), 256, 148 * 32), 256, 0, ix->stream>>>(
      ix->rows, n, dim, ix->Dp, ix->W, metric, (int64_t)ix->ntiles * 128, ix->scan);
  g_launch_count += 2;
  e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaStreamSynchronize(ix->stream);
  if (e != cudaSuccess) return bail(fail_fmt(SRS_ERR_CUDA, "index build failed: %s", cudaGetErrorString(e)));
  *out = ix;
  return SRS_OK;
}

void srs_index_destroy(srs_index* ix) { free_index(ix); }

int srs_index_search_device(srs_index* ix, const float* queries, int32_t q, int32_t dim, int32_t k,
                            const int32_t* exclude, int32_t* top_pos, float* top_scores, void* stream) {
  int rc = check_search(ix, q, dim, k);
  if (rc != SRS_OK) return rc;
  if (q == 0) return SRS_OK;
  if (!queries || !top_pos || !top_scores) return fail_fmt(SRS_ERR_INVALID, "null pointer");
  std::lock_guard<std::mutex> lock(ix->mu);
  return search_locked(ix, queries, q, dim, k, exclude, top_pos, top_scores, static_cast<cudaStream_t>(stream));
}

int srs_index_search_host(srs_index* ix, const float* queries, int32_t q, int32_t dim, int32_t k,
                          const int32_t* exclude, int32_t* top_pos, float* top_scores) {
  int rc = check_search(ix, q, dim, k);
  if (rc != SRS_OK) return rc;
  if (q == 0) return SRS_OK;
  if (!queries || !top_pos || !top_scores) return fail_fmt(SRS_ERR_INVALID, "null pointer");
  std::lock_guard<std::mutex> lock(ix->mu);
  RT_TRY(cudaSetDevice(ix->device));
  // exact byte counts for the copies; the staging offsets are rounded up to 16 bytes
  const size_t qn = (size_t)q * dim * 4, en = exclude ? (size_t)q * 4 : 0, on = (size_t)q * k * 4;
  const size_t qb = (qn + 15) & ~(size_t)15, eb = en, ob = (on + 15) & ~(size_t)15;
  if (qb + eb + 2 * ob > ix->stage_bytes) {           // grows only; earlier uses ended with a synchronise
    cudaFree(ix->stage);
    ix->stage = nullptr;
    ix->stage_bytes = 0;
    const size_t want = std::max<size_t>(qb + eb + 2 * ob, 1 << 20);
    RT_TRY(cudaMalloc(&ix->stage, want));
    ix->stage_bytes = want;
  }
  uint8_t* d = ix->stage;
  float* dq = reinterpret_cast<float*>(d);
  int32_t* dpos = reinterpret_cast<int32_t*>(d + qb);
  float* dsc = reinterpret_cast<float*>(d + qb + ob);
  int32_t* dex = exclude ? reinterpret_cast<int32_t*>(d + qb + 2 * ob) : nullptr;
  cudaStream_t s = ix->stream;
  cudaError_t e = cudaMemcpyAsync(dq, queries, qn, cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess && exclude) e = cudaMemcpyAsync(dex, exclude, en, cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) {
    rc = search_locked(ix, dq, q, dim, k, dex, dpos, dsc, s);
    if (rc == SRS_OK) {
      e = cudaMemcpyAsync(top_pos, dpos, on, cudaMemcpyDeviceToHost, s);
      if (e == cudaSuccess) e = cudaMemcpyAsync(top_scores, dsc, on, cudaMemcpyDeviceToHost, s);
      if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    }
  }
  cudaStreamSynchronize(s);
  if (rc != SRS_OK) return rc;
  if (e != cudaSuccess) return fail_fmt(SRS_ERR_CUDA, "search failed: %s", cudaGetErrorString(e));
  return SRS_OK;
}

}  // extern "C"
